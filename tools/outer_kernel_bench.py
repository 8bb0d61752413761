"""Time the projected Gram (dqgp_gram_projected, same = 2: the lower tiles the factorisation reads), the fused central-difference
gradient (dqgp_grad_projected) and the analytic gradient (dqgp_grad_projected_analytic, `grad_analytic_ms`) for every outer kernel at
the shard shapes of BASELINE configs 4 and 5, with CUDA events.

    python tools/outer_kernel_bench.py [--reps 5] [--rounds 3]

Inputs are seeded and synthetic: features uniform in [-1, 1] (where Pauli expectations lie), a random symmetric A^-1 and alpha,
and for the analytic gradient a random feature Jacobian (the gradients' cost does not depend on these values).  The outer
kernels are timed in turn, `rounds` times over, and each figure is the median of the rounds' mean times.  Prints one JSON line
with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dqgp_b200 as d  # noqa: E402
from dqgp_b200 import _lib  # noqa: E402

OUTERS = ["gaussian", "matern", "expsinesquared", "rationalquadratic", "dotproduct"]
CONFIGS = {"cfg4": dict(n=8192, q=8, P=48), "cfg5": dict(n=8192, q=10, P=120)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, float(power)
    except Exception:                                   # the name from the runtime, the power limit unknown
        return torch.cuda.get_device_name(), None


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("outer_kernel_bench needs a CUDA device")
    lib = d.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(0)
    results = {}
    for cname, c in CONFIGS.items():
        n, m, P = c["n"], 3 * c["q"], c["P"]
        F = torch.rand((2 * P + 1, n, m), dtype=torch.float64, device="cuda", generator=g) * 2 - 1
        B = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=g)
        ainv = B + B.T
        del B
        alpha = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
        K = torch.zeros((n, n), dtype=torch.float64, device="cuda")
        grad = torch.zeros(P, dtype=torch.float64, device="cuda")
        work = torch.empty(lib.dqgp_grad_workspace_bytes(n, P) // 8 + 1, dtype=torch.float64, device="cuda")
        J = torch.randn((P, n, m), dtype=torch.float64, device="cuda", generator=g)
        work_a = torch.empty(lib.dqgp_grad_analytic_workspace_bytes(n, m) // 8 + 1, dtype=torch.float64, device="cuda")
        samples = {o: {"gram_ms": [], "grad_ms": [], "grad_analytic_ms": []} for o in OUTERS}
        for _ in range(args.rounds):
            for o in OUTERS:
                oid, hyp = _lib.OUTER_KERNELS[o], _lib.hyp_array(d.kernels.outer_hyp(o))

                def gram():
                    assert lib.dqgp_gram_projected(oid, hyp, F.data_ptr(), n, F.data_ptr(), n, m, K.data_ptr(), n, 2, st) == 0, \
                        lib.dqgp_last_error()

                def gradient():
                    assert lib.dqgp_grad_projected(oid, hyp, ainv.data_ptr(), n, alpha.data_ptr(), F.data_ptr(), n, m, P, 0.39269908169872414,
                                                   grad.data_ptr(), work.data_ptr(), st) == 0, lib.dqgp_last_error()

                def gradient_analytic():
                    assert lib.dqgp_grad_projected_analytic(oid, hyp, ainv.data_ptr(), n, alpha.data_ptr(), F.data_ptr(), J.data_ptr(), n,
                                                            m, P, grad.data_ptr(), work_a.data_ptr(), st) == 0, lib.dqgp_last_error()

                samples[o]["gram_ms"].append(timed(gram, 4 * args.reps))
                samples[o]["grad_ms"].append(timed(gradient, args.reps))
                samples[o]["grad_analytic_ms"].append(timed(gradient_analytic, 4 * args.reps))
        results[cname] = {"n": n, "q": c["q"], "m": m, "P": P,
                          **{o: {k: round(sorted(v)[len(v) // 2], 4) for k, v in s.items()} for o, s in samples.items()},
                          "spread_ms": {o: {k: round(max(v) - min(v), 4) for k, v in s.items()} for o, s in samples.items()}}
        del F, ainv, K, work, J, work_a
        torch.cuda.empty_cache()
    name, power = card()
    print(json.dumps({"tool": "outer_kernel_bench", "card": name, "power_limit_w": power, "reps": args.reps, "rounds": args.rounds,
                      "results": results}))


if __name__ == "__main__":
    main()
