"""Time the NLL gradient with respect to the outer kernel's hyper-parameters (dqgp_grad_outer_hyperparameters) for every outer kernel
at the shard shapes of BASELINE configs 4 and 5, the noise entry (dqgp_grad_noise_std), and one config-4 AgentEngine.step with
hyper_gradient off and on, with CUDA events.

    python tools/hyper_gradient_bench.py [--reps 20] [--rounds 3] [--step-reps 5]

Inputs are seeded and synthetic: features uniform in [-1, 1] (where Pauli expectations lie), a random symmetric A^-1 and alpha (the
pass's cost does not depend on these values); A^-1 (512 MB at n = 8192) does not fit the 126 MB L2.  Each figure is the median of
`rounds` mean times; the two step engines are timed alternately.  Bytes and flops are counted from shapes: the pass reads the lower
half of A^-1 (8 B per entry) and spends 2m (the Gram identity's -d^2) + 2k (the contraction with B, k hyper-parameters) FP64
flops per lower entry; the transcendentals are not counted.  `bound` names the larger of bytes / 6547.5 GB/s and flops / 37.1 TF.
Prints one JSON line with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dqgp_b200 as d  # noqa: E402
from dqgp_b200 import _lib  # noqa: E402
from outer_kernel_bench import card, timed  # noqa: E402

OUTERS = {"gaussian": 1, "matern": 1, "expsinesquared": 2, "rationalquadratic": 2, "dotproduct": 1}
SHAPES = {"cfg4": dict(n=8192, m=24), "cfg5": dict(n=8192, m=30)}
HBM_GBS, FP64_TFLOPS = 6547.5, 37.1
STEP = dict(n=8192, d=4, encoding_type="yz_cx", kernel_type="projected", num_qubits=8, num_layers=3)     # config 4's agent shard


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--step-reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hyper_gradient_bench needs a CUDA device")
    lib = d.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(0)
    results = {}
    for sname, s in SHAPES.items():
        n, m = s["n"], s["m"]
        F = torch.rand((n, m), dtype=torch.float64, device="cuda", generator=g) * 2 - 1
        B = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=g)
        ainv = B + B.T
        del B
        alpha = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
        grad = torch.zeros(3, dtype=torch.float64, device="cuda")
        work = torch.empty(lib.dqgp_grad_outer_hyperparameters_workspace_bytes(n) // 8 + 1, dtype=torch.float64, device="cuda")
        samples = {o: [] for o in OUTERS}
        samples["noise_std"] = []
        for _ in range(args.rounds):
            for o in OUTERS:
                oid, hyp = _lib.OUTER_KERNELS[o], _lib.hyp_array(d.kernels.outer_hyp(o))

                def hyper():
                    assert lib.dqgp_grad_outer_hyperparameters(oid, hyp, ainv.data_ptr(), n, alpha.data_ptr(), F.data_ptr(), n, m,
                                                               grad.data_ptr(), work.data_ptr(), st) == 0, lib.dqgp_last_error()
                samples[o].append(timed(hyper, args.reps))

            def noise():
                assert lib.dqgp_grad_noise_std(ainv.data_ptr(), n, alpha.data_ptr(), n, 0.1, grad.data_ptr(), st) == 0, lib.dqgp_last_error()
            samples["noise_std"].append(timed(noise, args.reps))
        lower = n * (n + 1) // 2
        res = {"n": n, "m": m, "bytes": 8 * lower}
        for o, k in OUTERS.items():
            ms = sorted(samples[o])[len(samples[o]) // 2]
            flops = lower * (2 * m + 2 * k)
            t_bytes, t_flops = 8 * lower / (HBM_GBS * 1e6), flops / (FP64_TFLOPS * 1e9)
            res[o] = {"ms": round(ms, 4), "spread_ms": round(max(samples[o]) - min(samples[o]), 4), "flops": flops,
                      "bound": "hbm" if t_bytes >= t_flops else "fp64", "bound_ms": round(max(t_bytes, t_flops), 4),
                      "achieved_gbs": round(8 * lower / (ms * 1e6), 1)}
        res["noise_std_ms"] = round(sorted(samples["noise_std"])[len(samples["noise_std"]) // 2], 4)
        results[sname] = res
        del F, ainv, work
        torch.cuda.empty_cache()

    # one config-4 agent step, hyper_gradient off and on (training kernel Gaussian, gamma = 1, as config 4 runs)
    x, y = d.synthetic_dataset(STEP["n"], STEP["d"], STEP["encoding_type"])
    kw = {k: v for k, v in STEP.items() if k not in ("n", "d")}
    engines = {flag: d.AgentEngine(x, y, noise_std=0.1, rho=100.0, L=100.0, hyper_gradient=flag, **kw) for flag in (False, True)}
    P = engines[False].P
    z = d.kernels.dev_f64(np.random.RandomState(0).uniform(0.2, 2.9, P))
    psi = torch.zeros_like(z)
    outs = {flag: (torch.empty_like(z), torch.empty_like(z)) for flag in engines}
    steps = {flag: [] for flag in engines}
    for _ in range(args.rounds):
        for flag, eng in engines.items():
            steps[flag].append(timed(lambda: eng.step(z, psi, *outs[flag]), args.step_reps))
    assert torch.equal(outs[False][0], outs[True][0]), "the flag must not change the step's results"
    step = {("on" if f else "off"): {"ms": round(sorted(v)[len(v) // 2], 3), "spread_ms": round(max(v) - min(v), 3)} for f, v in steps.items()}
    step["added_pct"] = round(100.0 * (step["on"]["ms"] - step["off"]["ms"]) / step["off"]["ms"], 2)
    step["hyper_gradient"] = engines[True].hyper_gradient()
    name, power = card()
    print(json.dumps({"tool": "hyper_gradient_bench", "card": name, "power_limit_w": power, "reps": args.reps, "rounds": args.rounds,
                      "hbm_gbs": HBM_GBS, "fp64_tflops": FP64_TFLOPS, "results": results, "cfg4_step": dict(step, P=P)}))


if __name__ == "__main__":
    main()
