"""Time the analytic NLL gradient of the fidelity kernel against the central-difference path at the shard shape of BASELINE config 3
(hubregtsen q = 5, L = 2, n = 2048: the per-row kernel) and at q = 8 and q = 10 (L = 2, n = 2048 and 8192: the DMMA stages).

    python tools/fidelity_analytic_bench.py [--reps 3] [--rounds 3]

Per shape, with CUDA events: dqgp_states_jacobian, the whole dqgp_grad_fidelity_analytic, and dqgp_states_shifted +
dqgp_grad_fidelity (central difference).  The stages of the analytic gradient are kernels inside one entry point, so their times
come from a separate torch.profiler pass over the same calls.  Inputs are seeded and synthetic: the states and their Jacobian
from the circuit at random samples and parameters, a random symmetric A^-1 and alpha (the cost does not depend on the values).
Each figure is the median of the rounds' mean times.  Flops are counted from shapes: the weights stage 64 * 64 * 8 * 2^q per
lower 64 x 64 tile, the GEMM 2 * n_pad * 2^(q+1) * 2 n_pad, the contraction 2 * P * n * 2^(q+1), the central difference
2P * 64 * 64 * 8 * 2^q per lower tile.  Prints one JSON line with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import sys
from collections import defaultdict

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import dqgp_b200 as d  # noqa: E402
from outer_kernel_bench import card, timed  # noqa: E402

SHAPES = [("cfg3_q5_n2048", 5, 2048), ("q8_n2048", 8, 2048), ("q8_n8192", 8, 8192), ("q10_n2048", 10, 2048), ("q10_n8192", 10, 8192)]
# the stages' kernels as torch.profiler names them
STAGES = {"weights": "dqgp::fidelity_dmma_kernel<2>", "pack": "dqgp::grad_fid_pack_kernel", "table": "dqgp::grad_fid_task_kernel",
          "gemm": "dqgp::gemm_group_kernel", "contract": "dqgp::grad_fid_contract_kernel", "reduce": "dqgp::grad_reduce_kernel",
          "rows": "dqgp::grad_fid_analytic_rows_kernel", "sum": "dqgp::grad_analytic_sum_kernel"}


def stage_ms(fn, reps):
    """Mean device time per call of each stage kernel, from a torch.profiler trace of `reps` calls."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = defaultdict(float)
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
        for stage, prefix in STAGES.items():
            if prefix in ev.key:
                out[stage] += us / 1000.0 / reps
    return dict(out)


def flops(q, n, P):
    dim = 1 << q
    t = (n + 63) // 64
    tiles = t * (t + 1) // 2
    npad = (n + 127) // 128 * 128
    tp = npad // 64
    return {"weights": tp * (tp + 1) // 2 * 64 * 64 * 8 * dim if dim >= 128 else None,
            "gemm": 2 * npad * 2 * dim * 2 * npad if dim >= 128 else None,
            "contract": 2 * P * n * 2 * dim,
            "central_difference": 2 * P * tiles * 64 * 64 * 8 * dim}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fidelity_analytic_bench needs a CUDA device")
    lib = d.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    results = {}
    for name, q, n in SHAPES:
        if name not in args.shapes.split(","):
            continue
        rng = np.random.default_rng(q * 100003 + n)
        ec = d.EncodingCircuit("hubregtsen", q, 2, 2)
        P, dim = ec.num_parameters, 1 << q
        dx = d.kernels.dev_f64(rng.uniform(-2, 2, (n, 2)))
        z = rng.uniform(0.2, 2.9, P)
        pm = torch.empty((2 * P + 1, P), dtype=torch.float64, device="cuda")
        assert lib.dqgp_shift_parameter_sets(d.kernels.dev_f64(z).data_ptr(), P, np.pi / 8, np.pi, pm.data_ptr(), st) == 0
        psi = torch.empty((n, dim, 2), dtype=torch.float64, device="cuda")
        D = torch.empty((P, n, dim, 2), dtype=torch.float64, device="cuda")
        g = torch.Generator(device="cuda").manual_seed(q + n)
        B = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=g)
        ainv = B + B.T
        del B
        alpha = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
        grad = torch.zeros(P, dtype=torch.float64, device="cuda")
        work_a = torch.empty(lib.dqgp_grad_fidelity_analytic_workspace_bytes(n, dim) // 8 + 1, dtype=torch.float64, device="cuda")
        work = torch.empty(lib.dqgp_grad_workspace_bytes(n, P) // 8 + 1, dtype=torch.float64, device="cuda")

        def jacobian():
            assert lib.dqgp_states_jacobian(ec.handle, dx.data_ptr(), n, pm.data_ptr(), psi.data_ptr(), D.data_ptr(), st) == 0, \
                lib.dqgp_last_error()

        def analytic():
            assert lib.dqgp_grad_fidelity_analytic(ainv.data_ptr(), n, alpha.data_ptr(), psi.data_ptr(), D.data_ptr(), n, dim, P,
                                                   grad.data_ptr(), work_a.data_ptr(), st) == 0, lib.dqgp_last_error()

        samples = defaultdict(list)
        for _ in range(args.rounds):
            samples["states_jacobian_ms"].append(timed(jacobian, args.reps))
            samples["grad_analytic_ms"].append(timed(analytic, args.reps))
        stages = stage_ms(analytic, args.reps)
        del work_a
        # central difference: the 2P + 1 state sets replace the Jacobian
        sets = torch.empty((2 * P + 1, n, dim, 2), dtype=torch.float64, device="cuda")

        def shifted():
            assert lib.dqgp_states_shifted(ec.handle, dx.data_ptr(), n, pm.data_ptr(), P, sets.data_ptr(), st) == 0, lib.dqgp_last_error()

        def central():
            assert lib.dqgp_grad_fidelity(ainv.data_ptr(), n, alpha.data_ptr(), sets.data_ptr(), n, dim, P, np.pi / 8, grad.data_ptr(),
                                          work.data_ptr(), st) == 0, lib.dqgp_last_error()

        for _ in range(args.rounds):
            samples["states_shifted_ms"].append(timed(shifted, args.reps))
            samples["grad_central_ms"].append(timed(central, max(1, args.reps // 2) if q >= 10 else args.reps))
        med = {k: sorted(v)[len(v) // 2] for k, v in samples.items()}
        fl = flops(q, n, P)
        rates = {}
        for k, ms in (("weights", stages.get("weights")), ("gemm", stages.get("gemm")), ("contract", stages.get("contract")),
                      ("central_difference", med["grad_central_ms"])):
            if fl[k] is not None and ms:
                rates[k] = round(fl[k] / (ms * 1e-3) / 1e12, 2)
        an_total = med["states_jacobian_ms"] + med["grad_analytic_ms"]
        cd_total = med["states_shifted_ms"] + med["grad_central_ms"]
        results[name] = {"q": q, "n": n, "P": P, **{k: round(v, 4) for k, v in med.items()},
                         "spread_ms": {k: round(max(v) - min(v), 4) for k, v in samples.items()},
                         "stages_ms": {k: round(v, 4) for k, v in stages.items()},
                         "flops": {k: v for k, v in fl.items() if v is not None}, "tflops": rates,
                         "grad_ratio_central_over_analytic": round(med["grad_central_ms"] / med["grad_analytic_ms"], 2),
                         "step_ratio_central_over_analytic": round(cd_total / an_total, 2)}
        del psi, D, sets, ainv, work
        torch.cuda.empty_cache()
    name, power = card()
    print(json.dumps({"tool": "fidelity_analytic_bench", "card": name, "power_limit_w": power, "reps": args.reps, "rounds": args.rounds,
                      "results": results}))


if __name__ == "__main__":
    main()
