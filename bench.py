#!/usr/bin/env python
"""bench.py — ADMM iterations/s and quantum-kernel entries/s (fp64) of the dqgp hot path on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port), host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # also save each workload's final ADMM state as DIR/*.npy

A "step" is one ADMM iteration (SURVEY §8(d)): consensus z-update + every agent's train_and_update equivalent
(2P+1 parameter sets -> features -> Gram -> Cholesky/inverse -> fused central-difference gradient -> local
update) + the consensus exchange; the per-iteration CV of the reference (Q14) and printing are excluded.
`value` = kernel entries per second = (agents x (2P+1) x n_i^2 full-square entries per iteration) / time, with
all inputs resident in HBM; `e2e` = the same metric through RiemannianAgent.train_and_update with host buffers.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # the benchmark leaves the source tree as it found it (it may be read-only)

WORKLOADS = {
    # BASELINE.json configs[3]: the configuration the metric is quoted on at 1/2/4/8 GPUs
    "cfg4": dict(desc="synthetic 4D N=65536, yz_cx projected kernel, 8 qubits, 3 layers, gaussian outer, 8 agents",
                 N=65536, d=4, encoding="yz_cx", kernel="projected", q=8, layers=3, outer="gaussian", agents=8, honour_outer=False),
    "cfg3": dict(desc="synthetic 2D N=16384, hubregtsen fidelity kernel, 5 qubits, 2 layers, 8 agents",
                 N=16384, d=2, encoding="hubregtsen", kernel="fidelity", q=5, layers=2, outer="gaussian", agents=8, honour_outer=False),
    "cfg5": dict(desc="synthetic 6D N=131072, kyriienko projected kernel, 10 qubits, 4 layers, matern, 16 agents",
                 N=131072, d=6, encoding="kyriienko", kernel="projected", q=10, layers=4, outer="matern", agents=16, honour_outer=True),
    # BASELINE.json configs[1]: the SRTM .hgt tiles are absent from the reference checkout (.MISSING_LARGE_BLOBS) and its
    # sampling seed is time-based, so this is a synthetic stand-in of the same shape (BASELINE.md section 3)
    "cfg2": dict(desc="synthetic stand-in for SRTM maharashtra: 2D N=900 (4 x 225), chebyshev projected kernel, 4 qubits, 3 layers, 4 agents",
                 N=900, d=2, encoding="chebyshev", kernel="projected", q=4, layers=3, outer="matern", agents=4, honour_outer=False),
    "cfg1": dict(desc="synthetic 2D N=900 (4 x 225), chebyshev projected kernel, 3 qubits, 1 layer, 4 agents",
                 N=900, d=2, encoding="chebyshev", kernel="projected", q=3, layers=1, outer="matern", agents=4, honour_outer=False),
}
NOISE_STD, RHO, LIP, H = 0.1, 100.0, 100.0, np.pi / 8
HBM_COPY_GBS = 6547.5                    # denominator of the Gram's HBM roofline: copy bandwidth measured on a B200 (BASELINE.md section 2)


def load_json(path, default=None):
    try:
        with open(path) as f:
            return json.load(f)
    except Exception:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_problem(w, world, rank):
    import dqgp_b200 as d
    x, y = d.synthetic_dataset(w["N"], w["d"], w["encoding"])
    A = w["agents"]
    if A % world:
        raise SystemExit(f"{A} agents do not split over {world} GPUs")
    n_i = w["N"] // A
    per = A // world
    shards = [(x[a * n_i:(a + 1) * n_i], y[a * n_i:(a + 1) * n_i]) for a in range(rank * per, (rank + 1) * per)]   # main.py:665
    P = d.EncodingCircuit(w["encoding"], w["q"], w["d"], w["layers"]).num_parameters
    rs = np.random.RandomState(42)                       # main.py:2407-2408
    theta0, psi0 = np.round(rs.rand(A, P), 4), np.round(rs.rand(A, P), 4)
    return shards, theta0, psi0, n_i, P


def flops_per_entry(w):
    """SURVEY §8(d) algorithmic flops per Gram entry (FMA = 2)."""
    if w["kernel"] == "fidelity":
        return 8 * (1 << w["q"]) + 3
    c = 2 if (w["outer"] == "gaussian" or not w["honour_outer"]) else 6
    return 3 * (3 * w["q"]) + c


def run_ours(args, w):
    """The headline workload in full (e2e, CPU baseline, rooflines), then - same process, same box - the other BASELINE configs
    named in --also as compact entries under "other_workloads", so that config 5 (the scaling stress) and config 3 (the fidelity
    kernel) are in the ONE JSON line the driver records."""
    import gc
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        pg = dist.group.WORLD
    line = measure(args, w, args.workload, pg, world, rank, local_rank, full=True)
    import dqgp_b200.agent as _agent
    _agent._ENGINE_CACHE.clear()          # the e2e leg's engines (3 squares per agent) are not needed any more
    others = {}
    for name in [v for v in args.also.split(",") if v and v != args.workload]:
        wo = WORKLOADS[name]
        if wo["agents"] % world:
            continue
        gc.collect(); torch.cuda.empty_cache()
        sub = copy_args(args, steps=max(2, min(args.steps, 3 if name == "cfg5" else 20)), warmup=3 if name == "cfg5" else 5)
        r = measure(sub, wo, name, pg, world, rank, local_rank, full=False)
        if rank == 0:
            others[name] = {k: r[k] for k in ("ms_per_step", "value", "admm_iters_per_s", "steps", "warmup", "phases_ms_one_agent", "roofline",
                                              "step_level", "clocks", "final_z_head") if k in r}
            others[name]["workload"] = r["config"]["workload"]
            others[name]["rooflines_frac"] = {k: {"frac": v["frac"], **({"frac_executed": v["frac_executed"]} if "frac_executed" in v else {})}
                                              for k, v in r["rooflines"].items()}
    if rank == 0:
        if others:
            line["other_workloads"] = others
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def copy_args(args, **kw):
    out = argparse.Namespace(**vars(args))
    for k, v in kw.items():
        setattr(out, k, v)
    return out


def dump_outputs(out_dir, workload_name, **arrays):
    """What a caller of the timed path receives after its last step (AdmmEngine.state(): consensus z, every agent's theta and
    psi, every agent's NLL) as float64 DIR/<workload>_<name>.npy.  Inputs are seeded, so the same arguments give the same
    inputs on every run and two builds can be compared file by file.  A few KB per workload (A x P values)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{workload_name}_{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def measure(args, w, workload_name, pg, world, rank, local_rank, full):
    import torch
    import torch.distributed as dist
    import dqgp_b200 as d

    shards, theta0, psi0, n_i, P = make_problem(w, world, rank)
    kw = dict(encoding_type=w["encoding"], kernel_type=w["kernel"], num_qubits=w["q"], num_layers=w["layers"], noise_std=NOISE_STD,
              outer_kernel=w["outer"], shift_value=H, training_ignores_outer_kernel=not w["honour_outer"])
    if args.outer_blocks > 0:
        kw["cholesky_outer_blocks"] = args.outer_blocks
    eng = d.AdmmEngine(shards, theta0, psi0, rho=RHO, L=LIP, process_group=pg, rank=rank, world_size=world, **kw)
    S = 2 * P + 1
    entries_per_iter = w["agents"] * S * n_i * n_i

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_fn = eng.iteration
    use_graph = args.graph in ("on", "auto")
    if use_graph:
        try:
            eng.capture()                        # replay the whole iteration (all agent / look-ahead streams) as one CUDA graph
            step_fn = eng.replay
        except Exception as exc:                 # capture is an optimisation, not a requirement
            print(f"[bench] CUDA graph capture failed ({exc!r}); running eagerly", file=sys.stderr)
            use_graph = False
            torch.cuda.synchronize()
    for _ in range(args.warmup):
        step_fn()
    barrier()
    for a in eng.agents:
        a.check_info()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    try:                                     # no nvidia-smi sampler outlives a failed step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            step_fn()
        e1.record()
        barrier()
    finally:
        clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    z_final, theta_final, psi_final, nll = eng.state()
    if args.dump_outputs:
        nll_all = nll
        if world > 1:                        # z, theta, psi are replicated after the exchange; the NLLs are per rank
            local = torch.from_numpy(nll).cuda()
            gathered = torch.empty(world * local.numel(), dtype=local.dtype, device="cuda")
            dist.all_gather_into_tensor(gathered, local)
            nll_all = gathered.cpu().numpy()
        if rank == 0:
            dump_outputs(args.dump_outputs, workload_name, z=z_final, theta=theta_final, psi=psi_final, nll=nll_all)

    # ---- per-phase device times of ONE agent step (same stream, CUDA events), after the timed region -------------
    ag = eng.agents[0]
    phases = {}
    reps = 3
    def timed(name, fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        phases[name] = a.elapsed_time(b) / reps
    zz = eng.z.clone()
    timed("statevector", lambda: ag.simulate(zz))
    timed("gram", ag.gram)
    def fac():
        ag.gram(); ag.factor()
    timed("gram+factor", fac)
    phases["factor"] = phases.pop("gram+factor") - phases["gram"]
    timed("gradient", ag.gradient)
    fp64 = load_json(os.path.join(ROOT, "profiles", "r01_fp64_peak.json"), {})
    peak_tf = float(fp64.get("dmma_m8n8k4_tflops", 37.1))
    fpe = flops_per_entry(w)
    np_pad = ((n_i + 127) // 128) * 128
    grad_flops = 2 * P * n_i * n_i * fpe                     # algorithmic: full squares of the 2P shifted Grams
    chol_flops = float(np_pad) ** 3                          # potrf n^3/3 + trtri n^3/3 + lauum n^3/3
    t64 = (n_i + 63) // 64
    gram_entries = 64 * 64 * t64 * (t64 + 1) // 2 if w["kernel"] == "projected" else n_i * n_i
    # statevector: SURVEY 8(d) counts 14 * 2^q flops per gate per state over all S * n states (what a per-set simulation does);
    # the engine executes far fewer (shared circuit prefixes, both signs of a parameter from one fork, fused 1-qubit runs):
    # `executed` = 32 * 2^(q-1) flops (16 FMA per amplitude pair, FMA = 2) per fused 2x2 unitary application, counted by the
    # library's own plan
    lib = d.load()
    circ = ag.circuit
    sv_alg = float(S) * n_i * circ.num_gates * 14.0 * (1 << w["q"])
    sv_exec = float(n_i) * lib.dqgp_circuit_shifted_u2_applications(circ.handle) * 32.0 * (1 << (w["q"] - 1))
    roof = {
        "statevector": {"bound": "fp64", "achieved": sv_alg / (phases["statevector"] * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                        "executed": sv_exec / (phases["statevector"] * 1e-3) / 1e12,
                        "note": "achieved = SURVEY 8(d) algorithmic flops (14 * 2^q per gate per state, S * n states: a per-set simulation) / time, "
                                "can exceed the peak because prefix sharing and the linear-combination forks skip work; executed = fused 2x2 "
                                "unitary applications of the plan x 32 * 2^(q-1) flops (16 FMA per pair; Pauli-feature epilogues not counted) / time"},
        "gradient": {"bound": "fp64", "achieved": grad_flops / (phases["gradient"] * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                     "executed": 0.5 * (1.0 + 1.0 / t64) * grad_flops / (phases["gradient"] * 1e-3) / 1e12,
                     "note": "achieved = algorithmic flops (SURVEY 8d: full squares, transcendental = 1 flop) / time; executed = the lower "
                             "64x64 tiles only (symmetry), same per-entry count: the fraction of the pipe's peak that is comparable with 1"},
        "factor": {"bound": "fp64-dmma", "achieved": chol_flops / (phases["factor"] * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                   "note": "n^3 flops: potrf + triangular inverse + inverse product, DMMA.8x8x4 trailing updates"},
        "gram": {"bound": "hbm", "achieved": 8.0 * gram_entries / (phases["gram"] * 1e-3) / 1e9, "peak": HBM_COPY_GBS, "unit": "GB/s",
                 "note": "8 B per written entry of the unshifted Gram; the training Gram writes the 64x64 tiles of the lower "
                         "triangle only (all the factorisation reads)" if w["kernel"] == "projected" else "8 B per written entry of the unshifted Gram"},
    }
    for r in roof.values():
        r["frac"] = r["achieved"] / r["peak"]
        if "executed" in r:
            r["frac_executed"] = r["executed"] / r["peak"]
    # step level: executed FP64 work of all local agents (factorisation n^3, the gradient's lower tiles, the simulator's fused
    # unitaries) over the measured iteration time - what the whole step keeps of the pipe, agents overlapping on their streams
    step_exec = len(eng.agents) * (chol_flops + 0.5 * (1.0 + 1.0 / t64) * grad_flops + sv_exec)
    step_level = {"executed_tflops": step_exec / (total_ms / args.steps * 1e-3) / 1e12, "peak": peak_tf,
                  "note": "executed flops of this rank's agents (factorisation n^3 + gradient lower tiles + simulator 2x2 unitaries) / iteration time"}
    step_level["frac"] = step_level["executed_tflops"] / peak_tf
    dominant = max(("gradient", "factor", "statevector", "gram"), key=lambda k: phases[k])
    primary = dict(roof[dominant])
    if "executed" in primary:            # the headline fraction is the one that cannot exceed 1
        primary["achieved_algorithmic"], primary["achieved"] = primary["achieved"], primary["executed"]
        primary["frac"] = primary["frac_executed"]
    traffic_file = "r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_traffic.json")) else "r01_traffic.json"
    traffic = load_json(os.path.join(ROOT, "profiles", traffic_file), {})
    primary.update({"kernel": {"gradient": "grad_projected_dmma_kernel" if w["kernel"] == "projected" else "fidelity_dmma_kernel<1>",
                               "factor": "gemm_group_kernel" if os.environ.get("DQGP_GEMM_NO_TMAP") else "gemm_group_tmap_kernel", "gram": "gram_projected_dmma_kernel",
                               "statevector": ("statevec_lc2_kernel<%d>" if w["encoding"] in ("yz_cx", "kyriienko") else "statevec_lc_kernel<%d>") % w["q"]}[dominant], "phase": dominant,
                    "traffic": None, "peak_source": "profiles/r01_fp64_peak.json (pure DMMA/DFMA issue loops measured on a B200)"
                    if primary["bound"] != "hbm" else "BASELINE.md section 2 (HBM copy, read + write, measured on a B200)"})

    tk = traffic.get(primary["kernel"].replace("grad_projected_kernel", "grad_projected_dmma_kernel"), {})
    if tk.get("dram_bytes"):
        primary["traffic"] = tk["dram_bytes"]
        primary["traffic_note"] = (f"dram__bytes_read+write of one launch under ncu (profiles/{traffic_file}): " + tk.get("launch", tk.get("note", "")))

    # ---- e2e: host buffers through RiemannianAgent.train_and_update + host consensus ------------------------------
    e2e = None if (args.skip_e2e or not full) else run_e2e(args, w, d, torch, dist, world, rank, shards, theta0, psi0, n_i, P, entries_per_iter)

    cpu_base = None
    if full and rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_reference_sample(w, n_i, P)

    launches = (sum(a.launches_per_step() for a in eng.agents) + 2) * world    # + consensus, the row exchange; all ranks
    if rank == 0:
        ms_per_step = total_ms / args.steps
        line = {
            "metric": "quantum_kernel_entries_per_s", "value": entries_per_iter / (ms_per_step * 1e-3), "unit": "entries/s",
            "admm_iters_per_s": 1e3 / ms_per_step,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{workload_name}: {w['desc']}", "agents": w["agents"], "samples_per_agent": n_i, "parameters": P,
                       "parameter_sets": S, "entries_per_iteration": entries_per_iter, "agents_per_gpu": w["agents"] // world,
                       "training_outer_kernel": "gaussian" if not w["honour_outer"] else w["outer"],
                       "cache": "per-agent working set (3 x n_pad^2 fp64 = %.1f GB) exceeds the 126 MB L2; no flush needed" % (3 * 8 * np_pad ** 2 / 1e9),
                       "noise_std": NOISE_STD, "rho": RHO, "L": LIP, "shift": "pi/8", "cuda_graph": bool(use_graph)},
            "gpu_launches": launches * args.steps, "clocks": clocks, "e2e": e2e,
            "phases_ms_one_agent": phases, "roofline": primary, "rooflines": roof, "step_level": step_level, "cpu_baseline": cpu_base,
            "final_nll_rank0": [float(v) for v in nll], "final_z_head": [float(v) for v in z_final[:4]],
        }
        return line
    return None


def run_e2e(args, w, d, torch, dist, world, rank, shards, theta0, psi0, n_i, P, entries_per_iter):
    """Same iteration through the reference-facing API: host arrays into RiemannianAgent.train_and_update (H2D of the
    shard, z, psi and D2H of the result inside the timed region), consensus with the host RiemannianADMM.update_z."""
    A = w["agents"]
    per = A // world
    agents = [d.RiemannianAgent(f"agent_{rank * per + i + 1}", x, y, w["q"], NOISE_STD, RHO, LIP, use_parameter_shift=True,
                                shift_value=H, num_layers=w["layers"], encoding_type=w["encoding"], kernel_type=w["kernel"],
                                outer_kernel=w["outer"], training_ignores_outer_kernel=not w["honour_outer"],
                                reupload_shard="always")      # the e2e contract: every step's inputs cross PCIe inside the timed region
              for i, (x, y) in enumerate(shards)]
    _, _, admm = d.create_riemannian_framework(P, rho=RHO)
    streams = [torch.cuda.Stream() for _ in agents]
    theta, psi = theta0.copy(), psi0.copy()

    def one_iteration():
        nonlocal theta, psi
        z = np.round(admm.update_z(theta, psi), 4)
        loc = np.empty((per, 2, P))
        results = d.train_agents(agents, z, [psi[rank * per + i] for i in range(per)], streams)
        for i, (th, ps, _, _, _) in enumerate(results):
            loc[i, 0], loc[i, 1] = np.round(th, 4), np.round(ps, 4)
        if world > 1:
            buf = torch.from_numpy(loc).cuda()
            full = torch.empty((world,) + buf.shape, dtype=buf.dtype, device="cuda")
            dist.all_gather_into_tensor(full.view(-1), buf.view(-1))
            allv = full.cpu().numpy().reshape(A, 2, P)
        else:
            allv = loc
        theta, psi = allv[:, 0].copy(), allv[:, 1].copy()

    steps = max(1, min(args.steps, args.e2e_steps))
    one_iteration()                      # warm-up (engine cache, pinned buffers)
    one_iteration()                      # second call: every agent captures its step as a CUDA graph
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_iteration()
    torch.cuda.synchronize()
    el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    sec = float(el.item()) / steps
    return {"value": entries_per_iter / sec, "unit": "entries/s", "admm_iters_per_s": 1.0 / sec, "steps": steps,
            "h2d_bytes_per_step": int(sum(a.h2d_bytes for a in agents)) * world, "d2h_bytes_per_step": int(sum(a.d2h_bytes for a in agents)) * world,
            "api": "dqgp_b200.train_agents (= RiemannianAgent.train_and_update per agent, one stream each) with host arrays + host "
                   "RiemannianADMM.update_z; shard, z, psi staged through persistent pinned buffers and uploaded EVERY step "
                   "(reupload_shard='always'; the default keeps an unchanged shard resident)"}


# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(w, n_i, P, jobs=None):
    """The reference's CPU path (oracle port: the reference itself needs squlearn, absent here) on this box's host
    cores, bounded: `jobs` of the S = 2P+1 Gram jobs of ONE agent through a process pool of all cores (as
    agent_riemannian.py:261-262), plus the LAPACK sequence of agent_riemannian.py:410-418,442 (without the
    np.linalg.cond SVD) at a reduced n with n^3 extrapolation when n_i is large."""
    from oracle import agent_step, driver
    cores = os.cpu_count() or 1
    S = 2 * P + 1
    jobs = jobs or min(S, cores)
    x, y = driver.synthetic_dataset(w["N"], w["d"], w["encoding"])
    x, y = x[:n_i], y[:n_i]
    cfg = agent_step.KernelConfig(w["encoding"], w["kernel"], w["q"], w["layers"], w["outer"], training_ignores_outer_kernel=not w["honour_outer"])
    z = np.round(np.random.RandomState(42).rand(P), 4)
    sets = agent_step.shifted_parameter_sets(z, H)[:jobs]
    with agent_step.process_pool(cores) as pool:
        t0 = time.perf_counter()
        grams = list(pool.map(agent_step._gram_job, [(cfg, x, s) for s in sets]))
        t_gram = time.perf_counter() - t0
    n_la = min(n_i, 3072)
    c = grams[0][:n_la, :n_la]
    dk = np.zeros((1, n_la, n_la))
    t0 = time.perf_counter()
    agent_step.gp_terms(c, dk, y[:n_la], NOISE_STD, want_cond=False)
    t_la = (time.perf_counter() - t0) * (n_i / n_la) ** 3
    t_agent = t_gram * (S / jobs) + t_la + S * n_i * n_i * 8 / 2e9     # + the (P,n,n) dK pass at ~2 GB/s/…: negligible
    per_iter = t_agent * w["agents"]            # agents share the same cores (nested pools oversubscribe, they do not add cores)
    return {"value": w["agents"] * S * n_i * n_i / per_iter, "unit": "entries/s", "cores": cores, "kind": "port",
            "admm_iters_per_s_extrapolated": 1.0 / per_iter, "gram_entries_per_s_measured": jobs * n_i * n_i / t_gram,
            "sample": f"{jobs} of {S} Gram jobs of one agent (n_i={n_i}) over a {cores}-process pool: {t_gram:.2f} s; LAPACK sequence "
                      f"(cholesky, 4 solves, slogdet; no cond SVD) at n={n_la}, scaled by (n_i/n)^3 to {t_la:.2f} s; "
                      f"iteration time extrapolated to {S} jobs x {w['agents']} agents sharing the cores"}


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import circuits
    P = circuits.num_parameters(w["encoding"], w["q"], w["layers"])
    n_i = w["N"] // w["agents"]
    S = 2 * P + 1
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_reference_sample(w, n_i, P)
        if i >= args.warmup:
            vals.append(r)
    v = float(np.mean([r["value"] for r in vals]))
    base = dict(vals[-1]); base["value"] = v
    line = {"impl": "reference", "metric": "quantum_kernel_entries_per_s", "value": v, "unit": "entries/s",
            # each "step" of this arm is a BOUNDED SAMPLE of one iteration (see cpu_baseline.sample), not a whole iteration:
            # ms_per_step and admm_iters_per_s are extrapolations from the measured entries/s
            "extrapolated": True,
            "admm_iters_per_s": v / (w["agents"] * S * n_i * n_i), "n_gpus": world, "steps": len(vals), "warmup": args.warmup,
            "ms_per_step": 1e3 * (w["agents"] * S * n_i * n_i) / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {w['desc']}", "agents": w["agents"], "samples_per_agent": n_i, "parameters": P,
                       "parameter_sets": S, "note": "reference's own CPU implementation is not runnable (squlearn absent): oracle port "
                                                    "structured like the reference (process pool over Gram jobs + its LAPACK sequence)"},
            "cpu_baseline": base, "e2e": {"value": v, "unit": "entries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--also", default="cfg5,cfg3,cfg2,cfg1", help="other BASELINE workloads measured after the headline one (compact entries "
                                                        "under other_workloads); '' to skip")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only")
    ap.add_argument("--outer-blocks", type=int, default=0, help="Cholesky outer panel width in 128-blocks (0 = engine default)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"], help="replay the iteration as a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save each measured workload's final z / theta / psi / per-agent NLL as DIR/<workload>_<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times Gram samples, not whole iterations)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = max(args.warmup, 1)
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
