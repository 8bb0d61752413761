"""Throughput of the DMMA GEMM building block (dqgp_dgemm) against the measured FP64 peak.  Usage: python tools/gemm_bench.py

The test utility builds and frees the two tensor maps of its one task on every call (cudaMalloc / cudaFree): at K = 8192 that is
noise, at K <= 256 it dominates - for kernel rates of the small-K shapes, time a factorisation
(tools/factor_breakdown.py), where the maps are built once per solver."""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dqgp_b200 as d  # noqa: E402

lib = d.load()
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
for (M, N, K) in [(8192, 8192, 8192), (8192, 8192, 128), (8192, 8192, 256), (4096, 4096, 4096)]:
    for akc, bkc in [(1, 1), (0, 0), (1, 0)]:
        a = torch.randn((M, K) if akc else (K, M), dtype=torch.float64, device="cuda")
        b = torch.randn((N, K) if bkc else (K, N), dtype=torch.float64, device="cuda")
        c = torch.zeros((M, N), dtype=torch.float64, device="cuda")
        beta = 1.0 if K <= 256 else 0.0
        def run():
            rc = lib.dqgp_dgemm(akc, bkc, M, N, K, -1.0, a.data_ptr(), a.shape[1], b.data_ptr(), b.shape[1], beta, c.data_ptr(), N, st)
            assert rc == 0
        run(); torch.cuda.synchronize()
        reps = 3 if K > 1000 else 20
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        print(f"M={M} N={N} K={K} a_k={akc} b_k={bkc} beta={beta}: {ms:8.3f} ms  {2.0 * M * N * K / ms / 1e9:6.2f} TFLOP/s")
