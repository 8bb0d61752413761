// Small utility entry points of the C ABI that do not belong to a kernel file.
#include "gemm64.cuh"

extern "C" {

// Building block exposed for tests and for callers that want the DMMA GEMM directly:
// C(MxN) = alpha * A * B + beta * C with A given as [m][k] (a_k_contig=1) or [k][m] (0), B as [n][k] (1) or [k][n] (0).
// M and N must be multiples of 128, K a multiple of 16, leading dimensions even and pointers 16-byte aligned.
int dqgp_dgemm(int a_k_contig, int b_k_contig, int M, int N, int K, double alpha, const double* d_A, int lda, const double* d_B,
               int ldb, double beta, double* d_C, int ldc, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_A && d_B && d_C, "dqgp_dgemm: NULL argument");
    DQGP_REQUIRE(M > 0 && N > 0 && K > 0 && M % GM_BM == 0 && N % 128 == 0 && K % GM_KC == 0,
                 "dqgp_dgemm: M,N must be multiples of 128 and K of 16 (got %d,%d,%d)", M, N, K);
    DQGP_REQUIRE(lda % 2 == 0 && ldb % 2 == 0 && ldc % 2 == 0, "dqgp_dgemm: leading dimensions must be even");
    DQGP_REQUIRE(((uintptr_t)d_A % 16 == 0) && ((uintptr_t)d_B % 16 == 0) && ((uintptr_t)d_C % 16 == 0), "dqgp_dgemm: pointers must be 16-byte aligned");
    GemmTask t;
    t.A = d_A; t.B = d_B; t.C = d_C; t.M = M; t.N = N; t.K = K; t.lda = lda; t.ldb = ldb; t.ldc = ldc;
    t.a_k_contig = a_k_contig ? 1 : 0; t.b_k_contig = b_k_contig ? 1 : 0; t.lower_tiles = 0; t.krule = GM_KRULE_ALL;
    t.alpha = alpha; t.beta = beta; t.tile_begin = 0; t.tiles = gemm_task_tiles(t);
    cudaStream_t st = as_stream(stream);
    GemmTask* d_t = nullptr;
    DQGP_CUDA(cudaMallocAsync(&d_t, sizeof t, st));
    DQGP_CUDA(cudaMemcpyAsync(d_t, &t, sizeof t, cudaMemcpyHostToDevice, st));
    DQGP_CUDA(cudaStreamSynchronize(st));   // `t` lives on this stack frame
    gemm_register_maps(d_t, &t, 1);          // tensor maps of the operands
    int rc = launch_gemm_group(d_t, 1, t.tiles, st);
    DQGP_CUDA(cudaStreamSynchronize(st));    // the maps (if any) are freed below
    gemm_unregister_maps(d_t);
    cudaFreeAsync(d_t, st);
    return rc;
}
}
