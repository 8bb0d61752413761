// Grouped fp64 tile GEMM on the DMMA tensor path (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4), the one
// contraction engine behind the blocked Cholesky, triangular inverse and inverse product (chol.cu).
#pragma once
#include "common.cuh"

namespace dqgp {

constexpr int GM_BM = 128, GM_BN = 64, GM_KC = 16, GM_STAGES = 3, GM_THREADS = 256;
constexpr int GM_PITCH_K = GM_KC + 4;    // operand stored [row][k]  (k contiguous in HBM)
constexpr int GM_PITCH_M = GM_BM + 4;    // A operand stored [k][row]  (row contiguous in HBM)
constexpr int GM_PITCH_N = GM_BN + 4;    // B operand stored [k][col]
constexpr int GM_A_DOUBLES = (GM_BM * GM_PITCH_K > GM_KC * GM_PITCH_M) ? GM_BM * GM_PITCH_K : GM_KC * GM_PITCH_M;
constexpr int GM_B_DOUBLES = (GM_BN * GM_PITCH_K > GM_KC * GM_PITCH_N) ? GM_BN * GM_PITCH_K : GM_KC * GM_PITCH_N;
constexpr int GM_STAGE_DOUBLES = GM_A_DOUBLES + GM_B_DOUBLES;
constexpr size_t GM_SMEM_BYTES = size_t(GM_STAGES) * GM_STAGE_DOUBLES * sizeof(double);

// Tile shapes.  Big: 128x64 per CTA, 8 warps (4x2) of 32x32, two CTAs per SM - the throughput shape.  Small: 32x32 per
// CTA, 4 warps (2x2) of 16x16 - the latency shape for the two 128x128x128 products on the Cholesky's leaf chain,
// which it spreads over 16 (10 for the symmetric update) SMs instead of 2.
template <int BM_, int BN_, int WR_, int WC_>
struct GemmShape {
    static constexpr int BM = BM_, BN = BN_, WR = WR_, WC = WC_;
    static constexpr int THREADS = WR * WC * 32;
    static constexpr int MI = BM / WR / 8, NI = BN / WC / 8;          // 8x8 DMMA blocks per warp
    static constexpr int PITCH_M = BM + 4, PITCH_N = BN + 4;
    static constexpr int A_DOUBLES = (BM * GM_PITCH_K > GM_KC * PITCH_M) ? BM * GM_PITCH_K : GM_KC * PITCH_M;
    static constexpr int B_DOUBLES = (BN * GM_PITCH_K > GM_KC * PITCH_N) ? BN * GM_PITCH_K : GM_KC * PITCH_N;
    static constexpr int STAGE_DOUBLES = A_DOUBLES + B_DOUBLES;
    static constexpr size_t SMEM_BYTES = size_t(GM_STAGES) * STAGE_DOUBLES * sizeof(double);
};
using GemmBig = GemmShape<128, 64, 4, 2>;
using GemmSmall = GemmShape<32, 32, 2, 2>;

enum { GM_KRULE_ALL = 0, GM_KRULE_A_LOWER = 1, GM_KRULE_B_LOWER = 2, GM_KRULE_LAUUM = 3 };

// C(MxN) = alpha * A(MxK) * B(KxN) + beta * C.  M multiple of 128, N multiple of 64 (callers use 128); K multiple of 16.
struct GemmTask {
    const double* A;   // a_rowmajor_k ? A[m*lda + k] : A[k*lda + m]
    const double* B;   // b_rowmajor_k ? B[n*ldb + k] : B[k*ldb + n]
    double* C;         // C[m*ldc + n]
    int M, N, K;
    int lda, ldb, ldc;
    int a_k_contig, b_k_contig;
    int lower_tiles;   // only tiles with m0 >= n0 (square outputs)
    int krule;         // restrict the contraction range per tile when an operand is lower-triangular
    double alpha, beta;
    int tile_begin;    // first global tile id of this task within its launch group
    int tiles;         // number of tiles of this task
};

int launch_gemm_group(const GemmTask* d_tasks, int n_tasks, int total_tiles, cudaStream_t st);
// same table format with tile_begin / tiles counted in 32x32 tiles (gemm_task_tiles_small); GM_KRULE_ALL only
int launch_gemm_group_small(const GemmTask* d_tasks, int n_tasks, int total_tiles, cudaStream_t st);
int gemm_init();   // raises the dynamic shared memory limit once per process/device
// Operand tiles as two tensor-map boxes per k-chunk.  A task table registers its host copy once; launches whose device pointer lies
// inside a registered table use the tensor-map kernel, others (and tables whose maps the driver refused) the per-thread cp.async ring.
void gemm_register_maps(const GemmTask* d_tasks, const GemmTask* h_tasks, int n_tasks);
void gemm_unregister_maps(const GemmTask* d_tasks);

// lower_tiles: square output, only tiles that intersect the lower triangle: row block tm (128 rows) needs column
// blocks 0 .. (tm+1)*(BM/BN)-1, i.e. R*(tm+1) tiles with R = BM/BN.
static inline int gemm_task_tiles(const GemmTask& t) {
    const int tm = t.M / GM_BM, tn = t.N / GM_BN;
    constexpr int R = GM_BM / GM_BN;
    return t.lower_tiles ? R * tm * (tm + 1) / 2 : tm * tn;
}

static inline int gemm_task_tiles_small(const GemmTask& t) {
    const int tm = t.M / GemmSmall::BM, tn = t.N / GemmSmall::BN;
    return t.lower_tiles ? tm * (tm + 1) / 2 : tm * tn;
}

}  // namespace dqgp
