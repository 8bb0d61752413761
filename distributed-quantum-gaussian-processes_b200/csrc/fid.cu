// Fidelity kernel on the DMMA path: K[j][k] = |<psi2_k | psi1_j>|^2 as a complex tile contraction.
// A state of 2^q complex128 amplitudes is a real vector u of 2*2^q doubles (re, im interleaved):
//   Re<psi_k|psi_j> = u_j . u_k          Im<psi_k|psi_j> = J(u_j) . u_k,   J(u)[2i] = u[2i+1], J(u)[2i+1] = -u[2i]
// so one tile needs two real GEMMs that share the column operand; both run on DMMA.8x8x4 with the J-variant of the
// row fragment read from the same shared-memory tile at index t^1 with a sign flip (no extra staging, no extra HBM).
// MODE 0 writes the Gram (FidelityKernel.evaluate, reference main.py:118-124); MODE 1 is the fused central-difference
// gradient over the 2P shifted state sets (agent_riemannian.py:270-275,431-436), lower tiles only, B = A^-1 - alpha
// alpha^T in registers, deterministic two-stage reduction.  MODE 2 is the first stage of the analytic gradient for
// 2^q >= 128 (grad.cu): over the lower tiles of one state set it writes W = B o S, S_jk = <psi_k|psi_j>, as the real
// matrix [W_re | W_im] (row stride ldk = 2 n_pad) together with each off-diagonal tile's mirror (W_re symmetric, W_im
// antisymmetric).  Operand chunks of 32 doubles stream through a double-buffered ring filled by the TMA engine.
#include <cstring>
#include "pairwise.cuh"
#include "tensormap.cuh"

namespace dqgp {

constexpr int FD_KC = 32;                      // doubles per k-chunk (16 complex amplitudes)
constexpr int FD_PITCH = FD_KC + 4;            // = 4 (mod 16): conflict-free fragment loads
constexpr int FD_STAGE = 2 * PW_TILE * FD_PITCH;
constexpr size_t FD_SMEM = sizeof(double) * 2 * FD_STAGE;

// MODE 0 (two state arrays): one chunk through the bulk-copy (TMA) engine, one cp.async.bulk per state row (kc doubles, a multiple of
// 16 bytes from a 16-byte aligned row), bytes counted on `bar`
__device__ __forceinline__ void fd_stage_bulk(double* buf, const double* __restrict__ S1, const double* __restrict__ S2, int row0,
                                              int col0, int n1, int n2, int d2, int k0, int kc, unsigned long long* bar) {
    if (threadIdx.x == 0) mbar_arrive_expect_tx(bar, 2u * PW_TILE * kc * sizeof(double));
    if (threadIdx.x < 2 * PW_TILE) {
        const int r = threadIdx.x & (PW_TILE - 1), is_col = threadIdx.x >> 6;
        const double* src = is_col ? S2 + (size_t)min(col0 + r, n2 - 1) * d2 + k0 : S1 + (size_t)min(row0 + r, n1 - 1) * d2 + k0;
        bulk_copy_g2s(buf + (is_col * PW_TILE + r) * FD_PITCH, src, kc * sizeof(double), bar);
    }
}

// MODE 1 and 2 (one state array): the chunk as two boxes of a 3-D tensor map over Psi = [set][state][2 * 2^q doubles] (TMA proper, SASS UTMALDG), issued by one thread: box =
// 64 states x FD_PITCH doubles starting at the chunk; the four doubles beyond the chunk land in the padding of the fragment layout (never
// read), states beyond n arrive as zero rows (their bracket weights are zero).
__device__ __forceinline__ void fd_stage_tmap(double* buf, const void* tmap, int set, int row0, int col0, int k0, unsigned long long* bar) {
    if (threadIdx.x == 0) {
        mbar_arrive_expect_tx(bar, 2u * PW_TILE * FD_PITCH * sizeof(double));
        tensor_copy_3d_g2s(buf, tmap, k0, row0, set, bar);
        tensor_copy_3d_g2s(buf + PW_TILE * FD_PITCH, tmap, k0, col0, set, bar);
    }
}

// dim = 2^q amplitudes (d2 = 2 dim doubles, q >= 1) and 16-byte aligned states: the host entry points check both
template <int MODE>
__global__ void __launch_bounds__(PW_THREADS, 1) fidelity_dmma_kernel(const double* __restrict__ Psi1, int n1,
                                                                      const double* __restrict__ Psi2, int n2, int d2, int n_sets,
                                                                      double* __restrict__ K, int ldk,
                                                                      const double* __restrict__ Ainv, int ld,
                                                                      const double* __restrict__ alpha, int P,
                                                                      double* __restrict__ partial,
                                                                      const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(128) double fd_smem[];
    __shared__ double s_red[2][PW_THREADS / 32];
    __shared__ __align__(8) unsigned long long s_bar[2];
    if (threadIdx.x == 0) { mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_fence_init(); }
    __syncthreads();
    int bi, bj;
    if (MODE != 0) {
        bi = int((sqrt(8.0 * blockIdx.x + 1.0) - 1.0) * 0.5);
        while ((bi + 1) * (bi + 2) / 2 <= (int)blockIdx.x) ++bi;
        while (bi * (bi + 1) / 2 > (int)blockIdx.x) --bi;
        bj = blockIdx.x - bi * (bi + 1) / 2;
    } else {
        bi = blockIdx.y; bj = blockIdx.x;
    }
    const int row0 = bi * PW_TILE, col0 = bj * PW_TILE;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wr = warp >> 1, wc = warp & 1, g = lane >> 2, t = lane & 3;
    const int kc = d2 < FD_KC ? d2 : FD_KC;
    const int n_chunks = d2 / kc;
    const double jsign = (t & 1) ? -1.0 : 1.0;

    double br[2][4][2];
    if (MODE != 0) {
        const double weight = (MODE == 2 || bi == bj) ? 1.0 : 2.0;
#pragma unroll
        for (int rb = 0; rb < 2; ++rb) {
            const int r = row0 + wr * 16 + rb * 8 + g;
            const double ar = (r < n1) ? alpha[r] : 0.0;
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                const int c = col0 + wc * 32 + cb * 8 + 2 * t;
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    br[rb][cb][e] = (r < n1 && c + e < n1) ? weight * (Ainv[(size_t)r * ld + c + e] - ar * alpha[c + e]) : 0.0;
            }
        }
    }

    const size_t set_stride1 = (size_t)n1 * d2, set_stride2 = (size_t)n2 * d2;
    const int first_set = (MODE == 1) ? 1 : 0;
    const int total = n_sets * n_chunks;
    if (MODE != 0) fd_stage_tmap(fd_smem, &tmap, first_set, row0, col0, 0, &s_bar[0]);
    else fd_stage_bulk(fd_smem, Psi1 + first_set * set_stride1, Psi2 + first_set * set_stride2, row0, col0, n1, n2, d2, 0, kc, &s_bar[0]);
    double re[2][4][2], im[2][4][2];
    double pplus = 0.0;
    for (int it = 0; it < total; ++it) {
        const int set = it / n_chunks, ch = it - set * n_chunks;
        mbar_wait(&s_bar[it & 1], (it >> 1) & 1);
        __syncthreads();
        if (MODE == 1 && ch == 0 && set >= 2 && (set & 1) == 0 && threadIdx.x == 0) {
            const int i = (set >> 1) - 1;
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < PW_THREADS / 32; ++w) s += s_red[i & 1][w];
            partial[(size_t)blockIdx.x * P + i] = s;
        }
        if (it + 1 < total) {
            const int ns = (it + 1) / n_chunks, nch = (it + 1) - ns * n_chunks;
            if (MODE != 0)
                fd_stage_tmap(fd_smem + ((it + 1) & 1) * FD_STAGE, &tmap, first_set + ns, row0, col0, nch * kc, &s_bar[(it + 1) & 1]);
            else
                fd_stage_bulk(fd_smem + ((it + 1) & 1) * FD_STAGE, Psi1 + (size_t)(first_set + ns) * set_stride1,
                              Psi2 + (size_t)(first_set + ns) * set_stride2, row0, col0, n1, n2, d2, nch * kc, kc, &s_bar[(it + 1) & 1]);
        }
        if (ch == 0) {
#pragma unroll
            for (int rb = 0; rb < 2; ++rb)
#pragma unroll
                for (int cb = 0; cb < 4; ++cb) re[rb][cb][0] = re[rb][cb][1] = im[rb][cb][0] = im[rb][cb][1] = 0.0;
        }
        const double* buf = fd_smem + (it & 1) * FD_STAGE;
        const double* fr = buf + (wr * 16 + g) * FD_PITCH;
        const double* fc = buf + PW_TILE * FD_PITCH + (wc * 32 + g) * FD_PITCH + t;
        for (int kk = 0; kk < (kc >> 2); ++kk) {
            const double a0 = fr[kk * 4 + t], a1 = fr[8 * FD_PITCH + kk * 4 + t];
            const double j0 = jsign * fr[kk * 4 + (t ^ 1)], j1 = jsign * fr[8 * FD_PITCH + kk * 4 + (t ^ 1)];
            double b[4];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) b[cb] = fc[cb * 8 * FD_PITCH + kk * 4];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                dmma884(re[0][cb][0], re[0][cb][1], a0, b[cb]);
                dmma884(re[1][cb][0], re[1][cb][1], a1, b[cb]);
                dmma884(im[0][cb][0], im[0][cb][1], j0, b[cb]);
                dmma884(im[1][cb][0], im[1][cb][1], j1, b[cb]);
            }
        }
        if (ch == n_chunks - 1) {
            if (MODE == 0) {
#pragma unroll
                for (int rb = 0; rb < 2; ++rb) {
                    const int r = row0 + wr * 16 + rb * 8 + g;
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) {
                        const int c = col0 + wc * 32 + cb * 8 + 2 * t;
#pragma unroll
                        for (int e = 0; e < 2; ++e)
                            if (r < n1 && c + e < n2)
                                K[(size_t)r * ldk + c + e] = fma(re[rb][cb][e], re[rb][cb][e], im[rb][cb][e] * im[rb][cb][e]);
                    }
                }
            } else if (MODE == 2) {
                // every row and column below n_pad = ldk / 2 is written: states past n arrive as zero rows and B is zero there.
                // A diagonal tile computes all its entries itself (no mirror: two writers of one entry would race).
                const int npad = ldk >> 1;
#pragma unroll
                for (int rb = 0; rb < 2; ++rb) {
                    const int r = row0 + wr * 16 + rb * 8 + g;
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb) {
                        const int c = col0 + wc * 32 + cb * 8 + 2 * t;
                        const double2 wre = make_double2(br[rb][cb][0] * re[rb][cb][0], br[rb][cb][1] * re[rb][cb][1]);
                        const double2 wim = make_double2(br[rb][cb][0] * im[rb][cb][0], br[rb][cb][1] * im[rb][cb][1]);
                        *reinterpret_cast<double2*>(K + (size_t)r * ldk + c) = wre;
                        *reinterpret_cast<double2*>(K + (size_t)r * ldk + npad + c) = wim;
                        if (bi != bj) {
                            K[(size_t)c * ldk + r] = wre.x;
                            K[(size_t)(c + 1) * ldk + r] = wre.y;
                            K[(size_t)c * ldk + npad + r] = -wim.x;
                            K[(size_t)(c + 1) * ldk + npad + r] = -wim.y;
                        }
                    }
                }
            } else {
                double part = 0.0;
#pragma unroll
                for (int rb = 0; rb < 2; ++rb)
#pragma unroll
                    for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                        for (int e = 0; e < 2; ++e)
                            part = fma(br[rb][cb][e], fma(re[rb][cb][e], re[rb][cb][e], im[rb][cb][e] * im[rb][cb][e]), part);
                if (set & 1) {
                    const double v = warp_sum(pplus - part);
                    if (lane == 0) s_red[(set >> 1) & 1][warp] = v;
                } else {
                    pplus = part;
                }
            }
        }
    }
    if (MODE == 1) {
        __syncthreads();
        if (threadIdx.x == 0) {
            const int i = P - 1;
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < PW_THREADS / 32; ++w) s += s_red[i & 1][w];
            partial[(size_t)blockIdx.x * P + i] = s;
        }
    }
}

static int fd_attr() {
    static bool done_dev[64] = {false};      // the attribute is per DEVICE
    int dev = 0;
    cudaGetDevice(&dev);
    bool& done = done_dev[(dev >= 0 && dev < 64) ? dev : 0];
    if (!done) {
        DQGP_CUDA(cudaFuncSetAttribute(fidelity_dmma_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FD_SMEM));
        DQGP_CUDA(cudaFuncSetAttribute(fidelity_dmma_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FD_SMEM));
        DQGP_CUDA(cudaFuncSetAttribute(fidelity_dmma_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FD_SMEM));
        done = true;
    }
    return 0;
}

int fidelity_gram_dmma(const double* Psi1, int n1, const double* Psi2, int n2, int dim, double* K, int ldk, cudaStream_t st) {
    int rc = fd_attr();
    if (rc) return rc;
    dim3 grid((n2 + PW_TILE - 1) / PW_TILE, (n1 + PW_TILE - 1) / PW_TILE);
    CUtensorMap tmap;                                                       // unused by the Gram (two state arrays): per-row bulk copies
    memset(&tmap, 0, sizeof(tmap));
    fidelity_dmma_kernel<0><<<grid, PW_THREADS, FD_SMEM, st>>>(Psi1, n1, Psi2, n2, 2 * dim, 1, K, ldk, nullptr, 0, nullptr, 0, nullptr, tmap);
    DQGP_LAUNCH_CHECK("fidelity_dmma_kernel<0>");
    return 0;
}

int fidelity_grad_dmma(const double* Ainv, int ld, const double* alpha, const double* Psi, int n, int dim, int P, double* partial,
                       int tiles, cudaStream_t st) {
    int rc = fd_attr();
    if (rc) return rc;
    // the state tiles of a parameter set as two boxes of a 3-D tensor map (one issuing thread).  For the arguments the entry point
    // accepts (16-byte aligned base, 16 dim-byte rows, box of 36 x 64, dimensions below 2^32) the driver has no reason to refuse it.
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    DQGP_REQUIRE(make_rows_tensor_map(&tmap, Psi, 2 * dim, n, 2 * P + 1, FD_PITCH, PW_TILE),
                 "dqgp_grad_fidelity: the driver refused the tensor map of the states (n %d, dim %d, P %d)", n, dim, P);
    fidelity_dmma_kernel<1><<<tiles, PW_THREADS, FD_SMEM, st>>>(Psi, n, Psi, n, 2 * dim, 2 * P, nullptr, 0, Ainv, ld, alpha, P, partial, tmap);
    DQGP_LAUNCH_CHECK("fidelity_dmma_kernel<1>");
    return 0;
}

int fidelity_weights_dmma(const double* Ainv, int ld, const double* alpha, const double* Psi, int n, int dim, double* W, int n_pad,
                          cudaStream_t st) {
    int rc = fd_attr();
    if (rc) return rc;
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    DQGP_REQUIRE(make_rows_tensor_map(&tmap, Psi, 2 * dim, n, 1, FD_PITCH, PW_TILE),
                 "dqgp_grad_fidelity_analytic: the driver refused the tensor map of the states (n %d, dim %d)", n, dim);
    const int t = n_pad / PW_TILE;
    fidelity_dmma_kernel<2><<<t * (t + 1) / 2, PW_THREADS, FD_SMEM, st>>>(Psi, n, Psi, n, 2 * dim, 1, W, 2 * n_pad, Ainv, ld, alpha, 0,
                                                                         nullptr, tmap);
    DQGP_LAUNCH_CHECK("fidelity_dmma_kernel<2>");
    return 0;
}

}  // namespace dqgp
