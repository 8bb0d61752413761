// Gram-matrix kernels: projected kernel (outer kernel on Pauli features) and fidelity kernel.
// Replace ProjectedQuantumKernel.evaluate / FidelityKernel.evaluate (reference main.py:118-137, call
// sites main.py:245,1420-1430, agent_riemannian.py:118).  One 64x64 tile of K per CTA; the only HBM
// traffic besides the (tiny) feature tiles is the 8 B/entry store of K, issued as 128-bit stores.
#include "pairwise.cuh"

namespace dqgp {

// ---- DMMA formulation of the projected Gram (same machinery as the fused gradient, grad.cu): -gamma*d^2 from the
// Gram identity on DMMA.8x8x4, 11-instruction table exp, 16-byte stores.  SYM: only lower 64x64 tiles are computed
// and each is stored twice (K and K^T; the transposed stores still fill whole 32-byte sectors), the diagonal is
// exactly outer(0).  d^2 below 4e-15*(|f|^2+|g|^2) snaps to 0 so exact duplicates give exactly outer(0) = 1, as
// direct differences and SciPy's cdist do.
// v1 (direct differences, libm exp; since removed) ran at 22% of the HBM write roofline: 72 FP64 instructions per entry.
template <int OUTER, int SYM>   // 0 rectangular, 1 lower tiles + mirror, 2 lower tiles only (what the factorisation reads)
__global__ void __launch_bounds__(PW_THREADS) gram_projected_dmma_kernel(const double* __restrict__ F1, int n1,
                                                                         const double* __restrict__ F2, int n2, int m,
                                                                         OuterHyp hyp, double* __restrict__ K, int ldk) {
    __shared__ __align__(16) double Fr[PW_TILE * G2_PITCH];
    __shared__ __align__(16) double Fc[PW_TILE * G2_PITCH];
    __shared__ __align__(16) double nr[2 * PW_TILE];
    int bi, bj;
    if (SYM) {
        bi = int((sqrt(8.0 * blockIdx.x + 1.0) - 1.0) * 0.5);
        while ((bi + 1) * (bi + 2) / 2 <= (int)blockIdx.x) ++bi;
        while (bi * (bi + 1) / 2 > (int)blockIdx.x) --bi;
        bj = blockIdx.x - bi * (bi + 1) / 2;
    } else {
        bi = blockIdx.y; bj = blockIdx.x;
    }
    const int row0 = bi * PW_TILE, col0 = bj * PW_TILE;
    const int mp = (m + 3) & ~3;
    {   // stage both tiles (zero padding in k and past the matrix edge) and their squared norms
        const int r = threadIdx.x >> 2, l4 = threadIdx.x & 3;
        const bool vr = row0 + r < n1, vc = col0 + r < n2;
        const double* sr = F1 + (size_t)min(row0 + r, n1 - 1) * m;
        const double* sc = F2 + (size_t)min(col0 + r, n2 - 1) * m;
        double pr = 0.0, pc = 0.0;
        for (int k = l4; k < mp; k += 4) {
            const double a = (k < m && vr) ? sr[k] : 0.0, b = (k < m && vc) ? sc[k] : 0.0;
            Fr[r * G2_PITCH + k] = a; Fc[r * G2_PITCH + k] = b;
            pr = fma(a, a, pr); pc = fma(b, b, pc);
        }
        pr += __shfl_xor_sync(0xffffffffu, pr, 1); pr += __shfl_xor_sync(0xffffffffu, pr, 2);
        pc += __shfl_xor_sync(0xffffffffu, pc, 1); pc += __shfl_xor_sync(0xffffffffu, pc, 2);
        if (l4 == 0) { nr[r] = pr; nr[PW_TILE + r] = pc; }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wr = warp >> 1, wc = warp & 1, g = lane >> 2, t = lane & 3;
    const double gam = (OUTER == DQGP_OUTER_GAUSSIAN) ? hyp.a : 1.0;
    const double a_scale = 2.0 * gam;
    const double tab = exp_table_entry();
    const double* fr = Fr + (wr * 16 + g) * G2_PITCH + t;
    const double* fc = Fc + (wc * 32 + g) * G2_PITCH + t;
    double c[2][4][2], snap[2][4][2];
    {
        const double n0 = nr[wr * 16 + g], n1s = nr[wr * 16 + 8 + g];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            const double2 nc = *reinterpret_cast<const double2*>(&nr[PW_TILE + wc * 32 + cb * 8 + 2 * t]);
            c[0][cb][0] = -gam * (n0 + nc.x); c[0][cb][1] = -gam * (n0 + nc.y);
            c[1][cb][0] = -gam * (n1s + nc.x); c[1][cb][1] = -gam * (n1s + nc.y);
#pragma unroll
            for (int rb = 0; rb < 2; ++rb)
#pragma unroll
                for (int e = 0; e < 2; ++e) snap[rb][cb][e] = 4e-15 * c[rb][cb][e];      // (negative) snap threshold
        }
    }
    for (int kk = 0; kk < (mp >> 2); ++kk) {
        const double a0 = a_scale * fr[kk * 4], a1 = a_scale * fr[8 * G2_PITCH + kk * 4];
        double b[4];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) b[cb] = fc[cb * 8 * G2_PITCH + kk * 4];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            dmma884(c[0][cb][0], c[0][cb][1], a0, b[cb]);
            dmma884(c[1][cb][0], c[1][cb][1], a1, b[cb]);
        }
    }
    const bool vec_ok = ((ldk & 1) == 0) && ((reinterpret_cast<uintptr_t>(K) & 15) == 0);
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        const int r = row0 + wr * 16 + rb * 8 + g;
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            const int cc = col0 + wc * 32 + cb * 8 + 2 * t;
            double v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                double x = c[rb][cb][e];
                x = (x > snap[rb][cb][e]) ? 0.0 : x;                 // |gamma d^2| below rounding level (or negative d^2) -> 0
                if (SYM && r == cc + e) x = 0.0;
                v[e] = outer_from_neg_gd2<OUTER>(x, hyp, tab);
                // NaN features (arccos outside [-1,1]) must propagate as in NumPy: the clamps above would swallow them
                if (snap[rb][cb][e] != snap[rb][cb][e]) v[e] = snap[rb][cb][e];
            }
            if (r < n1) {
                double* dst = K + (size_t)r * ldk + cc;
                if (vec_ok && cc + 1 < n2) *reinterpret_cast<double2*>(dst) = make_double2(v[0], v[1]);
                else { if (cc < n2) dst[0] = v[0]; if (cc + 1 < n2) dst[1] = v[1]; }
            }
            if (SYM == 1 && bi != bj) {                               // mirror: K[c][r]
                if (cc < n1 && r < n2) K[(size_t)cc * ldk + r] = v[0];
                if (cc + 1 < n1 && r < n2) K[(size_t)(cc + 1) * ldk + r] = v[1];
            }
        }
    }
}

__global__ void add_diagonal_kernel(double* A, int n, int lda, double v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(size_t)i * lda + i] += v;
}

}  // namespace dqgp

extern "C" {

int dqgp_gram_projected(int outer, const double* h_hyp, const double* d_F1, int n1, const double* d_F2, int n2, int m,
                        double* d_K, int ldk, int same, void* stream) {
    using namespace dqgp;
    if (n1 == 0 || n2 == 0) return 0;
    DQGP_REQUIRE(d_F1 && d_F2 && d_K, "dqgp_gram_projected: NULL argument");
    DQGP_REQUIRE(m >= 1 && m <= PW_MAX_M, "dqgp_gram_projected: feature count %d outside [1,%d]", m, PW_MAX_M);
    DQGP_REQUIRE(n1 >= 0 && n2 >= 0 && ldk >= n2, "dqgp_gram_projected: bad shape (%d,%d) ld %d", n1, n2, ldk);
    OuterHyp hyp;
    if (make_outer_hyp(outer, h_hyp, &hyp)) return -1;
    if (n1 == 0 || n2 == 0) return 0;
    dim3 grid((n2 + PW_TILE - 1) / PW_TILE, (n1 + PW_TILE - 1) / PW_TILE);
    cudaStream_t st = as_stream(stream);
    const bool sym = same && d_F1 == d_F2 && n1 == n2;
    const int tsym = grid.y * (grid.y + 1) / 2;
#define DQGP_GRAM(OUT)                                                                                                     \
    do {                                                                                                                   \
        if (sym && same == 2) gram_projected_dmma_kernel<OUT, 2><<<tsym, PW_THREADS, 0, st>>>(d_F1, n1, d_F2, n2, m, hyp, d_K, ldk); \
        else if (sym) gram_projected_dmma_kernel<OUT, 1><<<tsym, PW_THREADS, 0, st>>>(d_F1, n1, d_F2, n2, m, hyp, d_K, ldk); \
        else gram_projected_dmma_kernel<OUT, 0><<<grid, PW_THREADS, 0, st>>>(d_F1, n1, d_F2, n2, m, hyp, d_K, ldk);        \
    } while (0)
    switch (outer) {
        case DQGP_OUTER_GAUSSIAN: DQGP_GRAM(DQGP_OUTER_GAUSSIAN); break;
        case DQGP_OUTER_MATERN15: DQGP_GRAM(DQGP_OUTER_MATERN15); break;
        default: DQGP_GRAM(DQGP_OUTER_EXPSINE2); break;
    }
#undef DQGP_GRAM
    DQGP_LAUNCH_CHECK("gram_projected_dmma_kernel");
    return 0;
}

int dqgp_gram_fidelity(const double* d_Psi1, int n1, const double* d_Psi2, int n2, int dim, double* d_K, int ldk, int same,
                       void* stream) {
    using namespace dqgp;
    (void)same;
    if (n1 == 0 || n2 == 0) return 0;
    DQGP_REQUIRE(d_Psi1 && d_Psi2 && d_K, "dqgp_gram_fidelity: NULL argument");
    DQGP_REQUIRE(n1 >= 0 && n2 >= 0 && ldk >= n2, "dqgp_gram_fidelity: bad shape");
    DQGP_REQUIRE(dim >= 2 && dim <= (1 << MAX_QUBITS) && (dim & (dim - 1)) == 0,
                 "dqgp_gram_fidelity: dim %d is not 2^q amplitudes with 1 <= q <= %d", dim, MAX_QUBITS);
    DQGP_REQUIRE(((reinterpret_cast<uintptr_t>(d_Psi1) | reinterpret_cast<uintptr_t>(d_Psi2)) & 15) == 0,
                 "dqgp_gram_fidelity: state arrays must be 16-byte aligned");
    if (n1 == 0 || n2 == 0) return 0;
    return fidelity_gram_dmma(d_Psi1, n1, d_Psi2, n2, dim, d_K, ldk, as_stream(stream));
}

int dqgp_add_diagonal(double* d_A, int n, int lda, double value, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_A && n >= 0 && lda >= n, "dqgp_add_diagonal: bad arguments");
    if (n == 0) return 0;
    add_diagonal_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(d_A, n, lda, value);
    DQGP_LAUNCH_CHECK("add_diagonal_kernel");
    return 0;
}
}
