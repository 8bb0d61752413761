// Fused central-difference gradient of the GP negative log marginal likelihood.
//   grad_i = 1/2 * sum_jk (A^-1 - alpha alpha^T)_jk * (K(p + h e_i) - K(p - h e_i))_kj / (2h)
// Replaces agent_riemannian.py:270-275 (the (P,n,n) dK tensor, 64 GB/agent at config 5) and :431-436 (the
// Python loop of n^2 elementwise products): no shifted Gram is ever written.  A CTA owns one 64x64 tile
// (lower tiles only; off-diagonal tiles weigh 2 by symmetry), keeps its tile of B = A^-1 - alpha alpha^T in
// registers, and loops over the 2P shifted feature sets staged through shared memory, evaluating the outer
// kernel and contracting on the fly.  Partial sums go to partial[tile][i]; a second kernel adds them in a
// fixed order, so the result is bit-reproducible run to run (the reference rounds it to 4 decimals).
// Bound: FP64 pipe (3m + outer-kernel flops per entry, SURVEY §8(d)); HBM traffic is one read of A^-1.
#include <algorithm>
#include <cstring>
#include "gemm64.cuh"
#include "pairwise.cuh"
#include "tensormap.cuh"

namespace dqgp {

__device__ __forceinline__ void tile_from_index(int local, int& bi, int& bj) {
    bi = int((sqrt(8.0 * local + 1.0) - 1.0) * 0.5);
    while ((bi + 1) * (bi + 2) / 2 <= local) ++bi;
    while (bi * (bi + 1) / 2 > local) --bi;
    bj = local - bi * (bi + 1) / 2;
}

// ---- v2: Gram-identity formulation on the DMMA pipe ---------------------------------------------------------------
// -gamma*||f-g||^2 = 2*gamma*f.g - gamma*||f||^2 - gamma*||g||^2: the accumulator of an 8x8 DMMA block is
// initialised with the (pre-scaled) norms, the row operand is scaled by 2*gamma at fragment load, and m/4
// DMMA.8x8x4 steps leave -gamma*d^2 in the accumulator, which goes straight into fast_exp.  Per entry that
// is 1 DADD + m MACs + 16 (exp) + 1 DFMA (contraction with B) on the FP64 pipe instead of 2m + 23 + 1 for the
// direct-difference form (the absolute error of d^2 is ~1e-15, harmless for exp/Matern/ExpSine outer kernels;
// the unshifted Gram that is *written* keeps direct differences).  CTA = 64x64 tile, 8 warps as 4x2, warp tile
// 16x32 = 2x4 DMMA blocks; B stays in registers for all 2P sets; feature tiles double-buffered.
constexpr int G2_STAGES = 2;
constexpr int G2_STAGE_DOUBLES = 2 * PW_TILE * G2_PITCH + 2 * PW_TILE;
constexpr size_t G2_SMEM = sizeof(double) * G2_STAGES * G2_STAGE_DOUBLES;
static_assert(PW_MAX_M <= G2_PITCH, "a staged sample row holds every feature");

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
    unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(gmem));
}

__device__ __forceinline__ void g2_stage_norms(double* nr, const double* __restrict__ Ns, int row0, int col0, int n) {
    if (threadIdx.x < PW_TILE) cp_async8(&nr[threadIdx.x], &Ns[min(row0 + threadIdx.x, n - 1)]);
    else if (threadIdx.x < 2 * PW_TILE) cp_async8(&nr[threadIdx.x], &Ns[min(col0 + threadIdx.x - PW_TILE, n - 1)]);
}

// Stage one parameter set's row and column feature tiles (64 x m each) + their squared norms with per-thread 8-byte cp.async: four
// threads per sample row, thread (row = tid>>2, lane4 = tid&3) copies features lane4, lane4+4, ... of its row.  Any m, any alignment.
__device__ __forceinline__ void g2_stage(double* buf, const double* __restrict__ Fs, const double* __restrict__ Ns, int row0, int col0,
                                         int n, int m) {
    const int r = threadIdx.x >> 2, l4 = threadIdx.x & 3;
    const double* src_r = Fs + (size_t)min(row0 + r, n - 1) * m;
    const double* src_c = Fs + (size_t)min(col0 + r, n - 1) * m;
    double* dst_r = buf + r * G2_PITCH;
    double* dst_c = buf + PW_TILE * G2_PITCH + r * G2_PITCH;
    for (int k = l4; k < m; k += 4) {
        cp_async8(dst_r + k, src_r + k);
        cp_async8(dst_c + k, src_c + k);
    }
    g2_stage_norms(buf + 2 * PW_TILE * G2_PITCH, Ns, row0, col0, n);
}

// Same tile as TWO boxes of a 3-D tensor map over F = [set][sample][feature] (TMA proper, SASS UTMALDG), issued by one thread: box =
// 64 samples x G2_PITCH features, so the features beyond m - outside the tensor - arrive as the zero padding of the fragment layout,
// and samples beyond n as zero rows (their bracket weights are zero).
__device__ __forceinline__ void g2_stage_tmap(double* buf, const void* tmap, int set, const double* __restrict__ Ns, int row0, int col0, int n,
                                              unsigned long long* bar) {
    if (threadIdx.x == 0) {
        mbar_arrive_expect_tx(bar, 2u * PW_TILE * G2_PITCH * sizeof(double));
        tensor_copy_3d_g2s(buf, tmap, 0, row0, set, bar);
        tensor_copy_3d_g2s(buf + PW_TILE * G2_PITCH, tmap, 0, col0, set, bar);
    }
    g2_stage_norms(buf + 2 * PW_TILE * G2_PITCH, Ns, row0, col0, n);
}

// CLAMP: guard the exponent against arguments below -700 (only reachable when gamma * 4m > 700; features lie in [-1, 1])
// TMAP: the feature tiles of a parameter set arrive as two boxes of the tensor map `tmap`, completion counted on an mbarrier per stage;
// otherwise per-thread cp.async (g2_stage)
// G2_PITCH: doubles per staged sample row, = 4 (mod 8) so the DMMA fragment loads are bank-conflict-free, >= m.  (Pitch 28 with three
// stages, the copy issued two sets ahead, measured 1% slower at config 4: 8.74 against 8.63 ms; the copy is hidden one set ahead.)
template <int OUTER, bool CLAMP, bool TMAP>
__global__ void __launch_bounds__(PW_THREADS, 2) grad_projected_dmma_kernel(const double* __restrict__ Ainv, int ld,
                                                                           const double* __restrict__ alpha,
                                                                           const double* __restrict__ F,
                                                                           const double* __restrict__ Nrm, int n, int m, int P,
                                                                           OuterHyp hyp, double* __restrict__ partial,
                                                                           const __grid_constant__ CUtensorMap tmap) {
    constexpr int STAGES = G2_STAGES, PITCH = G2_PITCH;
    extern __shared__ __align__(128) double g2_smem[];
    __shared__ double s_red[2][PW_THREADS / 32];
    __shared__ __align__(8) unsigned long long s_bar[STAGES];
    int bi, bj;
    tile_from_index(blockIdx.x, bi, bj);
    const int row0 = bi * PW_TILE, col0 = bj * PW_TILE;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wr = warp >> 1, wc = warp & 1, g = lane >> 2, t = lane & 3;
    const int ksteps = (m + 3) >> 2;
    if (TMAP) {
        if (threadIdx.x == 0) { mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_fence_init(); }
        __syncthreads();
    }
    constexpr bool STAT = outer_is_stationary(OUTER);
    const double gam = (OUTER == DQGP_OUTER_GAUSSIAN) ? hyp.a * DQGP_EXP_S32 : 1.0;      // Gaussian: argument in units of ln2/32
    const double a_scale = STAT ? 2.0 * gam : 1.0;                                      // dot product: sigma_0^2 + f.g
    const double tab = exp_table_entry();

    // zero the k-padding columns of both stages once (cp.async never writes them; the tensor map's boxes bring their own zeros)
    for (int e = threadIdx.x; !TMAP && e < STAGES * 2 * PW_TILE * (PITCH - m); e += PW_THREADS) {
        const int per = PITCH - m;
        const int row = e / per, k = m + (e - row * per);          // row in [0, 4*64): stage x operand x sample
        const int stage = row / (2 * PW_TILE), rr = row - stage * 2 * PW_TILE;
        g2_smem[stage * G2_STAGE_DOUBLES + rr * PITCH + k] = 0.0;
    }

    // B = weight * (A^-1 - alpha alpha^T) for this lane's 16 entries; zero outside the matrix, and on the diagonal where k(f, f) = 1
    // does not depend on the parameters (the dot product's sigma_0^2 + |f|^2 does)
    double br[2][4][2];
    const double weight = (bi == bj) ? 1.0 : 2.0;
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        const int r = row0 + wr * 16 + rb * 8 + g;
        const double ar = (r < n) ? alpha[r] : 0.0;
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            const int c = col0 + wc * 32 + cb * 8 + 2 * t;
#pragma unroll
            for (int e = 0; e < 2; ++e)
                br[rb][cb][e] = (r < n && c + e < n && (!STAT || r != c + e)) ? weight * (Ainv[(size_t)r * ld + c + e] - ar * alpha[c + e]) : 0.0;
        }
    }

    const size_t set_stride = (size_t)n * m;
    const int T = 2 * P;
    if (TMAP) g2_stage_tmap(g2_smem, &tmap, 1, Nrm + n, row0, col0, n, &s_bar[0]);
    else g2_stage(g2_smem, F + set_stride, Nrm + n, row0, col0, n, m);
    cp_async_commit();
    double pplus = 0.0, pminus = 0.0;
    for (int tt = 0; tt < T; ++tt) {
        const int cur = tt % STAGES;
        cp_async_wait<0>();
        if (TMAP) mbar_wait(&s_bar[cur], (tt / STAGES) & 1);
        __syncthreads();
        if (tt >= 2 && (tt & 1) == 0 && threadIdx.x == 0) {
            const int i = (tt >> 1) - 1;
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < PW_THREADS / 32; ++w) s += s_red[i & 1][w];
            partial[(size_t)blockIdx.x * P + i] = s;
        }
        {
            const int nx = tt + STAGES - 1;          // the set whose copy is issued now; its stage was last read at iteration tt - 1
            if (nx < T) {
                const int ns = nx % STAGES;
                if (TMAP) g2_stage_tmap(g2_smem + ns * G2_STAGE_DOUBLES, &tmap, nx + 1, Nrm + (size_t)(nx + 1) * n, row0, col0, n, &s_bar[ns]);
                else g2_stage(g2_smem + ns * G2_STAGE_DOUBLES, F + (size_t)(nx + 1) * set_stride, Nrm + (size_t)(nx + 1) * n, row0, col0, n, m);
            }
        }
        cp_async_commit();
        const double* buf = g2_smem + cur * G2_STAGE_DOUBLES;
        const double* Fr = buf + (wr * 16 + g) * PITCH + t;
        const double* Fc = buf + PW_TILE * PITCH + (wc * 32 + g) * PITCH + t;
        const double* nr = buf + 2 * PW_TILE * PITCH;
        double c[2][4][2];
        {
            const double n0 = nr[wr * 16 + g], n1 = nr[wr * 16 + 8 + g];            // already -gamma_eff |f|^2 (dot product: sigma_0^2 / 2)
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                const double2 nc = *reinterpret_cast<const double2*>(&nr[PW_TILE + wc * 32 + cb * 8 + 2 * t]);
                const double m0 = nc.x, m1 = nc.y;
                c[0][cb][0] = n0 + m0; c[0][cb][1] = n0 + m1;
                c[1][cb][0] = n1 + m0; c[1][cb][1] = n1 + m1;
            }
        }
#pragma unroll 2
        for (int kk = 0; kk < ksteps; ++kk) {
            const double a0 = a_scale * Fr[kk * 4], a1 = a_scale * Fr[8 * PITCH + kk * 4];
            double b[4];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) b[cb] = Fc[cb * 8 * PITCH + kk * 4];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                dmma884(c[0][cb][0], c[0][cb][1], a0, b[cb]);
                dmma884(c[1][cb][0], c[1][cb][1], a1, b[cb]);
            }
        }
        double part = 0.0;
#pragma unroll
        for (int rb = 0; rb < 2; ++rb)
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double kv = outer_grad_from_neg_gd2<OUTER, CLAMP>(c[rb][cb][e], hyp, tab);
                    part = fma(br[rb][cb][e], kv, part);
                }
        if (tt & 1) {
            pminus = part;
            double v = warp_sum(pplus - pminus);
            if (lane == 0) s_red[(tt >> 1) & 1][warp] = v;
        } else {
            pplus = part;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int i = P - 1;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < PW_THREADS / 32; ++w) s += s_red[i & 1][w];
        partial[(size_t)blockIdx.x * P + i] = s;
    }
}

// squared norms of every feature row: Nrm[s*n + j] = sum_k F[s][j][k]^2 (one warp per 4 rows)
__global__ void feature_norms_kernel(const double* __restrict__ F, long long rows, int m, double scale, double* __restrict__ Nrm) {
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    const double* f = F + row * m;
    double acc = 0.0;
    for (int k = 0; k < m; ++k) acc = fma(f[k], f[k], acc);
    Nrm[row] = scale * acc;
}

// grad[i] = scale * sum_tiles partial[tile][i], fixed summation order (strided per thread, then a fixed tree)
__global__ void __launch_bounds__(256) grad_reduce_kernel(const double* __restrict__ partial, int n_tiles, int P, double scale,
                                                          double* __restrict__ grad) {
    __shared__ double s[256];
    const int i = blockIdx.x;
    double acc = 0.0;
    for (int t = threadIdx.x; t < n_tiles; t += 256) acc += partial[(size_t)t * P + i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) grad[i] = scale * s[0];
}

// ---- analytic gradient (opt-in; SURVEY 8(f) row 3: NOT the reference's central difference, Q3) -------------------------------
// With B = A^-1 - alpha alpha^T (symmetric) and a stationary outer kernel K_jk = kappa(|f_j - f_k|^2),
//   grad_i = 1/2 sum_jk B_jk dK_jk/dp_i = 2 sum_j < df_j/dp_i , G_j >,   G_j = sum_k B_jk kappa'(s_jk) (f_j - f_k),
// so ONE pass over the n x n entries (one outer-kernel derivative per entry instead of 2P kernels) gives G (n x m), and the P
// parameters only enter through the feature Jacobian (dqgp_features_jacobian) in an O(P n m) contraction.  The per-pair weight
// is outer_analytic_weight (pairwise.cuh); the Gaussian's weight is e^{-gamma s} and its contraction scale -2 gamma.  The dot
// product K_jk = sigma_0^2 + f_j.f_k gives grad_i = sum_j < df_j/dp_i , (B F)_j >: G_j = sum_k B_jk f_k, diagonal included,
// contraction scale 1.
// grad_analytic_rows_kernel: thread = row r of a column segment; f_r and the running G_r live in registers (M = 3q at compile
// time), the segment's f_c stream through shared memory 64 columns at a time, A^-1 is read through its symmetric image
// A^-1[c][r] so consecutive threads read consecutive addresses.  Fixed summation order: bit-reproducible.
// hyp_a, hyp_b: the OuterHyp fields (hyp_a is the Gaussian's gamma; hyp_b is last so the parameter offsets before it are those
// of a kernel without it).  ALPHA1: see outer_analytic_weight.
constexpr int GA_ROWS = 128, GA_CHUNK = 64, GA_SEGMENTS = 16;

template <int OUTER, int M, bool ALPHA1>
__global__ void __launch_bounds__(GA_ROWS) grad_analytic_rows_kernel(const double* __restrict__ Ainv, int ld, const double* __restrict__ alpha,
                                                                    const double* __restrict__ F, int n, double hyp_a, int seg_cols,
                                                                    double* __restrict__ Gpart, double hyp_b) {
    __shared__ double Fc[GA_CHUNK * M];
    __shared__ double ac[GA_CHUNK];
    const OuterHyp hyp{hyp_a, hyp_b};
    const int r = blockIdx.x * GA_ROWS + threadIdx.x;
    const int c_begin = blockIdx.y * seg_cols, c_end = min(n, c_begin + seg_cols);
    const bool live = r < n;
    double fr[M], h[M];
#pragma unroll
    for (int k = 0; k < M; ++k) { fr[k] = live ? F[(size_t)r * M + k] : 0.0; h[k] = 0.0; }
    const double ar = live ? alpha[r] : 0.0;
    for (int c0 = c_begin; c0 < c_end; c0 += GA_CHUNK) {
        const int cnt = min(GA_CHUNK, c_end - c0);
        __syncthreads();
        for (int e = threadIdx.x; e < cnt * M; e += GA_ROWS) Fc[e] = F[(size_t)c0 * M + e];
        if (threadIdx.x < cnt) ac[threadIdx.x] = alpha[c0 + threadIdx.x];
        __syncthreads();
        if (!live) continue;
        for (int cc = 0; cc < cnt; ++cc) {
            const double* fc = Fc + cc * M;
            if (OUTER == DQGP_OUTER_DOTPRODUCT) {
                const double b = Ainv[(size_t)(c0 + cc) * ld + r] - ar * ac[cc];
#pragma unroll
                for (int k = 0; k < M; ++k) h[k] = fma(b, fc[k], h[k]);
                continue;
            }
            double df[M], d2 = 0.0;
#pragma unroll
            for (int k = 0; k < M; ++k) { df[k] = fr[k] - fc[k]; d2 = fma(df[k], df[k], d2); }
            const double q = (Ainv[(size_t)(c0 + cc) * ld + r] - ar * ac[cc]) * outer_analytic_weight<OUTER, ALPHA1>(d2, hyp);
#pragma unroll
            for (int k = 0; k < M; ++k) h[k] = fma(q, df[k], h[k]);
        }
    }
    if (live) {
        double* dst = Gpart + ((size_t)blockIdx.y * n + r) * M;
#pragma unroll
        for (int k = 0; k < M; ++k) dst[k] = h[k];
    }
}
// G = sum over segments, fixed order
__global__ void grad_analytic_sum_kernel(const double* __restrict__ Gpart, size_t count, int segments, double* __restrict__ G) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= count) return;
    double acc = 0.0;
    for (int sgm = 0; sgm < segments; ++sgm) acc += Gpart[(size_t)sgm * count + e];
    G[e] = acc;
}
// grad[i] = scale * <J_i, G>  (n*m products, strided per thread then a fixed tree)
__global__ void __launch_bounds__(256) grad_analytic_contract_kernel(const double* __restrict__ J, const double* __restrict__ G, size_t count,
                                                                     double scale, double* __restrict__ grad) {
    __shared__ double sred[256];
    const double* Ji = J + (size_t)blockIdx.x * count;
    double acc = 0.0;
    for (size_t e = threadIdx.x; e < count; e += 256) acc = fma(Ji[e], G[e], acc);
    sred[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sred[threadIdx.x] += sred[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) grad[blockIdx.x] = scale * sred[0];
}

// Fidelity kernel, analytic gradient: K_jk = |s_jk|^2, s_jk = <psi_k|psi_j>, and with d_i psi_j from dqgp_states_jacobian
//   grad_i = 1/2 sum_jk B_jk dK_jk/dp_i = 2 Re sum_j < G_j | d_i psi_j >,   G_j = sum_k B_jk s_jk psi_k.
// Thread = row j of a column segment; psi_j and the running G_j live in shared memory (one column per thread, [a][thread]),
// the segment's psi_k stream through shared memory 16 columns at a time.  DIM = 2^q <= 64.
constexpr int GF_ROWS = 64, GF_CHUNK = 16;
template <int DIM>
__global__ void __launch_bounds__(GF_ROWS) grad_fid_analytic_rows_kernel(const double* __restrict__ Ainv, int ld, const double* __restrict__ alpha,
                                                                        const double2* __restrict__ Psi, int n, int seg_cols,
                                                                        double2* __restrict__ Gpart) {
    extern __shared__ __align__(16) double2 gf_smem[];
    double2* sp = gf_smem;                          // psi_j: [DIM][GF_ROWS]
    double2* sg = sp + DIM * GF_ROWS;               // G_j:   [DIM][GF_ROWS]
    double2* sc = sg + DIM * GF_ROWS;               // psi_k chunk: [GF_CHUNK][DIM]
    __shared__ double ac[GF_CHUNK];
    const int tid = threadIdx.x;
    const int j = blockIdx.x * GF_ROWS + tid;
    const bool live = j < n;
    const int c_begin = blockIdx.y * seg_cols, c_end = min(n, c_begin + seg_cols);
    for (int a = 0; a < DIM; ++a) {
        sp[a * GF_ROWS + tid] = live ? Psi[(size_t)j * DIM + a] : make_double2(0.0, 0.0);
        sg[a * GF_ROWS + tid] = make_double2(0.0, 0.0);
    }
    const double aj = live ? alpha[j] : 0.0;
    for (int c0 = c_begin; c0 < c_end; c0 += GF_CHUNK) {
        const int cnt = min(GF_CHUNK, c_end - c0);
        __syncthreads();
        for (int e = tid; e < cnt * DIM; e += GF_ROWS) sc[e] = Psi[(size_t)c0 * DIM + e];
        if (tid < cnt) ac[tid] = alpha[c0 + tid];
        __syncthreads();
        if (!live) continue;
        for (int cc = 0; cc < cnt; ++cc) {
            const double2* pk = sc + cc * DIM;
            double sr = 0.0, si = 0.0;              // s = sum_a conj(psi_k[a]) psi_j[a]
            for (int a = 0; a < DIM; ++a) {
                const double2 u = pk[a], v = sp[a * GF_ROWS + tid];
                sr = fma(u.x, v.x, fma(u.y, v.y, sr));
                si = fma(u.x, v.y, fma(-u.y, v.x, si));
            }
            const double b = Ainv[(size_t)(c0 + cc) * ld + j] - aj * ac[cc];
            const double qr = b * sr, qi = b * si;
            for (int a = 0; a < DIM; ++a) {
                const double2 u = pk[a];
                double2 g = sg[a * GF_ROWS + tid];
                g.x = fma(qr, u.x, fma(-qi, u.y, g.x));
                g.y = fma(qr, u.y, fma(qi, u.x, g.y));
                sg[a * GF_ROWS + tid] = g;
            }
        }
    }
    if (live) {
        double2* dst = Gpart + ((size_t)blockIdx.y * n + j) * DIM;
        for (int a = 0; a < DIM; ++a) dst[a] = sg[a * GF_ROWS + tid];
    }
}

// Fidelity kernel, analytic gradient for 128 <= 2^q <= 4096 as two dense DMMA stages.  With R the states as a real n x 2 dim
// matrix (re, im interleaved) and R~ = R with (re, im) -> (-im, re) per amplitude:
//   1. W = B o S as [W_re | W_im] (fidelity_dmma_kernel<2>, fid.cu);
//   2. G = W_re R + W_im R~ = [W_re | W_im] [R; R~], one real GEMM on the grouped DMMA engine (gemm64.cu);
//   3. grad_i = 2 <D_i, G> over the first n rows, in slices (partial sums in the W region, free after the GEMM).
// Workspace (doubles): the one-task GEMM table, W (n_pad x 2 n_pad), [R; R~] (2 n_pad x 2 dim), G (n_pad x 2 dim), with
// n_pad = n rounded up to the GEMM's 128-row tile.
constexpr int GFD_TABLE = 16;                   // doubles reserved for the GemmTask
static_assert(sizeof(GemmTask) <= GFD_TABLE * sizeof(double), "the GEMM task must fit its workspace slot");
static inline size_t gfd_npad(int n) { return ((size_t)n + GM_BM - 1) / GM_BM * GM_BM; }

// [R; R~] with zero rows past n: row k < n_pad is psi_k, row n_pad + k is J psi_k
__global__ void grad_fid_pack_kernel(const double2* __restrict__ Psi, int n, int dim, int n_pad, double2* __restrict__ RR) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)n_pad * dim) return;
    const size_t k = e / dim;
    const double2 v = k < (size_t)n ? Psi[e] : make_double2(0.0, 0.0);
    RR[e] = v;
    RR[(size_t)n_pad * dim + e] = make_double2(-v.y, v.x);
}
// <D_i, G> in fixed slices of `count`, one CTA per (slice, parameter): P CTAs alone (40 at q = 10) cannot stream P n 2^(q+1) doubles
// of d psi at HBM rate.  partial[slice][i]; grad_reduce_kernel adds the slices in a fixed order.
constexpr int GFD_SLICES = 64;
__global__ void __launch_bounds__(256) grad_fid_contract_kernel(const double* __restrict__ D, const double* __restrict__ G, size_t count, int P,
                                                                double* __restrict__ partial) {
    __shared__ double sred[256];
    const size_t per = (count + gridDim.x - 1) / gridDim.x;
    const size_t b = (size_t)blockIdx.x * per, e = min(count, b + per);
    const double* Di = D + (size_t)blockIdx.y * count;
    double acc = 0.0;
#pragma unroll 4
    for (size_t k = b + threadIdx.x; k < e; k += 256) acc = fma(Di[k], G[k], acc);
    sred[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sred[threadIdx.x] += sred[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[(size_t)blockIdx.x * P + blockIdx.y] = sred[0];
}
// the task table is written on the device so the entry point stays capturable into a CUDA graph (a host copy would synchronise)
__global__ void grad_fid_task_kernel(GemmTask t, GemmTask* __restrict__ dst) { *dst = t; }

// ---- NLL gradient with respect to the outer kernel's hyper-parameters h: dNLL/dh = 1/2 sum_jk B_jk dK_jk/dh, B = A^-1 - alpha alpha^T.
// One CTA per lower 64x64 tile, the Gram kernel's layout: both feature tiles staged once, -d^2 from the Gram identity on DMMA, then
// the Gram's snap-to-zero and diagonal rules (so duplicates and the diagonal see the s = 0 of the K that was factored) and its NaN
// restore.  Entries j > k weigh 2, j = k weighs 1, j < k is never read: A^-1 may be the lower tiles only (want_inverse = 1).
// partial[tile][2] = {c0 sum B w0, c1 sum B w1} (outer_hyper_terms); grad_reduce_kernel adds the tiles in a fixed order.  The dot
// product's terms do not depend on the features: its tiles skip the staging and the DMMA.
template <int OUTER>
__global__ void __launch_bounds__(PW_THREADS) grad_hyper_dmma_kernel(const double* __restrict__ Ainv, int ld, const double* __restrict__ alpha,
                                                                     const double* __restrict__ F, int n, int m, OuterHyp hyp, double c0,
                                                                     double c1, double* __restrict__ partial) {
    __shared__ __align__(16) double Fr[PW_TILE * G2_PITCH];
    __shared__ __align__(16) double Fc[PW_TILE * G2_PITCH];
    __shared__ __align__(16) double nr[2 * PW_TILE];
    __shared__ double s_red[2][PW_THREADS / 32];
    constexpr bool STAT = outer_is_stationary(OUTER);
    int bi, bj;
    tile_from_index(blockIdx.x, bi, bj);
    const int row0 = bi * PW_TILE, col0 = bj * PW_TILE;
    const int mp = (m + 3) & ~3;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wr = warp >> 1, wc = warp & 1, g = lane >> 2, t = lane & 3;
    double c[2][4][2], snap[2][4][2];
    if (STAT) {
        {   // stage both tiles (zero padding in k and past the matrix edge) and their squared norms, as gram_projected_dmma_kernel
            const int r = threadIdx.x >> 2, l4 = threadIdx.x & 3;
            const bool vr = row0 + r < n, vc = col0 + r < n;
            const double* sr = F + (size_t)min(row0 + r, n - 1) * m;
            const double* sc = F + (size_t)min(col0 + r, n - 1) * m;
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
        const double* fr = Fr + (wr * 16 + g) * G2_PITCH + t;
        const double* fc = Fc + (wc * 32 + g) * G2_PITCH + t;
        const double n0 = nr[wr * 16 + g], n1 = nr[wr * 16 + 8 + g];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
            const double2 nc = *reinterpret_cast<const double2*>(&nr[PW_TILE + wc * 32 + cb * 8 + 2 * t]);
            c[0][cb][0] = -(n0 + nc.x); c[0][cb][1] = -(n0 + nc.y);
            c[1][cb][0] = -(n1 + nc.x); c[1][cb][1] = -(n1 + nc.y);
#pragma unroll
            for (int rb = 0; rb < 2; ++rb)
#pragma unroll
                for (int e = 0; e < 2; ++e) snap[rb][cb][e] = 4e-15 * c[rb][cb][e];
        }
        for (int kk = 0; kk < (mp >> 2); ++kk) {           // -d^2 = 2 f.g - |f|^2 - |g|^2
            const double a0 = 2.0 * fr[kk * 4], a1 = 2.0 * fr[8 * G2_PITCH + kk * 4];
            double b[4];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) b[cb] = fc[cb * 8 * G2_PITCH + kk * 4];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb) {
                dmma884(c[0][cb][0], c[0][cb][1], a0, b[cb]);
                dmma884(c[1][cb][0], c[1][cb][1], a1, b[cb]);
            }
        }
    }
    double p0 = 0.0, p1 = 0.0;
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        const int r = row0 + wr * 16 + rb * 8 + g;
        const double ar = r < n ? alpha[r] : 0.0;
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int cc = col0 + wc * 32 + cb * 8 + 2 * t + e;
                if (r >= n || cc > r) continue;
                double w0, w1;
                if (STAT) {
                    double x = c[rb][cb][e];
                    x = (x > snap[rb][cb][e] || r == cc) ? 0.0 : x;
                    outer_hyper_terms<OUTER>(-x, hyp, w0, w1);
                    if (snap[rb][cb][e] != snap[rb][cb][e]) w0 = w1 = snap[rb][cb][e];     // NaN features reach the result
                } else {
                    outer_hyper_terms<OUTER>(0.0, hyp, w0, w1);
                }
                const double bw = (r == cc ? 1.0 : 2.0) * (Ainv[(size_t)r * ld + cc] - ar * alpha[cc]);
                p0 = fma(bw, w0, p0);
                p1 = fma(bw, w1, p1);
            }
        }
    }
    p0 = warp_sum(p0);
    p1 = warp_sum(p1);
    if (lane == 0) { s_red[0][warp] = p0; s_red[1][warp] = p1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int w = 0; w < PW_THREADS / 32; ++w) { s0 += s_red[0][w]; s1 += s_red[1][w]; }
        partial[(size_t)blockIdx.x * 2] = c0 * s0;
        partial[(size_t)blockIdx.x * 2 + 1] = c1 * s1;
    }
}

// out = sigma tr(B) = sigma sum_j (A^-1_jj - alpha_j^2): strided per thread, then a fixed tree
__global__ void __launch_bounds__(256) grad_noise_kernel(const double* __restrict__ Ainv, int ld, const double* __restrict__ alpha, int n,
                                                         double sigma, double* __restrict__ out) {
    __shared__ double s[256];
    double acc = 0.0;
    for (int j = threadIdx.x; j < n; j += 256) acc += Ainv[(size_t)j * ld + j] - alpha[j] * alpha[j];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sigma * s[0];
}

static inline int grad_tiles(int n) {
    const int t = (n + PW_TILE - 1) / PW_TILE;
    return t * (t + 1) / 2;
}

template <int OUTER, bool ALPHA1>
static void launch_grad_analytic_rows(int m, dim3 grid, cudaStream_t st, const double* Ainv, int ld, const double* alpha, const double* F,
                                      int n, const OuterHyp& hyp, int seg_cols, double* Gpart) {
    switch (m / 3) {
#define DQGP_GA(QQ) case QQ: grad_analytic_rows_kernel<OUTER, 3 * QQ, ALPHA1><<<grid, GA_ROWS, 0, st>>>(Ainv, ld, alpha, F, n, hyp.a, seg_cols, Gpart, hyp.b); break;
        DQGP_GA(1) DQGP_GA(2) DQGP_GA(3) DQGP_GA(4) DQGP_GA(5) DQGP_GA(6) DQGP_GA(7) DQGP_GA(8) DQGP_GA(9) DQGP_GA(10) DQGP_GA(11) DQGP_GA(12)
#undef DQGP_GA
    }
}

}  // namespace dqgp

extern "C" {

size_t dqgp_grad_workspace_bytes(int n, int P) {
    if (n <= 0 || P <= 0) return 0;
    // partial sums [tiles][P] followed by the squared feature norms [(2P+1)][n] of the DMMA formulation
    return sizeof(double) * ((size_t)dqgp::grad_tiles(n) * (size_t)P + (size_t)(2 * P + 1) * (size_t)n);
}

int dqgp_grad_projected(int outer, const double* h_hyp, const double* d_Ainv, int ld, const double* d_alpha, const double* d_F,
                        int n, int m, int P, double h, double* d_grad, void* d_work, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Ainv && d_alpha && d_F && d_grad && d_work, "dqgp_grad_projected: NULL argument");
    DQGP_REQUIRE(n >= 1 && ld >= n && P >= 1 && m >= 1 && m <= PW_MAX_M && h != 0.0, "dqgp_grad_projected: bad shape / shift");
    OuterHyp hyp;
    if (make_outer_hyp(outer, h_hyp, &hyp)) return -1;
    const int tiles = grad_tiles(n);
    cudaStream_t st = as_stream(stream);
    double* partial = static_cast<double*>(d_work);
    double* norms = partial + (size_t)tiles * P;
    const long long rows = (long long)(2 * P + 1) * n;
    // the norms arrive pre-multiplied by -gamma_eff (and, Gaussian, by 32/ln2: the exponent's argument then leaves the DMMA in the
    // units its range reduction wants): the kernel only adds them.  The dot product's "norms" are sigma_0^2 / 2 each, so the
    // accumulator starts at exactly sigma_0^2.
    const double gam_eff = (outer == DQGP_OUTER_GAUSSIAN) ? hyp.a * DQGP_EXP_S32 : 1.0;
    if (outer_is_stationary(outer)) feature_norms_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(d_F, rows, m, -gam_eff, norms);
    else launch_self_kernel(nullptr, rows, m, 0.5 * hyp.a, false, norms, st);
    // Pauli features lie in [-1, 1]: gamma d^2 <= 4 m gamma, so the exponent guard is only needed for large gamma
    // the exponent's argument is bounded below by -gamma 4m (Gaussian), -sqrt(3) 2 sqrt(m) / l (Matern), -2 / l^2 (ExpSineSquared)
    const double worst = outer == DQGP_OUTER_GAUSSIAN ? 4.0 * m * hyp.a
                         : outer == DQGP_OUTER_MATERN15 ? 1.7320508075688772 * 2.0 * sqrt((double)m) * hyp.a : 2.0 * hyp.a * hyp.a;
    const bool no_clamp = hyp.a > 0.0 && worst < 650.0;
    // feature tiles as two boxes of a 3-D tensor map per parameter set (one thread issues them); odd m (rows not 16-byte multiples),
    // a misaligned d_F or a map the driver refuses take the per-thread cp.async kernel, with the exponent guard (CLAMP only changes
    // results below -700, where no_clamp is never set, so both kernels give the same gradient)
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    const bool have_tmap = (m & 1) == 0 && (reinterpret_cast<uintptr_t>(d_F) & 15) == 0 &&
                           make_rows_tensor_map(&tmap, d_F, m, n, 2 * P + 1, G2_PITCH, PW_TILE);
#define DQGP_G2(OUT)                                                                                                         \
    do {                                                                                                                     \
        static bool attr_done_dev[64] = {false};        /* the attribute is per DEVICE (as gemm_init's flags) */            \
        int dev_ = 0;                                                                                                        \
        cudaGetDevice(&dev_);                                                                                                \
        bool& attr_done = attr_done_dev[(dev_ >= 0 && dev_ < 64) ? dev_ : 0];                                                \
        if (!attr_done) {                                                                                                    \
            DQGP_CUDA(cudaFuncSetAttribute(grad_projected_dmma_kernel<OUT, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G2_SMEM)); \
            DQGP_CUDA(cudaFuncSetAttribute(grad_projected_dmma_kernel<OUT, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G2_SMEM)); \
            DQGP_CUDA(cudaFuncSetAttribute(grad_projected_dmma_kernel<OUT, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G2_SMEM)); \
            attr_done = true;                                                                                                \
        }                                                                                                                    \
        if (have_tmap && no_clamp) grad_projected_dmma_kernel<OUT, false, true><<<tiles, PW_THREADS, G2_SMEM, st>>>(d_Ainv, ld, d_alpha, d_F, norms, n, m, P, hyp, partial, tmap); \
        else if (have_tmap) grad_projected_dmma_kernel<OUT, true, true><<<tiles, PW_THREADS, G2_SMEM, st>>>(d_Ainv, ld, d_alpha, d_F, norms, n, m, P, hyp, partial, tmap); \
        else grad_projected_dmma_kernel<OUT, true, false><<<tiles, PW_THREADS, G2_SMEM, st>>>(d_Ainv, ld, d_alpha, d_F, norms, n, m, P, hyp, partial, tmap); \
    } while (0)
    // RationalQuadratic and DotProduct have no exponent to guard: only their CLAMP = false kernels exist, one per staging path
#define DQGP_G2_NOEXP(OUT)                                                                                                   \
    do {                                                                                                                     \
        static bool attr_done_dev[64] = {false};                                                                             \
        int dev_ = 0;                                                                                                        \
        cudaGetDevice(&dev_);                                                                                                \
        bool& attr_done = attr_done_dev[(dev_ >= 0 && dev_ < 64) ? dev_ : 0];                                                \
        if (!attr_done) {                                                                                                    \
            DQGP_CUDA(cudaFuncSetAttribute(grad_projected_dmma_kernel<OUT, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G2_SMEM)); \
            DQGP_CUDA(cudaFuncSetAttribute(grad_projected_dmma_kernel<OUT, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G2_SMEM)); \
            attr_done = true;                                                                                                \
        }                                                                                                                    \
        if (have_tmap) grad_projected_dmma_kernel<OUT, false, true><<<tiles, PW_THREADS, G2_SMEM, st>>>(d_Ainv, ld, d_alpha, d_F, norms, n, m, P, hyp, partial, tmap); \
        else grad_projected_dmma_kernel<OUT, false, false><<<tiles, PW_THREADS, G2_SMEM, st>>>(d_Ainv, ld, d_alpha, d_F, norms, n, m, P, hyp, partial, tmap); \
    } while (0)
    switch (outer) {
        case DQGP_OUTER_GAUSSIAN: DQGP_G2(DQGP_OUTER_GAUSSIAN); break;
        case DQGP_OUTER_MATERN15: DQGP_G2(DQGP_OUTER_MATERN15); break;
        case DQGP_OUTER_RATQUAD: DQGP_G2_NOEXP(DQGP_OUTER_RATQUAD); break;
        case DQGP_OUTER_DOTPRODUCT: DQGP_G2_NOEXP(DQGP_OUTER_DOTPRODUCT); break;
        default: DQGP_G2(DQGP_OUTER_EXPSINE2); break;
    }
#undef DQGP_G2_NOEXP
#undef DQGP_G2
    DQGP_LAUNCH_CHECK("grad_projected_dmma_kernel");
    grad_reduce_kernel<<<P, 256, 0, st>>>(partial, tiles, P, 0.5 / (2.0 * h), d_grad);
    DQGP_LAUNCH_CHECK("grad_reduce_kernel");
    return 0;
}

size_t dqgp_grad_outer_hyperparameters_workspace_bytes(int n) {
    if (n <= 0) return 0;
    return sizeof(double) * 2 * (size_t)dqgp::grad_tiles(n);
}

int dqgp_grad_outer_hyperparameters(int outer, const double* h_hyp, const double* d_Ainv, int ld, const double* d_alpha, const double* d_F,
                                    int n, int m, double* d_grad, void* d_work, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Ainv && d_alpha && d_F && d_grad && d_work, "dqgp_grad_outer_hyperparameters: NULL argument");
    DQGP_REQUIRE(n >= 1 && ld >= n && m >= 1 && m <= PW_MAX_M, "dqgp_grad_outer_hyperparameters: bad shape (n %d, ld %d, m %d)", n, ld, m);
    OuterHyp hyp;
    if (make_outer_hyp(outer, h_hyp, &hyp)) return -1;
    // c0, c1 of outer_hyper_terms, from the values as given in h_hyp (NULL = all 1)
    const double pi = 3.14159265358979323846;
    const double h0 = h_hyp ? h_hyp[0] : 1.0;
    double c0 = 1.0, c1 = 0.0;
    int count = 1;
    switch (outer) {
        case DQGP_OUTER_MATERN15: c0 = hyp.a; break;
        case DQGP_OUTER_EXPSINE2: c0 = 4.0 * hyp.a * hyp.a * hyp.a; c1 = 4.0 * hyp.a * hyp.a * hyp.b * hyp.b / pi; count = 2; break;
        case DQGP_OUTER_RATQUAD: c0 = 2.0 * hyp.b / h0; c1 = 1.0; count = 2; break;
        case DQGP_OUTER_DOTPRODUCT: c0 = 2.0 * h0; break;
        default: break;
    }
    const int tiles = grad_tiles(n);
    cudaStream_t st = as_stream(stream);
    double* partial = static_cast<double*>(d_work);
    switch (outer) {
#define DQGP_GH(OUT) case OUT: grad_hyper_dmma_kernel<OUT><<<tiles, PW_THREADS, 0, st>>>(d_Ainv, ld, d_alpha, d_F, n, m, hyp, c0, c1, partial); break;
        DQGP_GH(DQGP_OUTER_GAUSSIAN) DQGP_GH(DQGP_OUTER_MATERN15) DQGP_GH(DQGP_OUTER_EXPSINE2) DQGP_GH(DQGP_OUTER_RATQUAD)
        DQGP_GH(DQGP_OUTER_DOTPRODUCT)
#undef DQGP_GH
    }
    DQGP_LAUNCH_CHECK("grad_hyper_dmma_kernel");
    grad_reduce_kernel<<<count, 256, 0, st>>>(partial, tiles, 2, 0.5, d_grad);
    DQGP_LAUNCH_CHECK("grad_reduce_kernel");
    return 0;
}

int dqgp_grad_noise_std(const double* d_Ainv, int ld, const double* d_alpha, int n, double noise_std, double* d_out, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Ainv && d_alpha && d_out, "dqgp_grad_noise_std: NULL argument");
    DQGP_REQUIRE(n >= 1 && ld >= n, "dqgp_grad_noise_std: bad shape (n %d, ld %d)", n, ld);
    grad_noise_kernel<<<1, 256, 0, as_stream(stream)>>>(d_Ainv, ld, d_alpha, n, noise_std, d_out);
    DQGP_LAUNCH_CHECK("grad_noise_kernel");
    return 0;
}

size_t dqgp_grad_analytic_workspace_bytes(int n, int m) {
    if (n <= 0 || m <= 0) return 0;
    return sizeof(double) * (size_t)(dqgp::GA_SEGMENTS + 1) * (size_t)n * (size_t)m;
}

int dqgp_grad_projected_analytic(int outer, const double* h_hyp, const double* d_Ainv, int ld, const double* d_alpha, const double* d_F,
                                 const double* d_J, int n, int m, int P, double* d_grad, void* d_work, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Ainv && d_alpha && d_F && d_J && d_grad && d_work && h_hyp, "dqgp_grad_projected_analytic: NULL argument");
    DQGP_REQUIRE(n >= 1 && ld >= n && P >= 1 && m >= 3 && m <= 36 && m % 3 == 0, "dqgp_grad_projected_analytic: bad shape (m = 3q, q <= 12)");
    OuterHyp hyp;
    if (make_outer_hyp(outer, h_hyp, &hyp)) return -1;
    cudaStream_t st = as_stream(stream);
    double* Gpart = static_cast<double*>(d_work);
    double* G = Gpart + (size_t)GA_SEGMENTS * n * m;
    const int seg_cols = ((n + GA_SEGMENTS - 1) / GA_SEGMENTS + GA_CHUNK - 1) / GA_CHUNK * GA_CHUNK;
    const int segments = (n + seg_cols - 1) / seg_cols;
    dim3 grid((n + GA_ROWS - 1) / GA_ROWS, segments);
    double scale = 2.0;                        // stationary: 2 sum_j <J_j, G_j>
    switch (outer) {
        case DQGP_OUTER_GAUSSIAN:
            launch_grad_analytic_rows<DQGP_OUTER_GAUSSIAN, false>(m, grid, st, d_Ainv, ld, d_alpha, d_F, n, hyp, seg_cols, Gpart);
            scale = -2.0 * hyp.a;              // the weight is e^{-gamma s}: kappa' = -gamma e^{-gamma s}
            break;
        case DQGP_OUTER_MATERN15: launch_grad_analytic_rows<DQGP_OUTER_MATERN15, false>(m, grid, st, d_Ainv, ld, d_alpha, d_F, n, hyp, seg_cols, Gpart); break;
        case DQGP_OUTER_EXPSINE2: launch_grad_analytic_rows<DQGP_OUTER_EXPSINE2, false>(m, grid, st, d_Ainv, ld, d_alpha, d_F, n, hyp, seg_cols, Gpart); break;
        case DQGP_OUTER_RATQUAD:
            if (hyp.b == 1.0) launch_grad_analytic_rows<DQGP_OUTER_RATQUAD, true>(m, grid, st, d_Ainv, ld, d_alpha, d_F, n, hyp, seg_cols, Gpart);
            else launch_grad_analytic_rows<DQGP_OUTER_RATQUAD, false>(m, grid, st, d_Ainv, ld, d_alpha, d_F, n, hyp, seg_cols, Gpart);
            break;
        default:                               // DQGP_OUTER_DOTPRODUCT: make_outer_hyp refused every other id
            launch_grad_analytic_rows<DQGP_OUTER_DOTPRODUCT, false>(m, grid, st, d_Ainv, ld, d_alpha, d_F, n, hyp, seg_cols, Gpart);
            scale = 1.0;                       // sum_j <J_j, (B F)_j>
            break;
    }
    DQGP_LAUNCH_CHECK("grad_analytic_rows_kernel");
    const size_t count = (size_t)n * m;
    grad_analytic_sum_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(Gpart, count, segments, G);
    grad_analytic_contract_kernel<<<P, 256, 0, st>>>(d_J, G, count, scale, d_grad);
    DQGP_LAUNCH_CHECK("grad_analytic kernels");
    return 0;
}

size_t dqgp_grad_fidelity_analytic_workspace_bytes(int n, int dim) {
    if (n <= 0 || dim <= 0) return 0;
    if (dim <= 64) return sizeof(double) * 2 * (size_t)(dqgp::GA_SEGMENTS + 1) * (size_t)n * (size_t)dim;
    const size_t npad = dqgp::gfd_npad(n);
    return sizeof(double) * (dqgp::GFD_TABLE + 2 * npad * npad + 6 * npad * (size_t)dim);
}

int dqgp_grad_fidelity_analytic(const double* d_Ainv, int ld, const double* d_alpha, const double* d_Psi, const double* d_D, int n, int dim,
                                int P, double* d_grad, void* d_work, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Ainv && d_alpha && d_Psi && d_D && d_grad && d_work, "dqgp_grad_fidelity_analytic: NULL argument");
    DQGP_REQUIRE(n >= 1 && ld >= n && P >= 1, "dqgp_grad_fidelity_analytic: bad shape");
    DQGP_REQUIRE(dim >= 2 && dim <= (1 << MAX_QUBITS) && (dim & (dim - 1)) == 0,
                 "dqgp_grad_fidelity_analytic: dim %d is not 2^q amplitudes with 1 <= q <= %d", dim, MAX_QUBITS);
    cudaStream_t st = as_stream(stream);
    if (dim > 64) {
        DQGP_REQUIRE((reinterpret_cast<uintptr_t>(d_Psi) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_work) & 15) == 0,
                     "dqgp_grad_fidelity_analytic: the state array and the workspace must be 16-byte aligned for 2^q >= 128");
        const int npad = (int)gfd_npad(n), d2 = 2 * dim;
        GemmTask* task = static_cast<GemmTask*>(d_work);
        double* W = static_cast<double*>(d_work) + GFD_TABLE;
        double* RR = W + (size_t)2 * npad * npad;
        double* G = RR + (size_t)2 * npad * d2;
        int rc = fidelity_weights_dmma(d_Ainv, ld, d_alpha, d_Psi, n, dim, W, npad, st);
        if (rc) return rc;
        const size_t pairs = (size_t)npad * dim;
        grad_fid_pack_kernel<<<(unsigned)((pairs + 255) / 256), 256, 0, st>>>(reinterpret_cast<const double2*>(d_Psi), n, dim, npad,
                                                                               reinterpret_cast<double2*>(RR));
        GemmTask t;
        memset(&t, 0, sizeof(t));
        t.A = W; t.B = RR; t.C = G;
        t.M = npad; t.N = d2; t.K = 2 * npad;
        t.lda = 2 * npad; t.ldb = d2; t.ldc = d2;
        t.a_k_contig = 1; t.b_k_contig = 0;
        t.lower_tiles = 0; t.krule = GM_KRULE_ALL;
        t.alpha = 1.0; t.beta = 0.0;
        t.tile_begin = 0; t.tiles = gemm_task_tiles(t);
        grad_fid_task_kernel<<<1, 1, 0, st>>>(t, task);
        DQGP_LAUNCH_CHECK("grad_fid_pack_kernel / grad_fid_task_kernel");
        rc = launch_gemm_group(task, 1, t.tiles, st);       // an unregistered table: the cp.async ring
        if (rc) return rc;
        const size_t count = (size_t)n * d2;
        const int slices = (int)std::max<size_t>(1, std::min<size_t>(GFD_SLICES, (size_t)2 * npad * npad / P));
        grad_fid_contract_kernel<<<dim3(slices, P), 256, 0, st>>>(d_D, G, count, P, W);
        grad_reduce_kernel<<<P, 256, 0, st>>>(W, slices, P, 2.0, d_grad);
        DQGP_LAUNCH_CHECK("grad_fid_contract_kernel");
        return 0;
    }
    double2* Gpart = static_cast<double2*>(d_work);
    double2* G = Gpart + (size_t)GA_SEGMENTS * n * dim;
    const int seg_cols = ((n + GA_SEGMENTS - 1) / GA_SEGMENTS + GF_CHUNK - 1) / GF_CHUNK * GF_CHUNK;
    const int segments = (n + seg_cols - 1) / seg_cols;
    dim3 grid((n + GF_ROWS - 1) / GF_ROWS, segments);
    const size_t smem = sizeof(double2) * ((size_t)2 * dim * GF_ROWS + (size_t)GF_CHUNK * dim);
    const double2* psi = reinterpret_cast<const double2*>(d_Psi);
    switch (dim) {
#define DQGP_GF(DD)                                                                                                            \
    case DD:                                                                                                                   \
        DQGP_CUDA(cudaFuncSetAttribute(grad_fid_analytic_rows_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        grad_fid_analytic_rows_kernel<DD><<<grid, GF_ROWS, smem, st>>>(d_Ainv, ld, d_alpha, psi, n, seg_cols, Gpart);          \
        break;
        DQGP_GF(2) DQGP_GF(4) DQGP_GF(8) DQGP_GF(16) DQGP_GF(32) DQGP_GF(64)
#undef DQGP_GF
    }
    DQGP_LAUNCH_CHECK("grad_fid_analytic_rows_kernel");
    const size_t count = (size_t)n * dim * 2;      // complex arrays as interleaved reals: Re<G|D> = sum of the real products
    grad_analytic_sum_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(reinterpret_cast<const double*>(Gpart), count, segments,
                                                                            reinterpret_cast<double*>(G));
    grad_analytic_contract_kernel<<<P, 256, 0, st>>>(d_D, reinterpret_cast<const double*>(G), count, 2.0, d_grad);
    DQGP_LAUNCH_CHECK("grad_fid_analytic kernels");
    return 0;
}

int dqgp_grad_fidelity(const double* d_Ainv, int ld, const double* d_alpha, const double* d_Psi, int n, int dim, int P, double h,
                       double* d_grad, void* d_work, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Ainv && d_alpha && d_Psi && d_grad && d_work, "dqgp_grad_fidelity: NULL argument");
    DQGP_REQUIRE(n >= 1 && ld >= n && P >= 1 && h != 0.0, "dqgp_grad_fidelity: bad shape / shift");
    DQGP_REQUIRE(dim >= 2 && dim <= (1 << MAX_QUBITS) && (dim & (dim - 1)) == 0,
                 "dqgp_grad_fidelity: dim %d is not 2^q amplitudes with 1 <= q <= %d", dim, MAX_QUBITS);
    DQGP_REQUIRE((reinterpret_cast<uintptr_t>(d_Psi) & 15) == 0, "dqgp_grad_fidelity: the state array must be 16-byte aligned");
    const int tiles = grad_tiles(n);
    cudaStream_t st = as_stream(stream);
    double* partial = static_cast<double*>(d_work);
    int rc = fidelity_grad_dmma(d_Ainv, ld, d_alpha, d_Psi, n, dim, P, partial, tiles, st);
    if (rc) return rc;
    grad_reduce_kernel<<<P, 256, 0, st>>>(partial, tiles, P, 0.5 / (2.0 * h), d_grad);
    DQGP_LAUNCH_CHECK("grad_reduce_kernel");
    return 0;
}
}
