// Blocked fp64 Cholesky + explicit SPD inverse + solve on one GPU (sm_100a).
// Replaces the LAPACK sequence of RiemannianAgent.train_and_update (reference agent_riemannian.py:410-418:
// cholesky, 4x general solve incl. an explicit inverse against eye(n); :442 slogdet) with
//   potrf   right-looking, nb = 128: [leaf: factor + invert the diagonal block] -> [panel = panel * inv(Lkk)^T]
//           -> [trailing -= panel panel^T]           (trailing update on DMMA, n^3/3 flops), scheduled as three
//           dependency classes on three streams (potrf_lookahead): the leaf chain runs at 68 us per 128 columns
//   trtri   W = L^-1 by recursive halving: W21 = -W22 (L21 W11), all products of one level in ONE grouped
//           launch (2 launches per level, log2(n/128) levels, n^3/3 flops on DMMA)
//   lauum   A^-1 = W^T W, lower tiles only, contraction range clipped to the triangular support (n^3/3)
//   solve   alpha = W^T (W y);  logdet = 2 sum log Lii (accumulated by the leaves)
// The matrix is padded to a multiple of 128 with an identity block, so no kernel has edge cases.
#include <cmath>
#include <cstdlib>
#include "gemm64.cuh"

namespace dqgp {
constexpr int NB = 128;
}  // namespace dqgp

struct dqgp_solver {
    int n, np, ld, nblk, device;
    // full mode: A factor (in place), W = L^-1, T scratch / A^-1 - three padded squares.
    // lean mode (prediction at sizes where three squares do not fit): A only; W holds just the nblk inverted diagonal
    // blocks (128 x 128 each, ldw = 128) and T two rotating outer-panel buffers (np x OB*128 each).
    int lean, ldw, ldt;
    double *A, *W, *T;
    double* w_block(int k) const { return lean ? W + (size_t)k * 128 * 128 : W + (size_t)k * 128 * ld + (size_t)k * 128; }
    // outer panels: panel p covers block columns [pan_lo[p], pan_hi[p]); widths may vary (wide while the trailing updates
    // bound the factorisation, narrow once the leaf chain does)
    std::vector<int> pan_of, pan_lo, pan_hi;
    double* t_block(int r, int k) const {   // block (r, k) of the panel storage
        return lean ? T + (size_t)(pan_of[k] & 1) * np * ldt + (size_t)r * 128 * ldt + (size_t)(k - pan_lo[pan_of[k]]) * 128
                    : T + (size_t)r * 128 * ld + (size_t)k * 128;
    }
    dqgp::GemmTask* d_dyn;        // per-call task table of the in-place substitution (dqgp_solver_quadform_rows_inplace)
    int dyn_capacity;
    double* tmp;                  // (rows x 128) product buffer of the substitution, grown on demand
    size_t tmp_rows;
    double *y_pad, *w, *partial;  // padded rhs, W y, column partial sums
    double *strip, *V;            // prediction: padded 128-row strip of K(test,train), V = W strip^T
    dqgp::GemmTask* d_tasks;
    // launch groups: [first task, task count, tiles]
    struct Group { int first, count, tiles; };
    int ob;                                           // outer panel width in 128-blocks (1 = single-level)
    cudaStream_t helper;                              // HIGH-priority stream carrying the critical path (leaf, panel solve, next column)
    cudaEvent_t ev_fork, ev_join;
    std::vector<cudaEvent_t> ev_rest;
    // potrf launch groups: three dependency classes, see potrf_lookahead
    std::vector<Group> trsmA, updA, trsmB, updB;      // per 128-column step: critical block row / everything else
    std::vector<Group> next1, next2, rest;            // per outer panel: rank-(OB*128) updates by distance from the panel
    cudaStream_t mid;                                 // second internal stream (panel work off the leaf chain)
    std::vector<cudaEvent_t> ev_leaf, ev_a, ev_b, ev_n1, ev_n2;
    cudaEvent_t ev_join2;
    int potrf_launches;
    std::vector<Group> tri_t, tri_w;       // per trtri level
    Group lauum, quad;
    size_t bytes;
};

namespace dqgp {

// ---- leaf: Cholesky of a 128x128 diagonal block and its triangular inverse, one CTA, 256 threads -----------
// One shared 128x130 array M holds both results: the strict upper triangle keeps L transposed
// (M[k][i] = L[i][k], k < i) and the strict lower triangle receives W = L^-1 (M[k][j] = W[k][j], j < k);
// the diagonals live in s_diag / s_rdiag.
// Phase 1 is a left-looking Cholesky in panels of 8 columns.  Row i is owned by the thread pair (i, i+128): both
// run the update loop over half of the k range each (per k: 1 conflict-free LDS + 4 broadcast LDS.128 for 8 DFMA),
// the helper hands its partial sums over through shared memory, and the primary thread factors the 8x8 diagonal
// block redundantly in registers (no cross-lane chain) and forward-substitutes its row.
// Phase 2 inverts L by recursive doubling (leaf_join): 8x8 diagonal blocks by substitution, then four levels of
// W21 = -W22 (L21 W11) as 8x8 DMMA tiles, 8 strips per level = 8 warps (round 1's column-substitution phase took 70K
// of the leaf's 155K cycles; measured with clock64: v3 spent 32K cycles in the phase-1 k-loops, 50K in the per-panel
// serial part).
constexpr int LEAF_THREADS = 256;
constexpr int LP = 132;     // pitch = 4 mod 16 doubles: the DMMA fragment patterns (t*LP + g and g*LP + t) are bank-conflict-free
constexpr size_t LEAF_SMEM_V2 = sizeof(double) * (NB * LP + 2 * NB + 8 * NB);

// Left-looking update of one 8-column panel for NT (1 or 2) 8-row tiles of one warp, on DMMA:
//   s_pan[c][row] = A[row][j0+c] - sum_{k<j0} L[row][k] L[j0+c][k],  with L[i][k] = M[k*LP + i].
// Four interleaved accumulators per tile keep the dependent DMMA chain j0/16 long; the B fragment is shared by the tiles.
template <int NT>
__device__ __forceinline__ void leaf_panel_update(const double* __restrict__ M, double* __restrict__ s_pan, int j0, int r0, int r1, int g,
                                                  int t, const double2 (&av)[2], long long* tq = nullptr) {
#ifdef DQGP_LEAF_TIMING
    long long q0 = clock64();
#define LEAF_Q(slot) do { const long long n__ = clock64(); tq[slot] += n__ - q0; q0 = n__; } while (0)
#else
#define LEAF_Q(slot) do { } while (0)
#endif
    double acc[NT][4][2];
#pragma unroll
    for (int x = 0; x < NT; ++x)
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[x][u][0] = acc[x][u][1] = 0.0;
    const double* mb = M + t * LP + j0 + g;
    const double* ma[2] = {M + t * LP + r0 + g, M + t * LP + r1 + g};
    const int full = j0 & ~15;                  // j0 is a multiple of 8: full rounds of 16 columns, then one half round
    for (int k0 = 0; k0 < full; k0 += 16) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double b = mb[(k0 + 4 * u) * LP];
#pragma unroll
            for (int x = 0; x < NT; ++x) dmma884(acc[x][u][0], acc[x][u][1], ma[x][(k0 + 4 * u) * LP], b);
        }
    }
    LEAF_Q(0);
    if (j0 & 8) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const double b = mb[(full + 4 * u) * LP];
#pragma unroll
            for (int x = 0; x < NT; ++x) dmma884(acc[x][u][0], acc[x][u][1], ma[x][(full + 4 * u) * LP], b);
        }
    }
#ifdef DQGP_LEAF_TIMING
    if (acc[0][0][0] + acc[0][1][0] + acc[0][2][0] + acc[0][3][0] == 1.2345e300) tq[3] += 1;      // wait for the DMMAs here
#endif
    LEAF_Q(1);
#ifdef DQGP_LEAF_TIMING
    if (av[0].x == 1.2345e300) tq[3] += 1;                                                       // wait for the prefetched A here
#endif
    LEAF_Q(2);
#pragma unroll
    for (int x = 0; x < NT; ++x) {
        const int r = (x == 0 ? r0 : r1) + g;
        s_pan[(2 * t) * NB + r] = av[x].x - ((acc[x][0][0] + acc[x][1][0]) + (acc[x][2][0] + acc[x][3][0]));
        s_pan[(2 * t + 1) * NB + r] = av[x].y - ((acc[x][0][1] + acc[x][1][1]) + (acc[x][2][1] + acc[x][3][1]));
    }
    LEAF_Q(4);
}

// One level of the triangular inverse inside the leaf: every pair of inverted BxB diagonal blocks (W11, W22) of the
// 128x128 factor is joined into a 2Bx2B inverse, W21 = -W22 (L21 W11), as 8x8 DMMA tiles.  M holds L transposed in its
// strict upper triangle and W in its strict lower triangle (diagonals in s_diag / rdiag), so operand fragments
// that straddle the diagonal are masked.  Each level has exactly 8 strips of tiles = 8 warps: product 1 (P = L21 W11,
// written where W21 will live) by row strips, product 2 by column strips - a warp only overwrites P tiles it alone reads.
template <int B>
__device__ __forceinline__ void leaf_join(double* __restrict__ M, const double* __restrict__ rdiag, int warp, int lane) {
    constexpr int NT = B / 8;
    const int pair = warp / NT, strip = warp % NT;
    const int r0 = pair * 2 * B;
    const int g = lane >> 2, t = lane & 3;
    {
        const int i0 = r0 + B + 8 * strip;
        double acc[NT][2];
#pragma unroll
        for (int x = 0; x < NT; ++x) acc[x][0] = acc[x][1] = 0.0;
#pragma unroll
        for (int ks = 0; ks < B / 4; ++ks) {
            const int kr = r0 + 4 * ks + t;
            const double a = M[kr * LP + i0 + g];                    // L[i0+g][kr]
#pragma unroll
            for (int tj = 0; tj < NT; ++tj) {
                if (4 * ks >= 8 * tj) {                              // W11 is lower-triangular: k >= j0
                    const int jc = r0 + 8 * tj + g;
                    double b = M[kr * LP + jc];                      // W[kr][jc]
                    if (4 * ks < 8 * tj + 8) b = (jc < kr) ? b : (jc == kr ? rdiag[kr] : 0.0);
                    dmma884(acc[tj][0], acc[tj][1], a, b);
                }
            }
        }
#pragma unroll
        for (int tj = 0; tj < NT; ++tj)
            *reinterpret_cast<double2*>(&M[(i0 + g) * LP + r0 + 8 * tj + 2 * t]) = make_double2(acc[tj][0], acc[tj][1]);
    }
    __syncthreads();
    {
        const int j0 = r0 + 8 * strip;
        double acc[NT][2];
#pragma unroll
        for (int x = 0; x < NT; ++x) acc[x][0] = acc[x][1] = 0.0;
#pragma unroll
        for (int ks = 0; ks < B / 4; ++ks) {
            const int kc = r0 + B + 4 * ks + t;
            const double b = M[kc * LP + j0 + g];                    // P[kc][j0+g]
#pragma unroll
            for (int ti = 0; ti < NT; ++ti) {
                if (4 * ks < 8 * ti + 8) {                           // W22 is lower-triangular: k <= i
                    const int ir = r0 + B + 8 * ti + g;
                    double a = M[ir * LP + kc];                      // W[ir][kc]
                    if (4 * ks >= 8 * ti) a = (kc < ir) ? a : (kc == ir ? rdiag[ir] : 0.0);
                    dmma884(acc[ti][0], acc[ti][1], a, b);
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int ti = 0; ti < NT; ++ti)
            *reinterpret_cast<double2*>(&M[(r0 + B + 8 * ti + g) * LP + j0 + 2 * t]) = make_double2(-acc[ti][0], -acc[ti][1]);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(LEAF_THREADS, 1) potrf_leaf_kernel(double* __restrict__ A, int ld, double* __restrict__ Wblk,
                                                                      int ldw, int blk, double* logdet, int* info, int n_real) {
    extern __shared__ __align__(16) double leaf_smem[];
    double* M = leaf_smem;
    double* s_diag = M + NB * LP;
    double* s_rdiag = s_diag + NB;
    double* s_part = s_rdiag + NB;            // [8][128] the current panel after its left-looking update
    __shared__ double s_red[LEAF_THREADS / 32];
    __shared__ int s_bad;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int i = tid & (NB - 1);             // row owned in phase 1
    const bool helper = tid >= NB;
    double* Ablk = A + (size_t)blk * NB * ld + (size_t)blk * NB;
    if (tid == 0) s_bad = 0;
    __syncthreads();

    // ---------------- phase 1: Cholesky, left-looking in panels of 8 columns ----------------
    // (a) all 8 warps: the panel's rows >= j0 minus the contribution of every earlier column, on DMMA: 8x8 tiles
    //     P = A[rows, j0..j0+8) - L[rows, 0..j0) L[j0..j0+8, 0..j0)^T, four interleaved accumulators per tile so the
    //     dependent DMMA chain is j0/16 long; the A entries are prefetched one panel ahead.  Result -> s_pan[c][row].
    // (b) the 128 row threads: every thread factors the 8x8 diagonal block redundantly in registers (no cross-lane
    //     chain), substitutes its own row, and stores L to M (transposed) and to HBM.
    const int g = lane >> 2, t = lane & 3;
    double* s_pan = s_part;                    // [8][128]
    double2 av[2];
#pragma unroll
    for (int x = 0; x < 2; ++x) {
        const int ti = warp + 8 * x;
        av[x] = *reinterpret_cast<const double2*>(Ablk + (size_t)(8 * ti + g) * ld + 2 * t);
    }
#ifdef DQGP_LEAF_TIMING
    long long tk[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ta[16], tw = 0, t_prev = clock64(), t_begin = t_prev, tq[5] = {0, 0, 0, 0, 0}, tr[2] = {0, 0};
#define LEAF_TICK(slot) do { const long long now__ = clock64(); tk[slot] += now__ - t_prev; t_prev = now__; } while (0)
#else
#define LEAF_TICK(slot) do { } while (0)
#endif
    for (int j0 = 0; j0 < NB; j0 += 8) {
        const int tb = j0 >> 3;
        {
            // this warp's row tiles: tb + warp and tb + warp + 8; the B fragment (rows j0..j0+7 of L) is shared by both
            const int ti0 = tb + warp, ti1 = ti0 + 8;
            const bool has0 = ti0 < NB / 8, has1 = ti1 < NB / 8;     // warp-uniform
            // no predicated mma.sync inside the loops: a predicate makes the compiler fence every DMMA with WARPSYNC
            // (measured: 180 cycles per DMMA instead of 16), so the one- and two-tile cases are separate instantiations
#ifdef DQGP_LEAF_TIMING
            const long long c_pre = clock64();
            if (has1) leaf_panel_update<2>(M, s_pan, j0, 8 * ti0, 8 * ti1, g, t, av, tq);
            else if (has0) leaf_panel_update<1>(M, s_pan, j0, 8 * ti0, 8 * ti0, g, t, av, tq);
            const long long c_post = clock64();
            tr[0] += c_pre - t_prev; tr[1] += c_post - c_pre;
#else
            if (has1) leaf_panel_update<2>(M, s_pan, j0, 8 * ti0, 8 * ti1, g, t, av);
            else if (has0) leaf_panel_update<1>(M, s_pan, j0, 8 * ti0, 8 * ti0, g, t, av);
#endif
            if (j0 + 8 < NB) {                                      // prefetch this warp's tiles of the next panel
                if (ti0 + 1 < NB / 8) av[0] = *reinterpret_cast<const double2*>(Ablk + (size_t)(8 * (ti0 + 1) + g) * ld + j0 + 8 + 2 * t);
                if (ti1 + 1 < NB / 8) av[1] = *reinterpret_cast<const double2*>(Ablk + (size_t)(8 * (ti1 + 1) + g) * ld + j0 + 8 + 2 * t);
            }
        }
#ifdef DQGP_LEAF_TIMING
        { const long long now__ = clock64(); ta[tb] = now__ - t_prev; }
#endif
        LEAF_TICK(0);
        __syncthreads();
        LEAF_TICK(1);
        if (!helper && i >= j0) {
            double a[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) a[c] = s_pan[c * NB + i];
            double l[8][8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c <= r; ++c) l[r][c] = s_pan[c * NB + j0 + r];
            double rd[8];
#ifdef DQGP_LEAF_TIMING
            if (l[7][7] == 1.2345e300) tk[7] += 1;     // force the loads to complete here
            LEAF_TICK(2);
#endif
            // The thread's own row rides along as a ninth row of the block (column-oriented substitution: as soon as x_c is known it
            // is removed from all later columns): its independent instructions fill the latency of the rsqrt chain.  The rows of
            // the diagonal block take the same path (no divergence in their warp): the recurrence reproduces their row of L
            // operation by operation, and what it leaves right of the diagonal is never stored.
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const double piv = l[c][c];
                if (!(piv > 0.0) && i == j0 && s_bad == 0) s_bad = j0 + c + 1;
                rd[c] = rsqrt(piv);
                l[c][c] = piv * rd[c];
                const double x = a[c] * rd[c];
                a[c] = x;
#pragma unroll
                for (int r = c + 1; r < 8; ++r) l[r][c] *= rd[c];
#pragma unroll
                for (int c2 = c + 1; c2 < 8; ++c2) {
#pragma unroll
                    for (int r = c2; r < 8; ++r) l[r][c2] = fma(-l[r][c], l[c2][c], l[r][c2]);
                    a[c2] = fma(-x, l[c2][c], a[c2]);
                }
            }
#ifdef DQGP_LEAF_TIMING
            if (l[7][7] == 1.2345e300) tk[7] += 1;
            LEAF_TICK(3);
#endif
            if (i < j0 + 8) {
                const int r0 = i - j0;
                double dv = a[0], rv = rd[0];
#pragma unroll
                for (int r = 1; r < 8; ++r)
                    if (r == r0) { dv = a[r]; rv = rd[r]; }
                s_diag[i] = dv;
                s_rdiag[i] = rv;
            }
#ifdef DQGP_LEAF_TIMING
            if (a[7] == 1.2345e300) tk[7] += 1;
            LEAF_TICK(4);
#endif
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (i > j0 + c) M[(j0 + c) * LP + i] = a[c];
            double2* dst = reinterpret_cast<double2*>(Ablk + (size_t)i * ld + j0);
#pragma unroll
            for (int c = 0; c < 4; ++c)
                dst[c] = make_double2((i >= j0 + 2 * c) ? a[2 * c] : 0.0, (i >= j0 + 2 * c + 1) ? a[2 * c + 1] : 0.0);
        }
        LEAF_TICK(5);
        __syncthreads();
        LEAF_TICK(6);
    }
#ifdef DQGP_LEAF_TIMING
    const long long t_phase1 = clock64();
#endif
    // logdet: the helper warps (idle in level 0 of phase 2) take the logarithms; the read-modify-write of the global accumulator
    // (a round trip to L2) waits until the end of the kernel, off the path of the barriers below
    if (helper) {
        double v = warp_sum(log(s_diag[tid - NB]));
        if (lane == 0) s_red[warp] = v;
    }

    // ---------------- phase 2: W = L^-1 by recursive doubling on the DMMA pipe ----------------
    // level 0: the 16 diagonal 8x8 blocks by substitution, one thread per column
    if (tid < NB) {
        const int j = tid, b0 = j & ~7;
        double w[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int row = b0 + r;
            double v = 0.0;
            if (row == j) v = s_rdiag[j];
            else if (row > j) {
                double sres = 0.0;
#pragma unroll
                for (int r2 = 0; r2 < r; ++r2)
                    if (b0 + r2 >= j) sres = fma(M[(b0 + r2) * LP + row], w[r2], sres);
                v = -sres * s_rdiag[row];
            }
            w[r] = v;
        }
#pragma unroll
        for (int r = 0; r < 8; ++r)
            if (b0 + r > j) M[(b0 + r) * LP + j] = w[r];
    }
    __syncthreads();
    leaf_join<8>(M, s_rdiag, warp, lane);
    leaf_join<16>(M, s_rdiag, warp, lane);
    leaf_join<32>(M, s_rdiag, warp, lane);
    leaf_join<64>(M, s_rdiag, warp, lane);
#ifdef DQGP_LEAF_TIMING
    const long long t_phase2 = clock64();
#endif
    // lower triangle only: the strict upper triangle of W's diagonal blocks is zeroed once, at solver creation
#pragma unroll 4
    for (int e = tid; e < NB * NB / 2; e += LEAF_THREADS) {
        const int r = e >> 6, c = (e & 63) * 2;
        if (c > r) continue;
        double2 v;
        v.x = (c < r) ? M[r * LP + c] : s_rdiag[r];
        v.y = (c + 1 < r) ? M[r * LP + c + 1] : (c + 1 == r ? s_rdiag[r] : 0.0);
        *reinterpret_cast<double2*>(Wblk + (size_t)r * ldw + c) = v;
    }
    if (tid == LEAF_THREADS - 1) {      // s_red[4..7] were written before the barriers of phase 2
        double tot = 0.0;
#pragma unroll
        for (int w = NB / 32; w < LEAF_THREADS / 32; ++w) tot += s_red[w];
        *logdet += 2.0 * tot;
        if (s_bad && *info == 0 && blk * NB + s_bad <= n_real) *info = blk * NB + s_bad;
    }
#ifdef DQGP_LEAF_TIMING
    if (tid == NB - 1 && blk == 1)
        printf("panel update cycles per panel: %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld\n", ta[0], ta[1], ta[2],
               ta[3], ta[4], ta[5], ta[6], ta[7], ta[8], ta[9], ta[10], ta[11], ta[12], ta[13], ta[14], ta[15]);
    if (tid == NB - 1 && blk == 1)
        printf("panel update split (thread 127, all panels): zero + full rounds %lld | half round + DMMA drain %lld | wait for prefetched A %lld | s_pan stores %lld\n",
               tq[0], tq[1], tq[2], tq[4]);
    if (tid == NB - 1 && blk == 1) printf("   before the call %lld | inside the call %lld | (rest of 'dmma update': the prefetch loads of the next panel)\n", tr[0], tr[1]);
    if (tid == NB - 1 && blk == 1)
        printf("leaf cycles (thread 127): dmma update %lld | sync wait %lld | loads %lld | 8x8 factor %lld | substitution %lld | stores %lld | "
               "end sync %lld | (a: dmma loops %lld, wait for prefetched A %lld) || phase1 %lld  logdet+phase2 %lld  W store %lld\n", tk[0], tk[1], tk[2], tk[3], tk[4], tk[5], tk[6], tk[7], tw,
               t_phase1 - t_begin, t_phase2 - t_phase1, clock64() - t_phase2);
#endif
}

// ---- padding: rows/cols >= n become the identity ---------------------------------------------------------
__global__ void pad_identity_kernel(double* A, int n, int np, int ld) {
    const int r = blockIdx.x;   // np rows
    for (int c = threadIdx.x; c < np; c += blockDim.x) {
        if (r >= n || c >= n) A[(size_t)r * ld + c] = (r == c) ? 1.0 : 0.0;
    }
}
__global__ void pad_vector_kernel(const double* y, int n, int np, double* out, double* logdet, int* info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < np) out[i] = (y != nullptr && i < n) ? y[i] : 0.0;
    if (i == 0) { *logdet = 0.0; *info = 0; }
}

// ---- copy the strictly-lower 128x128 blocks of src into dst (panels of L: T -> A) ---------------------------
__global__ void copy_lower_blocks_kernel(const double* __restrict__ src, double* __restrict__ dst, int ld) {
    const int rb = blockIdx.y + 1, cb = blockIdx.x;
    if (cb >= rb) return;
    const double2* s2 = reinterpret_cast<const double2*>(src + (size_t)rb * NB * ld + (size_t)cb * NB);
    double2* d2 = reinterpret_cast<double2*>(dst + (size_t)rb * NB * ld + (size_t)cb * NB);
    for (int e = threadIdx.x; e < NB * NB / 2; e += blockDim.x) {
        const int r = e >> 6, c = e & 63;
        d2[(size_t)r * (ld / 2) + c] = s2[(size_t)r * (ld / 2) + c];
    }
}

// ---- w = W y (lower-triangular, one warp per row) --------------------------------------------------------
__global__ void trmv_lower_kernel(const double* __restrict__ W, int np, int ld, const double* __restrict__ y, double* __restrict__ w) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= np) return;
    double acc = 0.0;
    for (int k = lane; k <= row; k += 32) acc = fma(W[(size_t)row * ld + k], y[k], acc);
    acc = warp_sum(acc);
    if (lane == 0) w[row] = acc;
}
// ---- alpha = W^T w: per (row block, column block) partial sums, then a fixed-order reduction --------------
__global__ void trmv_lower_T_partial_kernel(const double* __restrict__ W, int ld, const double* __restrict__ w, double* __restrict__ partial, int np) {
    const int rb = blockIdx.y, cb = blockIdx.x;
    const int col = cb * NB + threadIdx.x;
    double acc = 0.0;
    if (rb >= cb) {
        const int r0 = rb * NB;
        for (int r = 0; r < NB; ++r) acc = fma(W[(size_t)(r0 + r) * ld + col], w[r0 + r], acc);   // zero above the diagonal
    }
    partial[(size_t)rb * np + col] = acc;
}
__global__ void reduce_partial_kernel(const double* __restrict__ partial, int nblk, int np, int n, double* __restrict__ out) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= n) return;
    double acc = 0.0;
    for (int rb = 0; rb < nblk; ++rb) acc += partial[(size_t)rb * np + col];
    out[col] = acc;
}
// ---- mirror the lower triangle of a padded square into the upper one (tiled transpose through smem) --------
__global__ void symmetrize_lower_kernel(double* A, int ld) {
    __shared__ double tile[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    for (int r = ty; r < 32; r += 8) tile[r][tx] = A[(size_t)(bi * 32 + r) * ld + bj * 32 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int gr = bj * 32 + r, gc = bi * 32 + tx;
        if (bi != bj || gc > gr) A[(size_t)gr * ld + gc] = tile[tx][r];
    }
}
__global__ void colsumsq_kernel(const double* __restrict__ V, int rows, int ld, int ncols, double* __restrict__ out) {
    // out[c] = sum_r V[r][c]^2, fixed order; one thread per column, coalesced across threads
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncols) return;
    double acc = 0.0;
    for (int r = 0; r < rows; ++r) { const double v = V[(size_t)r * ld + c]; acc = fma(v, v, acc); }
    out[c] = acc;
}
__global__ void copy_pad_rows_kernel(const double* __restrict__ B, int nb, int n, int ldb, double* __restrict__ out, int nbp, int np, int ldo) {
    const int r = blockIdx.x;
    for (int c = threadIdx.x; c < np; c += blockDim.x) out[(size_t)r * ldo + c] = (r < nb && c < n) ? B[(size_t)r * ldb + c] : 0.0;
}


// ---- lean mode: copy one solved block column of the panel storage back over its (dead) input, A(k+1.., k) <- T(k+1.., k)
__global__ void copy_panel_column_kernel(const double* __restrict__ src, int lds, double* __restrict__ dst, int ldd, int rows) {
    const double2* s2 = reinterpret_cast<const double2*>(src);
    double2* d2 = reinterpret_cast<double2*>(dst);
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < (size_t)rows * (NB / 2); e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / (NB / 2), c = e % (NB / 2);
        d2[r * (ldd / 2) + c] = s2[r * (lds / 2) + c];
    }
}
// ---- lean mode, vector solves with L (blocked substitution; the diagonal blocks are applied through their inverses)
// out[0..127] = Wkk in  (trans = 0)  or  Wkk^T in  (trans = 1); in == out allowed
__global__ void diag_block_mv_kernel(const double* __restrict__ Wk, int ldw, const double* in, double* out, int trans) {
    __shared__ double x[NB];
    const int i = threadIdx.x;
    x[i] = in[i];
    __syncthreads();
    double acc = 0.0;
    if (!trans) { for (int j = 0; j <= i; ++j) acc = fma(Wk[(size_t)i * ldw + j], x[j], acc); }
    else        { for (int j = i; j < NB; ++j) acc = fma(Wk[(size_t)j * ldw + i], x[j], acc); }
    out[i] = acc;
}
// y[r] -= sum_c L[r][k*128 + c] * wk[c]  for the rows below block k (one warp per row)
__global__ void subst_forward_update_kernel(const double* __restrict__ L, int ld, int k, int np, const double* __restrict__ wk,
                                            double* __restrict__ y) {
    const int row = (k + 1) * NB + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= np) return;
    const double* lr = L + (size_t)row * ld + (size_t)k * NB;
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < NB / 32; ++c) acc = fma(lr[lane + 32 * c], wk[lane + 32 * c], acc);
    acc = warp_sum(acc);
    if (lane == 0) y[row] -= acc;
}
// w[j] -= sum_r L[k*128 + r][j] * xk[r]  for the columns left of block k (one thread per column)
__global__ void subst_backward_update_kernel(const double* __restrict__ L, int ld, int k, const double* __restrict__ xk, double* __restrict__ w) {
    __shared__ double x[NB];
    if (threadIdx.x < NB) x[threadIdx.x] = xk[threadIdx.x];
    __syncthreads();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k * NB) return;
    const double* lc = L + (size_t)k * NB * ld + j;
    double acc = 0.0;
    for (int r = 0; r < NB; ++r) acc = fma(lc[(size_t)r * ld], x[r], acc);
    w[j] -= acc;
}
// in-place substitution on row-major right-hand sides: B[:, k-block] <- tmp, out[i] += sum_c tmp[i][c]^2 (fixed order)
__global__ void subst_store_sumsq_kernel(const double* __restrict__ tmp, double* __restrict__ B, int ldb, int k, int rows,
                                         double* __restrict__ out, int first) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const double2* t2 = reinterpret_cast<const double2*>(tmp + (size_t)row * NB);
    double2* b2 = reinterpret_cast<double2*>(B + (size_t)row * ldb + (size_t)k * NB);
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < NB / 64; ++c) {
        const double2 v = t2[lane + 32 * c];
        b2[lane + 32 * c] = v;
        acc = fma(v.x, v.x, acc); acc = fma(v.y, v.y, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) out[row] = first ? acc : out[row] + acc;
}

static GemmTask make_task3(const double* A, int lda, const double* B, int ldb, double* C, int ldc, int M, int N, int K, int a_k, int b_k,
                           int lower, int krule, double alpha, double beta) {
    GemmTask t;
    t.A = A; t.B = B; t.C = C; t.M = M; t.N = N; t.K = K; t.lda = lda; t.ldb = ldb; t.ldc = ldc;
    t.a_k_contig = a_k; t.b_k_contig = b_k; t.lower_tiles = lower; t.krule = krule; t.alpha = alpha; t.beta = beta;
    t.tile_begin = 0; t.tiles = gemm_task_tiles(t);
    return t;
}
static GemmTask make_task(const double* A, const double* B, double* C, int M, int N, int K, int ld, int a_k, int b_k, int lower,
                          int krule, double alpha, double beta) {
    GemmTask t;
    t.A = A; t.B = B; t.C = C; t.M = M; t.N = N; t.K = K; t.lda = t.ldb = t.ldc = ld;
    t.a_k_contig = a_k; t.b_k_contig = b_k; t.lower_tiles = lower; t.krule = krule; t.alpha = alpha; t.beta = beta;
    t.tile_begin = 0; t.tiles = gemm_task_tiles(t);
    return t;
}

}  // namespace dqgp

// Right-looking blocked Cholesky as three dependency classes on three streams.
//   crit (highest priority): leaf_k -> trsmA_k -> updA_k -> leaf_{k+1}: the chain that bounds a lone factorisation.
//        A leaf needs 133 KB of shared memory and only fits beside ONE resident GEMM CTA, so it must win the slot a
//        retiring GEMM CTA frees.
//   mid: the rest of step k (solve of the rows below, rank-128 updates of the panel's own columns and of the FIRST
//        column of the next panel), then, at a panel end, the rank-(OB*128) update of the next OB columns.
//   st (caller): the bulk rank-(OB*128) update of everything further right, one panel behind.
// Every block receives its updates in the same order as in the sequential algorithm (events order all writers of a
// block), so the factor does not depend on timing.
static int potrf_lookahead(dqgp_solver* s, double* d_logdet, int* d_info, cudaStream_t st) {
    using namespace dqgp;
    const int ld = s->ld, nblk = s->nblk, OB = s->ob;
    cudaStream_t crit = s->helper, mid = s->mid;
    auto run = [&](const dqgp_solver::Group& g, cudaStream_t on) { return launch_gemm_group(s->d_tasks + g.first, g.count, g.tiles, on); };
    auto run_small = [&](const dqgp_solver::Group& g, cudaStream_t on) { return launch_gemm_group_small(s->d_tasks + g.first, g.count, g.tiles, on); };
    DQGP_CUDA(cudaEventRecord(s->ev_fork, st));
    DQGP_CUDA(cudaStreamWaitEvent(crit, s->ev_fork, 0));
    DQGP_CUDA(cudaStreamWaitEvent(mid, s->ev_fork, 0));
    // DQGP_POTRF_TRACE=1: time stamps on the critical stream (diagnostics; synchronises and prints to stderr)
    static const bool trace = getenv("DQGP_POTRF_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    auto stamp = [&]() { if (trace) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, crit); tev.push_back(e); } };
    int last_rest = -1;
    for (int k = 0; k < nblk; ++k) {
        const int p = s->pan_of[k], p0 = s->pan_lo[p], pend = s->pan_hi[p];
        stamp();
        potrf_leaf_kernel<<<1, LEAF_THREADS, LEAF_SMEM_V2, crit>>>(s->A, ld, s->w_block(k), s->ldw, k, d_logdet, d_info, s->n);
        DQGP_LAUNCH_CHECK("potrf_leaf_kernel");
        stamp();
        if (k + 1 >= nblk) break;
        DQGP_CUDA(cudaEventRecord(s->ev_leaf[k], crit));
        // critical block row
        if (k > 0) DQGP_CUDA(cudaStreamWaitEvent(crit, s->ev_b[k - 1], 0));            // A(k+1,k) has all its updates
        if (s->lean && p >= 2 && k == p0 && s->rest[p - 2].tiles > 0)                  // this panel's buffer was panel p-2's:
            DQGP_CUDA(cudaStreamWaitEvent(crit, s->ev_rest[p - 2], 0));                // its bulk update must have read it
        int rc = run_small(s->trsmA[k], crit);
        if (rc) return rc;
        DQGP_CUDA(cudaEventRecord(s->ev_a[k], crit));
        stamp();
        if (p > 0 && k == p0) DQGP_CUDA(cudaStreamWaitEvent(crit, s->ev_n1[p - 1], 0));     // column p0+1 got the previous panel
        if (p > 0 && k == p0 + 1) DQGP_CUDA(cudaStreamWaitEvent(crit, s->ev_n2[p - 1], 0)); // columns p0+2.. likewise
        rc = run_small(s->updA[k], crit);
        if (rc) return rc;
        stamp();
        // the rest of the step
        DQGP_CUDA(cudaStreamWaitEvent(mid, s->ev_leaf[k], 0));
        rc = run(s->trsmB[k], mid);
        if (rc) return rc;
        DQGP_CUDA(cudaStreamWaitEvent(mid, s->ev_a[k], 0));
        rc = run(s->updB[k], mid);
        if (rc) return rc;
        DQGP_CUDA(cudaEventRecord(s->ev_b[k], mid));
        if (s->lean) {    // the panel buffers rotate: L's block column goes back over its own input now
            const int rows = s->np - (k + 1) * NB;
            copy_panel_column_kernel<<<std::min(rows, 2048), 256, 0, mid>>>(s->t_block(k + 1, k), s->ldt, s->A + (size_t)(k + 1) * NB * ld + (size_t)k * NB, ld, rows);
            DQGP_LAUNCH_CHECK("copy_panel_column_kernel");
        }
        if (k + 1 == pend && pend < nblk) {            // the panel's columns of L are complete
            if (last_rest >= 0) DQGP_CUDA(cudaStreamWaitEvent(mid, s->ev_rest[last_rest], 0));   // bulk updates hit these columns
            rc = run(s->next1[p], mid);
            if (rc) return rc;
            DQGP_CUDA(cudaEventRecord(s->ev_n1[p], mid));
            rc = run(s->next2[p], mid);
            if (rc) return rc;
            DQGP_CUDA(cudaEventRecord(s->ev_n2[p], mid));
            if (s->rest[p].tiles > 0) {
                DQGP_CUDA(cudaStreamWaitEvent(st, s->ev_b[k], 0));
                rc = run(s->rest[p], st);
                if (rc) return rc;
                DQGP_CUDA(cudaEventRecord(s->ev_rest[p], st));
                last_rest = p;
            }
        }
    }
    DQGP_CUDA(cudaEventRecord(s->ev_join, crit));
    DQGP_CUDA(cudaStreamWaitEvent(st, s->ev_join, 0));
    DQGP_CUDA(cudaEventRecord(s->ev_join2, mid));
    DQGP_CUDA(cudaStreamWaitEvent(st, s->ev_join2, 0));
    if (trace) {
        cudaStreamSynchronize(st);
        // per step: [start, leaf end, trsmA end, updA end]
        double t_leaf = 0, t_trsm = 0, t_upd = 0, t_gap = 0;
        for (int k = 0; k + 1 < nblk; ++k) {
            float a = 0, b = 0, c = 0, d = 0;
            cudaEventElapsedTime(&a, tev[4 * k], tev[4 * k + 1]);
            cudaEventElapsedTime(&b, tev[4 * k + 1], tev[4 * k + 2]);
            cudaEventElapsedTime(&c, tev[4 * k + 2], tev[4 * k + 3]);
            cudaEventElapsedTime(&d, tev[4 * k + 3], tev[4 * k + 4]);
            t_leaf += a; t_trsm += b; t_upd += c; t_gap += d;
            if (k % 2 == 0 || k + 2 >= nblk) fprintf(stderr, "  step %3d: leaf %.1f us  (wait evB +) trsmA %.1f  (wait next +) updA %.1f  gap %.1f\n", k, a * 1e3, b * 1e3, c * 1e3, d * 1e3);
        }
        fprintf(stderr, "potrf trace n=%d OB=%d: leaf %.2f ms  trsmA %.2f  updA %.2f  gaps %.2f\n", s->n, OB, t_leaf, t_trsm, t_upd, t_gap);
        for (auto e : tev) cudaEventDestroy(e);
    }
    return 0;
}

static int solver_create_impl(int n, int outer_blocks, int lean, dqgp_solver** out);

extern "C" {

int dqgp_solver_create(int n, dqgp_solver** out) { return dqgp_solver_create_ex(n, 0, out); }
int dqgp_solver_create_ex(int n, int outer_blocks, dqgp_solver** out) { return solver_create_impl(n, outer_blocks, 0, out); }
int dqgp_solver_create_lean(int n, int outer_blocks, dqgp_solver** out) { return solver_create_impl(n, outer_blocks, 1, out); }
int dqgp_solver_is_lean(const dqgp_solver* s) { return s ? s->lean : -1; }

}  // extern "C"

static int solver_create_impl(int n, int outer_blocks, int lean, dqgp_solver** out) {
    using namespace dqgp;
    DQGP_REQUIRE(out != nullptr, "dqgp_solver_create: out is NULL");
    *out = nullptr;
    DQGP_REQUIRE(n >= 1 && n <= (1 << 17), "dqgp_solver_create: n = %d outside [1, 131072]", n);
    dqgp_solver* s = new dqgp_solver();
    s->n = n;
    // widest panel.  Default (0): rank-128 panels up to n = 6144, where a factorisation is bound by its leaf chain and every extra
    // panel-boundary dependency costs (potrf at n = 2048: 0.88 / 0.94 / 1.02 ms with 1 / 2 / 4 blocks; 4096: 2.1 / 2.3 / 2.5;
    // 6144: 4.28 / 4.33 / 4.69), rank-512 above (throughput of several concurrent factorisations; 8192: 8.4 / 8.1 / 8.3 alone)
    s->ob = outer_blocks > 0 ? (outer_blocks > 16 ? 16 : outer_blocks) : (outer_blocks == 0 && !lean && n <= 6144 ? 1 : 4);
    s->nblk = (n + NB - 1) / NB;
    {
        // outer_blocks < 0: rank-512 panels while more than 28 block columns remain (there the rank-k trailing updates bound
        // the factorisation and want the long contraction), rank-256 panels afterwards (the leaf chain bounds it)
        s->pan_of.assign(s->nblk, 0);
        for (int k0 = 0, p = 0; k0 < s->nblk; ++p) {
            const int w = std::min(outer_blocks < 0 ? (s->nblk - k0 > 28 ? 4 : 2) : s->ob, s->nblk - k0);
            s->pan_lo.push_back(k0); s->pan_hi.push_back(k0 + w);
            for (int k = k0; k < k0 + w; ++k) s->pan_of[k] = p;
            k0 += w;
        }
    }
    s->np = s->nblk * NB;
    s->ld = s->np;
    s->A = s->W = s->T = s->y_pad = s->w = s->partial = s->strip = s->V = nullptr;
    s->d_tasks = nullptr; s->d_dyn = nullptr; s->dyn_capacity = 0; s->tmp = nullptr; s->tmp_rows = 0;
    s->lean = lean ? 1 : 0;
    s->ldw = lean ? NB : s->ld;
    s->ldt = lean ? s->ob * NB : s->ld;
    s->helper = nullptr; s->mid = nullptr; s->ev_fork = nullptr; s->ev_join = nullptr; s->ev_join2 = nullptr;
    cudaError_t e = cudaGetDevice(&s->device);
    const size_t mat = sizeof(double) * (size_t)s->np * s->ld;
    const size_t wbytes = lean ? sizeof(double) * (size_t)s->nblk * NB * NB : mat;
    const size_t tbytes = lean ? sizeof(double) * 2 * (size_t)s->np * s->ldt : mat;
    s->bytes = mat + wbytes + tbytes;
    if (e == cudaSuccess) e = cudaMalloc(&s->A, mat);
    if (e == cudaSuccess) e = cudaMalloc(&s->W, wbytes);
    if (e == cudaSuccess) e = cudaMemset(s->W, 0, wbytes);   // the leaves write only the lower triangle of W's diagonal blocks
    if (e == cudaSuccess) e = cudaMalloc(&s->T, tbytes);
    if (e == cudaSuccess) e = cudaMalloc(&s->y_pad, sizeof(double) * s->np);
    if (e == cudaSuccess) e = cudaMalloc(&s->w, sizeof(double) * s->np);
    if (!lean) {
        if (e == cudaSuccess) e = cudaMalloc(&s->partial, sizeof(double) * (size_t)s->nblk * s->np);
        if (e == cudaSuccess) e = cudaMalloc(&s->strip, sizeof(double) * (size_t)NB * s->ld);
        if (e == cudaSuccess) e = cudaMalloc(&s->V, sizeof(double) * (size_t)s->np * NB);
    } else if (e == cudaSuccess) {
        e = cudaMalloc(&s->partial, sizeof(double) * s->np);     // apply_factor's output staging
    }
    if (e != cudaSuccess) { dqgp_solver_destroy(s); return cuda_fail(e, "dqgp_solver_create (allocation; this library has no CPU fallback)"); }

    std::vector<GemmTask> tasks;
    auto push_group = [&](std::vector<GemmTask>& grp) {
        dqgp_solver::Group g;
        g.first = (int)tasks.size(); g.count = (int)grp.size(); g.tiles = 0;
        for (auto& t : grp) { t.tile_begin = g.tiles; g.tiles += t.tiles; tasks.push_back(t); }
        grp.clear();
        return g;
    };
    const int ld = s->ld, np = s->np, nblk = s->nblk;
    auto at = [&](double* base, int rb, int cb) { return base + (size_t)rb * NB * ld + (size_t)cb * NB; };
    std::vector<GemmTask> grp;
    auto small = [](GemmTask t) { t.tiles = gemm_task_tiles_small(t); return t; };
    // ---- look-ahead schedule.  Step k (panel p = k / OB, columns [p0, pend)):
    //   trsmA[k]  T(k+1,k)   = A(k+1,k) Wkk^T                       (one block row: what the next leaf waits for)
    //   updA[k]   A(k+1,k+1) -= T(k+1,k) T(k+1,k)^T
    //   trsmB[k]  T(k+2..,k) = A(k+2..,k) Wkk^T
    //   updB[k]   columns k+1 .. pend (INCLUDING the first column of the next panel) -= rank-128 terms of column k
    // Panel p, once its last column is solved (K = w*128):
    //   next1[p]  column pend+1;  next2[p]  columns pend+2 .. pend+OB;  rest[p]  columns > pend+OB (lower tiles)
    const int ldw = s->ldw, ldt = s->ldt;
    auto tW = [&](int k) { return s->w_block(k); };
    auto tT = [&](int r, int k) { return s->t_block(r, k); };
    for (int k = 0; k + 1 < nblk; ++k) {
        const int pend = s->pan_hi[s->pan_of[k]];
        // the two products on the leaf chain run on the small-tile kernel: 16 (10 for the symmetric update) CTAs of 32x32
        grp.push_back(small(make_task3(at(s->A, k + 1, k), ld, tW(k), ldw, tT(k + 1, k), ldt, NB, NB, NB, 1, 1, 0, GM_KRULE_ALL, 1.0, 0.0)));
        s->trsmA.push_back(push_group(grp));
        grp.push_back(small(make_task3(tT(k + 1, k), ldt, tT(k + 1, k), ldt, at(s->A, k + 1, k + 1), ld, NB, NB, NB, 1, 1, 1, GM_KRULE_ALL, -1.0, 1.0)));
        s->updA.push_back(push_group(grp));
        const int below = np - (k + 2) * NB;
        if (below > 0)
            grp.push_back(make_task3(at(s->A, k + 2, k), ld, tW(k), ldw, tT(k + 2, k), ldt, below, NB, NB, 1, 1, 0, GM_KRULE_ALL, 1.0, 0.0));
        s->trsmB.push_back(push_group(grp));
        if (below > 0)     // column k+1 below its diagonal block
            grp.push_back(make_task3(tT(k + 2, k), ldt, tT(k + 1, k), ldt, at(s->A, k + 2, k + 1), ld, below, NB, NB, 1, 1, 0, GM_KRULE_ALL, -1.0, 1.0));
        for (int c = k + 2; c <= std::min(pend, nblk - 1); ++c)
            grp.push_back(make_task3(tT(c, k), ldt, tT(c, k), ldt, at(s->A, c, c), ld, np - c * NB, NB, NB, 1, 1, 0, GM_KRULE_ALL, -1.0, 1.0));
        s->updB.push_back(push_group(grp));
    }
    for (size_t p = 0; p < s->pan_lo.size(); ++p) {
        const int p0 = s->pan_lo[p], pend = s->pan_hi[p], w = pend - p0;
        const int pnext = p + 1 < s->pan_hi.size() ? s->pan_hi[p + 1] : nblk;      // end of the next panel
        const int c1 = pend + 1, c2 = pend + 2, c2e = std::min(pnext, nblk - 1), c3 = pnext + 1;
        if (c1 < nblk)
            grp.push_back(make_task3(tT(c1, p0), ldt, tT(c1, p0), ldt, at(s->A, c1, c1), ld, np - c1 * NB, NB, w * NB, 1, 1, 0, GM_KRULE_ALL, -1.0, 1.0));
        s->next1.push_back(push_group(grp));
        if (c2 <= c2e)
            grp.push_back(make_task3(tT(c2, p0), ldt, tT(c2, p0), ldt, at(s->A, c2, c2), ld, np - c2 * NB, (c2e - c2 + 1) * NB, w * NB, 1, 1, 0, GM_KRULE_ALL, -1.0, 1.0));
        s->next2.push_back(push_group(grp));
        if (c3 < nblk)
            grp.push_back(make_task3(tT(c3, p0), ldt, tT(c3, p0), ldt, at(s->A, c3, c3), ld, np - c3 * NB, np - c3 * NB, w * NB, 1, 1, 1, GM_KRULE_ALL, -1.0, 1.0));
        s->rest.push_back(push_group(grp));
    }
    if (!s->lean) {
    // trtri levels: spans of `span` blocks are already inverted; join neighbours pairwise
    for (int span = 1; span < nblk; span *= 2) {
        std::vector<GemmTask> gt, gw;
        for (int o = 0; o + span < nblk; o += 2 * span) {
            const int h1 = span, h2 = std::min(span, nblk - (o + span));
            // T21 = L21 * W11   (W11 lower-triangular as the K x N operand)
            gt.push_back(make_task(at(s->A, o + h1, o), at(s->W, o, o), at(s->T, o + h1, o), h2 * NB, h1 * NB, h1 * NB, ld, 1, 0, 0, GM_KRULE_B_LOWER, 1.0, 0.0));
            // W21 = -W22 * T21  (W22 lower-triangular as the M x K operand)
            gw.push_back(make_task(at(s->W, o + h1, o + h1), at(s->T, o + h1, o), at(s->W, o + h1, o), h2 * NB, h1 * NB, h2 * NB, ld, 1, 0, 0, GM_KRULE_A_LOWER, -1.0, 0.0));
        }
        s->tri_t.push_back(push_group(gt));
        s->tri_w.push_back(push_group(gw));
    }
    // lauum: Ainv = W^T W  (both operands row-contiguous: A[k][m] = W[k][m])
    grp.push_back(make_task(s->W, s->W, s->T, np, np, np, ld, 0, 0, 1, GM_KRULE_LAUUM, 1.0, 0.0));
    s->lauum = push_group(grp);
    // prediction: V[m][c] = sum_k W[m][k] strip[c][k]  (W lower-triangular, both operands k-contiguous)
    {
        GemmTask t = make_task(s->W, s->strip, s->V, np, NB, np, ld, 1, 1, 0, GM_KRULE_A_LOWER, 1.0, 0.0);
        t.ldc = NB;
        grp.push_back(t);
        s->quad = push_group(grp);
    }
    }   // !lean

    e = cudaMalloc(&s->d_tasks, sizeof(GemmTask) * tasks.size());
    if (e == cudaSuccess) e = cudaMemcpy(s->d_tasks, tasks.data(), sizeof(GemmTask) * tasks.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) gemm_register_maps(s->d_tasks, tasks.data(), (int)tasks.size());      // tensor maps of the operands
    if (e == cudaSuccess) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        e = cudaStreamCreateWithPriority(&s->helper, cudaStreamNonBlocking, hi);
        // panel work: above the caller's bulk updates, below the leaf chain when the device has a level in between
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s->mid, cudaStreamNonBlocking, (hi + 1 < lo) ? hi + 1 : hi);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_join2, cudaEventDisableTiming);
    auto make_events = [&](std::vector<cudaEvent_t>& v, int count) {
        for (int i = 0; i < count && e == cudaSuccess; ++i) {
            cudaEvent_t ev;
            e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (e == cudaSuccess) v.push_back(ev);
        }
    };
    make_events(s->ev_leaf, nblk); make_events(s->ev_a, nblk); make_events(s->ev_b, nblk);
    make_events(s->ev_n1, (int)s->pan_lo.size()); make_events(s->ev_n2, (int)s->pan_lo.size());
    {
        int cnt = nblk;
        for (int k = 0; k + 1 < nblk; ++k) cnt += 2 + (s->trsmB[k].tiles > 0) + (s->updB[k].tiles > 0);
        for (size_t p = 0; p < s->rest.size(); ++p) cnt += (s->next1[p].tiles > 0) + (s->next2[p].tiles > 0) + (s->rest[p].tiles > 0);
        s->potrf_launches = cnt;
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming);
    make_events(s->ev_rest, (int)s->pan_lo.size());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(potrf_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LEAF_SMEM_V2);
    if (e != cudaSuccess) { dqgp_solver_destroy(s); return cuda_fail(e, "dqgp_solver_create (task table)"); }
    int rc = gemm_init();
    if (rc) { dqgp_solver_destroy(s); return rc; }
    *out = s;
    return 0;
}

extern "C" {

void dqgp_solver_destroy(dqgp_solver* s) {
    if (!s) return;
    for (auto* v : {&s->ev_leaf, &s->ev_a, &s->ev_b, &s->ev_n1, &s->ev_n2, &s->ev_rest})
        for (auto ev : *v) cudaEventDestroy(ev);
    if (s->ev_join2) cudaEventDestroy(s->ev_join2);
    if (s->mid) cudaStreamDestroy(s->mid);
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
    if (s->helper) cudaStreamDestroy(s->helper);
    dqgp::gemm_unregister_maps(s->d_tasks);
    cudaFree(s->A); cudaFree(s->W); cudaFree(s->T); cudaFree(s->y_pad); cudaFree(s->w); cudaFree(s->partial); cudaFree(s->strip); cudaFree(s->V); cudaFree(s->d_tasks); cudaFree(s->d_dyn); cudaFree(s->tmp);
    delete s;
}
int dqgp_solver_n(const dqgp_solver* s) { return s ? s->n : -1; }
int dqgp_solver_ld(const dqgp_solver* s) { return s ? s->ld : -1; }
double* dqgp_solver_matrix(dqgp_solver* s) { return s ? s->A : nullptr; }
double* dqgp_solver_inverse(dqgp_solver* s) { return (s && !s->lean) ? s->T : nullptr; }
double* dqgp_solver_factor(dqgp_solver* s) { return s ? s->A : nullptr; }
size_t dqgp_solver_bytes(const dqgp_solver* s) { return s ? s->bytes : 0; }
int dqgp_solver_potrf_launches(const dqgp_solver* s) { return s ? s->potrf_launches : -1; }

int dqgp_potrf_solve_inv(dqgp_solver* s, const double* d_y, double* d_alpha, double* d_logdet, int* d_info, int want_inverse,
                         void* stream) {
    using namespace dqgp;
    const bool factor_only = want_inverse < 0;
    DQGP_REQUIRE(s && d_logdet && d_info && (factor_only || (d_y && d_alpha)), "dqgp_potrf_solve_inv: NULL argument");
    cudaStream_t st = as_stream(stream);
    const int np = s->np, ld = s->ld, nblk = s->nblk;
    pad_vector_kernel<<<(np + 255) / 256, 256, 0, st>>>(factor_only ? nullptr : d_y, s->n, np, s->y_pad, d_logdet, d_info);
    if (np != s->n) pad_identity_kernel<<<np, 256, 0, st>>>(s->A, s->n, np, ld);
    DQGP_LAUNCH_CHECK("pad kernels");
    {
        int rc = potrf_lookahead(s, d_logdet, d_info, st);
        if (rc) return rc;
    }
    if (s->lean) {
        // L is already in place.  alpha = L^-T (L^-1 y) by blocked substitution through the inverted diagonal blocks.
        DQGP_REQUIRE(want_inverse <= 0, "dqgp_potrf_solve_inv: a lean solver holds no triangular inverse / A^-1 (want_inverse must be <= 0)");
        if (factor_only) return 0;
        double* y = s->y_pad;
        for (int k = 0; k < nblk; ++k) {
            diag_block_mv_kernel<<<1, NB, 0, st>>>(s->w_block(k), s->ldw, y + (size_t)k * NB, y + (size_t)k * NB, 0);
            const int rows = np - (k + 1) * NB;
            if (rows > 0) subst_forward_update_kernel<<<(rows + 7) / 8, 256, 0, st>>>(s->A, ld, k, np, y + (size_t)k * NB, y);
        }
        for (int k = nblk - 1; k >= 0; --k) {
            diag_block_mv_kernel<<<1, NB, 0, st>>>(s->w_block(k), s->ldw, y + (size_t)k * NB, y + (size_t)k * NB, 1);
            if (k > 0) subst_backward_update_kernel<<<(k * NB + 255) / 256, 256, 0, st>>>(s->A, ld, k, y + (size_t)k * NB, y);
        }
        DQGP_LAUNCH_CHECK("substitution kernels");
        DQGP_CUDA(cudaMemcpyAsync(d_alpha, y, sizeof(double) * s->n, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    if (nblk > 1) {
        copy_lower_blocks_kernel<<<dim3(nblk - 1, nblk - 1), 256, 0, st>>>(s->T, s->A, ld);
        DQGP_LAUNCH_CHECK("copy_lower_blocks_kernel");
    }
    if (factor_only) return 0;      // L is in place (dqgp_solver_factor); its diagonal-block inverses are in W
    for (size_t l = 0; l < s->tri_t.size(); ++l) {
        int rc = launch_gemm_group(s->d_tasks + s->tri_t[l].first, s->tri_t[l].count, s->tri_t[l].tiles, st);
        if (rc) return rc;
        rc = launch_gemm_group(s->d_tasks + s->tri_w[l].first, s->tri_w[l].count, s->tri_w[l].tiles, st);
        if (rc) return rc;
    }
    // alpha = W^T (W y)
    trmv_lower_kernel<<<(np + 7) / 8, 256, 0, st>>>(s->W, np, ld, s->y_pad, s->w);
    trmv_lower_T_partial_kernel<<<dim3(nblk, nblk), NB, 0, st>>>(s->W, ld, s->w, s->partial, np);
    reduce_partial_kernel<<<(s->n + 255) / 256, 256, 0, st>>>(s->partial, nblk, np, s->n, d_alpha);
    DQGP_LAUNCH_CHECK("solve kernels");
    if (want_inverse) {
        int rc = launch_gemm_group(s->d_tasks + s->lauum.first, s->lauum.count, s->lauum.tiles, st);
        if (rc) return rc;
        if (want_inverse > 1) {
            symmetrize_lower_kernel<<<dim3(np / 32, np / 32), 256, 0, st>>>(s->T, ld);
            DQGP_LAUNCH_CHECK("symmetrize_lower_kernel");
        }
    }
    return 0;
}

int dqgp_solver_apply_factor(dqgp_solver* s, const double* d_x, double* d_y, void* stream) {
    // y = L x with the Cholesky factor held by the solver (sampling from N(0, K): main.py:272-274)
    using namespace dqgp;
    DQGP_REQUIRE(s && d_x && d_y, "dqgp_solver_apply_factor: NULL argument");
    cudaStream_t st = as_stream(stream);
    pad_vector_kernel<<<(s->np + 255) / 256, 256, 0, st>>>(d_x, s->n, s->np, s->y_pad, s->w, reinterpret_cast<int*>(s->w + 1));
    trmv_lower_kernel<<<(s->np + 7) / 8, 256, 0, st>>>(s->A, s->np, s->ld, s->y_pad, s->partial);
    DQGP_LAUNCH_CHECK("apply_factor kernels");
    DQGP_CUDA(cudaMemcpyAsync(d_y, s->partial, sizeof(double) * s->n, cudaMemcpyDeviceToDevice, st));
    return 0;
}

int dqgp_solver_quadform_rows_inplace(dqgp_solver* s, double* d_B, int nb_pad, int ldb, double* d_out, void* stream) {
    // Row i of B (nb_pad, ldb) is replaced by (L^-1 b_i)^T and d_out[i] = || L^-1 b_i ||^2 (main.py:1462-1463), by blocked
    // forward substitution on the DMMA GEMM: for every 128-column block k
    //     B[:, k] -= B[:, 0..k) L[k, 0..k)^T        (contraction over everything already solved)
    //     B[:, k]  = B[:, k] Wkk^T                  (inverted diagonal block)
    // Needs only L and the diagonal-block inverses, so it works on a lean solver: the right-hand sides are the only
    // other large buffer (n^2 nb flops in place, no second square).
    using namespace dqgp;
    DQGP_REQUIRE(s && d_B && d_out && nb_pad > 0 && nb_pad % NB == 0 && ldb >= s->np && (ldb & 1) == 0,
                 "dqgp_solver_quadform_rows_inplace: B must have a multiple of 128 rows and an even leading dimension >= %d "
                 "(columns n..n_pad zero)", s ? s->np : 0);
    DQGP_REQUIRE((reinterpret_cast<uintptr_t>(d_B) & 15) == 0, "dqgp_solver_quadform_rows_inplace: B must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const int nblk = s->nblk, ld = s->ld;
    if ((size_t)nb_pad > s->tmp_rows) {
        DQGP_CUDA(cudaStreamSynchronize(st));
        cudaFree(s->tmp); s->tmp = nullptr; s->tmp_rows = 0;
        DQGP_CUDA(cudaMalloc(&s->tmp, sizeof(double) * (size_t)nb_pad * NB));
        s->tmp_rows = nb_pad;
    }
    if (2 * nblk > s->dyn_capacity) {
        DQGP_CUDA(cudaStreamSynchronize(st));
        cudaFree(s->d_dyn); s->d_dyn = nullptr; s->dyn_capacity = 0;
        DQGP_CUDA(cudaMalloc(&s->d_dyn, sizeof(GemmTask) * 2 * nblk));
        s->dyn_capacity = 2 * nblk;
    }
    std::vector<GemmTask> dyn(2 * nblk);
    for (int k = 0; k < nblk; ++k) {
        // [2k]   B[:, k] -= B[:, 0..k) L[k, 0..k)^T ;  [2k+1] tmp = B[:, k] Wkk^T
        dyn[2 * k] = make_task3(d_B, ldb, s->A + (size_t)k * NB * ld, ld, d_B + (size_t)k * NB, ldb, nb_pad, NB, std::max(k, 1) * NB, 1, 1, 0,
                                GM_KRULE_ALL, -1.0, 1.0);
        dyn[2 * k + 1] = make_task3(d_B + (size_t)k * NB, ldb, s->w_block(k), s->ldw, s->tmp, NB, nb_pad, NB, NB, 1, 1, 0, GM_KRULE_ALL, 1.0, 0.0);
    }
    DQGP_CUDA(cudaMemcpyAsync(s->d_dyn, dyn.data(), sizeof(GemmTask) * dyn.size(), cudaMemcpyHostToDevice, st));
    for (int k = 0; k < nblk; ++k) {
        int rc = 0;
        if (k > 0) rc = launch_gemm_group(s->d_dyn + 2 * k, 1, dyn[2 * k].tiles, st);
        if (rc) return rc;
        rc = launch_gemm_group(s->d_dyn + 2 * k + 1, 1, dyn[2 * k + 1].tiles, st);
        if (rc) return rc;
        subst_store_sumsq_kernel<<<(nb_pad + 7) / 8, 256, 0, st>>>(s->tmp, d_B, ldb, k, nb_pad, d_out, k == 0);
        DQGP_LAUNCH_CHECK("subst_store_sumsq_kernel");
    }
    return 0;
}

int dqgp_solver_quadform_rows(dqgp_solver* s, const double* d_B, int nb, int ldb, double* d_out, void* stream) {
    // d_out[i] = || L^-1 b_i ||^2 for every row b_i of B (nb, n): V = W B^T in strips of 128 rows of B on the
    // DMMA GEMM, then fixed-order column sums of squares (main.py:1462-1463).
    using namespace dqgp;
    DQGP_REQUIRE(s && d_B && d_out && nb >= 0 && ldb >= s->n, "dqgp_solver_quadform_rows: bad arguments");
    DQGP_REQUIRE(!s->lean, "dqgp_solver_quadform_rows: a lean solver has no L^-1; use dqgp_solver_quadform_rows_inplace");
    cudaStream_t st = as_stream(stream);
    for (int r0 = 0; r0 < nb; r0 += NB) {
        const int cnt = std::min(NB, nb - r0);
        copy_pad_rows_kernel<<<NB, 256, 0, st>>>(d_B + (size_t)r0 * ldb, cnt, s->n, ldb, s->strip, NB, s->np, s->ld);
        int rc = launch_gemm_group(s->d_tasks + s->quad.first, s->quad.count, s->quad.tiles, st);
        if (rc) return rc;
        colsumsq_kernel<<<1, NB, 0, st>>>(s->V, s->n, NB, cnt, d_out + r0);
        DQGP_LAUNCH_CHECK("quadform kernels");
    }
    return 0;
}

}  // extern "C"
