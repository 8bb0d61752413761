// Device-side LU fallback for matrices the Cholesky rejects (sm_100a; fp64).
//
// The reference walks a ladder when np.linalg.cholesky raises: the agent step factors C + sigma^2 I with
// scipy.linalg.lu_factor and solves for alpha and for the explicit inverse against eye(n)
// (agent_riemannian.py:419-425); the prediction path inverts with np.linalg.inv = getrf + getri (main.py:1479-1486).
// Both are partial-pivoting LU, so this file is one: a right-looking blocked LU (32-column panels, row-major storage,
// LAPACK's pivot rule: first entry of maximal modulus), the two blocked triangular solves for any number of right-hand
// sides, slogdet (agent_riemannian.py:442), and a general tile GEMM for the prediction's K(test,train) A^-1 product.
// It is the EXCEPTION path - e.g. ExpSineSquared of a Euclidean distance is indefinite in more than one dimension - so
// it is written for correctness and bounded cost (O(n^3) on the FP64 pipe with coalesced tiles, every loop bound known on
// the host so the whole sequence is stream-ordered and needs no host synchronisation), not to the factorisation's roofline.
// Everything is deterministic: single-CTA panel, fixed-order reductions.
#include "common.cuh"

namespace dqgp {

constexpr int LU_PB = 32;          // panel width
constexpr int LU_PANEL_THREADS = 1024;

// ---- panel: columns [k0, k0+pb) of rows [k0, n), unblocked with partial pivoting, one CTA -------------------------------
__global__ void __launch_bounds__(LU_PANEL_THREADS) lu_panel_kernel(double* __restrict__ A, int ld, int n, int k0, int pb,
                                                                    int* __restrict__ piv) {
    __shared__ double s_val[LU_PANEL_THREADS / 32];
    __shared__ int s_idx[LU_PANEL_THREADS / 32];
    __shared__ double s_row[LU_PB];
    __shared__ int s_p;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int j = 0; j < pb; ++j) {
        const int col = k0 + j;
        // pivot: first row of maximal |A[i][col]|, i >= col (LAPACK idamax); NaN never wins a comparison, as in LAPACK
        double best = -1.0;
        int bi = col;
        for (int i = col + tid; i < n; i += LU_PANEL_THREADS) {
            const double v = fabs(A[(size_t)i * ld + col]);
            if (v > best) { best = v; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) { s_val[warp] = best; s_idx[warp] = bi; }
        __syncthreads();
        if (tid == 0) {
            double b = s_val[0];
            int p = s_idx[0];
            for (int w = 1; w < LU_PANEL_THREADS / 32; ++w)
                if (s_val[w] > b || (s_val[w] == b && s_idx[w] < p)) { b = s_val[w]; p = s_idx[w]; }
            s_p = p;
            piv[col] = p;
        }
        __syncthreads();
        const int p = s_p;
        // swap rows col <-> p inside the panel, keep the pivot row's tail in shared memory
        if (tid < pb) {
            const double a = A[(size_t)col * ld + k0 + tid], b = A[(size_t)p * ld + k0 + tid];
            if (p != col) { A[(size_t)col * ld + k0 + tid] = b; A[(size_t)p * ld + k0 + tid] = a; }
            s_row[tid] = (p != col) ? b : a;
        }
        __syncthreads();
        const double d = s_row[j];
        if (d != 0.0) {                     // exact zero pivot: the column is already eliminated (LAPACK continues, info > 0)
            for (int i = col + 1 + tid; i < n; i += LU_PANEL_THREADS) {
                double* row = A + (size_t)i * ld + k0;
                const double l = row[j] / d;
                row[j] = l;
                for (int c = j + 1; c < pb; ++c) row[c] = fma(-l, s_row[c], row[c]);
            }
        }
        __syncthreads();
    }
}

// apply the panel's row interchanges to the columns outside the panel (thread = column)
__global__ void lu_swap_rows_kernel(double* __restrict__ A, int ld, int n, int k0, int pb, const int* __restrict__ piv) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n - pb) return;
    if (c >= k0) c += pb;
    for (int j = 0; j < pb; ++j) {
        const int r1 = k0 + j, r2 = piv[r1];
        if (r1 != r2) {
            const double a = A[(size_t)r1 * ld + c], b = A[(size_t)r2 * ld + c];
            A[(size_t)r1 * ld + c] = b;
            A[(size_t)r2 * ld + c] = a;
        }
    }
}

// X = T^-1 B for one 32-row block of right-hand sides, in place (thread = rhs column):
//   UNIT_LOWER: T = unit lower triangle of LU[k0:k0+pb, k0:k0+pb];  otherwise T = its upper triangle (with diagonal).
template <bool UNIT_LOWER>
__global__ void __launch_bounds__(128) lu_trsm_block_kernel(const double* __restrict__ LU, int ld, int k0, int pb, double* __restrict__ B,
                                                            int ldb, int c0, int ncols) {
    __shared__ double T[LU_PB][LU_PB + 1];
    for (int e = threadIdx.x; e < LU_PB * LU_PB; e += blockDim.x) {
        const int r = e / LU_PB, c = e % LU_PB;
        T[r][c] = (r < pb && c < pb) ? LU[(size_t)(k0 + r) * ld + k0 + c] : (r == c ? 1.0 : 0.0);
    }
    __syncthreads();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncols) return;
    double* b = B + (size_t)k0 * ldb + c0 + c;
    double x[LU_PB];
#pragma unroll
    for (int r = 0; r < LU_PB; ++r) x[r] = (r < pb) ? b[(size_t)r * ldb] : 0.0;
    if (UNIT_LOWER) {
#pragma unroll
        for (int r = 1; r < LU_PB; ++r) {
            double acc = x[r];
#pragma unroll
            for (int k = 0; k < r; ++k) acc = fma(-T[r][k], x[k], acc);
            x[r] = acc;
        }
    } else {
#pragma unroll
        for (int r = LU_PB - 1; r >= 0; --r) {
            double acc = x[r];
#pragma unroll
            for (int k = r + 1; k < LU_PB; ++k) acc = fma(-T[r][k], x[k], acc);
            x[r] = acc / T[r][r];
        }
    }
#pragma unroll
    for (int r = 0; r < LU_PB; ++r)
        if (r < pb) b[(size_t)r * ldb] = x[r];
}

// C(MxN) = beta*C + alpha * A(MxK) B(KxN); row-major, any sizes; 64x64 tile, 256 threads, 4x4 micro-tiles, K in chunks of 16
constexpr int LG_T = 64, LG_K = 16;
__global__ void __launch_bounds__(256) lu_gemm_kernel(int M, int N, int K, double alpha, const double* __restrict__ A, int lda,
                                                      const double* __restrict__ B, int ldb, double beta, double* __restrict__ C, int ldc) {
    __shared__ double As[LG_K][LG_T + 1];
    __shared__ double Bs[LG_K][LG_T];
    const int m0 = blockIdx.y * LG_T, n0 = blockIdx.x * LG_T;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    for (int k0 = 0; k0 < K; k0 += LG_K) {
        for (int e = threadIdx.x; e < LG_T * LG_K; e += 256) {
            const int r = e / LG_K, k = e % LG_K;             // A tile: consecutive threads walk k (contiguous in memory)
            As[k][r] = (m0 + r < M && k0 + k < K) ? A[(size_t)(m0 + r) * lda + k0 + k] : 0.0;
            const int kb = e / LG_T, c = e % LG_T;            // B tile: consecutive threads walk columns
            Bs[kb][c] = (k0 + kb < K && n0 + c < N) ? B[(size_t)(k0 + kb) * ldb + n0 + c] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < LG_K; ++k) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty + 16 * i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = m0 + ty + 16 * i;
        if (r >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = n0 + tx + 16 * j;
            if (c >= N) continue;
            double* dst = C + (size_t)r * ldc + c;
            *dst = (beta == 0.0) ? alpha * acc[i][j] : fma(beta, *dst, alpha * acc[i][j]);
        }
    }
}

// perm = the row permutation of the factorisation (row i of P A is row perm[i] of A): getrs' laswp on an index vector
__global__ void lu_perm_kernel(const int* __restrict__ piv, int n, int* __restrict__ perm) {
    extern __shared__ int s_perm[];
    int* p = s_perm;
    for (int i = threadIdx.x; i < n; i += blockDim.x) p[i] = i;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 0; i < n; ++i) {
            const int j = piv[i];
            if (j != i) { const int t = p[i]; p[i] = p[j]; p[j] = t; }
        }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) perm[i] = p[i];
}
__global__ void lu_perm_global_kernel(const int* __restrict__ piv, int n, int* __restrict__ perm) {      // n too large for shared memory
    for (int i = threadIdx.x; i < n; i += blockDim.x) perm[i] = i;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 0; i < n; ++i) {
            const int j = piv[i];
            if (j != i) { const int t = perm[i]; perm[i] = perm[j]; perm[j] = t; }
        }
}
// B = P (the permuted identity: B[i][perm[i]] = 1), y_p[i] = y[perm[i]]
__global__ void lu_init_rhs_kernel(const int* __restrict__ perm, int n, double* __restrict__ B, int ldb, const double* __restrict__ y,
                                   double* __restrict__ yp) {
    const int i = blockIdx.x;
    const int pi = perm[i];
    if (B)
        for (int c = threadIdx.x; c < n; c += blockDim.x) B[(size_t)i * ldb + c] = (c == pi) ? 1.0 : 0.0;
    if (threadIdx.x == 0 && y) yp[i] = y[pi];
}
// slogdet: out[0] = sum log|u_ii| (fixed-order tree), out[1] = sign (product of the signs of u_ii times the permutation's parity; 0 if singular)
__global__ void __launch_bounds__(256) lu_slogdet_kernel(const double* __restrict__ LU, int ld, int n, const int* __restrict__ piv,
                                                         double* __restrict__ out) {
    __shared__ double s_log[256];
    __shared__ int s_neg[256], s_zero[256];
    double acc = 0.0;
    int neg = 0, zero = 0;
    for (int i = threadIdx.x; i < n; i += 256) {
        const double u = LU[(size_t)i * ld + i];
        acc += log(fabs(u));
        neg += (u < 0.0) + (piv[i] != i);
        zero += (u == 0.0);
    }
    s_log[threadIdx.x] = acc; s_neg[threadIdx.x] = neg; s_zero[threadIdx.x] = zero;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { s_log[threadIdx.x] += s_log[threadIdx.x + o]; s_neg[threadIdx.x] += s_neg[threadIdx.x + o]; s_zero[threadIdx.x] += s_zero[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = s_log[0];
        out[1] = s_zero[0] ? 0.0 : ((s_neg[0] & 1) ? -1.0 : 1.0);
    }
}
// rows of (T o K): out[i] = sum_k T[i][k] K[i][k]   (one warp per row)
__global__ void lu_rowdot_kernel(const double* __restrict__ T, int ldt, const double* __restrict__ Kst, int ldk, int nt, int n,
                                 double* __restrict__ out) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= nt) return;
    double acc = 0.0;
    for (int k = lane; k < n; k += 32) acc = fma(T[(size_t)row * ldt + k], Kst[(size_t)row * ldk + k], acc);
    acc = warp_sum(acc);
    if (lane == 0) out[row] = acc;
}

static int lu_gemm(int M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb, double beta, double* C, int ldc,
                   cudaStream_t st) {
    if (M <= 0 || N <= 0) return 0;
    dim3 grid((N + LG_T - 1) / LG_T, (M + LG_T - 1) / LG_T);
    lu_gemm_kernel<<<grid, 256, 0, st>>>(M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
    DQGP_LAUNCH_CHECK("lu_gemm_kernel");
    return 0;
}

// in-place solve of (P A = L U) X = B for the ncols columns of B starting at column c0; rows of B must already be permuted
static int lu_solve_permuted(const double* LU, int ld, int n, double* B, int ldb, int c0, int ncols, cudaStream_t st) {
    const unsigned cb = (unsigned)((ncols + 127) / 128);
    for (int k0 = 0; k0 < n; k0 += LU_PB) {                                   // L Y = B
        const int pb = min(LU_PB, n - k0), rest = n - k0 - pb;
        lu_trsm_block_kernel<true><<<cb, 128, 0, st>>>(LU, ld, k0, pb, B, ldb, c0, ncols);
        int rc = lu_gemm(rest, ncols, pb, -1.0, LU + (size_t)(k0 + pb) * ld + k0, ld, B + (size_t)k0 * ldb + c0, ldb, 1.0,
                         B + (size_t)(k0 + pb) * ldb + c0, ldb, st);
        if (rc) return rc;
    }
    for (int k0 = ((n - 1) / LU_PB) * LU_PB; k0 >= 0; k0 -= LU_PB) {          // U X = Y
        const int pb = min(LU_PB, n - k0);
        lu_trsm_block_kernel<false><<<cb, 128, 0, st>>>(LU, ld, k0, pb, B, ldb, c0, ncols);
        int rc = lu_gemm(k0, ncols, pb, -1.0, LU + k0, ld, B + (size_t)k0 * ldb + c0, ldb, 1.0, B + c0, ldb, st);
        if (rc) return rc;
    }
    DQGP_LAUNCH_CHECK("lu solve kernels");
    return 0;
}

}  // namespace dqgp

extern "C" {

size_t dqgp_lu_workspace_bytes(int n) { return n > 0 ? (size_t)n * (2 * sizeof(int) + sizeof(double)) + 64 : 0; }

int dqgp_lu_solve_inv(double* d_A, int lda, int n, const double* d_y, double* d_alpha, double* d_Ainv, int ldi, double* d_slogdet,
                      void* d_work, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_A && d_work && n >= 1 && lda >= n, "dqgp_lu_solve_inv: bad arguments");
    DQGP_REQUIRE((d_y == nullptr) == (d_alpha == nullptr), "dqgp_lu_solve_inv: d_y and d_alpha go together");
    DQGP_REQUIRE(d_Ainv == nullptr || ldi >= n, "dqgp_lu_solve_inv: ldi < n");
    DQGP_REQUIRE(d_Ainv != d_A, "dqgp_lu_solve_inv: the inverse cannot overwrite the factors");
    cudaStream_t st = as_stream(stream);
    int* piv = static_cast<int*>(d_work);
    int* perm = piv + n;
    double* yp = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(perm + n) + 15) & ~uintptr_t(15));
    for (int k0 = 0; k0 < n; k0 += LU_PB) {
        const int pb = min(LU_PB, n - k0), rest = n - k0 - pb;
        lu_panel_kernel<<<1, LU_PANEL_THREADS, 0, st>>>(d_A, lda, n, k0, pb, piv);
        if (n > pb) lu_swap_rows_kernel<<<(n - pb + 255) / 256, 256, 0, st>>>(d_A, lda, n, k0, pb, piv);
        if (rest > 0) {
            lu_trsm_block_kernel<true><<<(rest + 127) / 128, 128, 0, st>>>(d_A, lda, k0, pb, d_A, lda, k0 + pb, rest);
            int rc = lu_gemm(rest, rest, pb, -1.0, d_A + (size_t)(k0 + pb) * lda + k0, lda, d_A + (size_t)k0 * lda + k0 + pb, lda, 1.0,
                             d_A + (size_t)(k0 + pb) * lda + k0 + pb, lda, st);
            if (rc) return rc;
        }
    }
    DQGP_LAUNCH_CHECK("lu factorisation kernels");
    if (d_slogdet) lu_slogdet_kernel<<<1, 256, 0, st>>>(d_A, lda, n, piv, d_slogdet);
    if (!d_Ainv && !d_y) return 0;
    if ((size_t)n * sizeof(int) <= 160 * 1024) {
        int rc = set_max_dynamic_smem<lu_perm_kernel>(160 * 1024);
        if (rc) return rc;
        lu_perm_kernel<<<1, 256, (size_t)n * sizeof(int), st>>>(piv, n, perm);
    } else {
        lu_perm_global_kernel<<<1, 256, 0, st>>>(piv, n, perm);
    }
    lu_init_rhs_kernel<<<n, 128, 0, st>>>(perm, n, d_Ainv, ldi, d_y, yp);
    DQGP_LAUNCH_CHECK("lu rhs kernels");
    if (d_y) {
        int rc = lu_solve_permuted(d_A, lda, n, yp, 1, 0, 1, st);
        if (rc) return rc;
        DQGP_CUDA(cudaMemcpyAsync(d_alpha, yp, sizeof(double) * n, cudaMemcpyDeviceToDevice, st));
    }
    if (d_Ainv) return lu_solve_permuted(d_A, lda, n, d_Ainv, ldi, 0, n, st);
    return 0;
}

int dqgp_dgemm_general(int M, int N, int K, double alpha, const double* d_A, int lda, const double* d_B, int ldb, double beta, double* d_C,
                       int ldc, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(M >= 0 && N >= 0 && K >= 0 && d_A && d_B && d_C && lda >= K && ldb >= N && ldc >= N, "dqgp_dgemm_general: bad arguments");
    return lu_gemm(M, N, K, alpha, d_A, lda, d_B, ldb, beta, d_C, ldc, as_stream(stream));
}

int dqgp_rowdot(const double* d_T, int ldt, const double* d_K, int ldk, int rows, int n, double* d_out, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_T && d_K && d_out && rows >= 0 && n >= 1 && ldt >= n && ldk >= n, "dqgp_rowdot: bad arguments");
    if (rows == 0) return 0;
    lu_rowdot_kernel<<<(rows + 7) / 8, 256, 0, as_stream(stream)>>>(d_T, ldt, d_K, ldk, rows, n, d_out);
    DQGP_LAUNCH_CHECK("lu_rowdot_kernel");
    return 0;
}
}
