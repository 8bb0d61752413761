/* dqgp.h — C-ABI of the B200-native engine for the distributed quantum-GP hot path.
 *
 * The reference (mpala-lab/distributed-quantum-gaussian-processes) has no FFI: its seams are Python
 * duck-typed calls into squlearn and NumPy.  Each entry point below names the reference interface it
 * replaces (file:line relative to the reference checkout).  INTEGRATION.md shows the ctypes stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory on the current CUDA device, contiguous row-major fp64
 *     (complex128 = interleaved re,im doubles); h_* is HOST memory;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all work is enqueued on it
 *     and nothing synchronises unless stated;
 *   - return value: 0 = ok, <0 = error (dqgp_last_error() gives a thread-local message); nothing throws;
 *   - no global mutable state; handles are immutable after creation and may be shared by streams,
 *     except dqgp_solver (owns scratch and internal streams: one in-flight use at a time);
 *   - read from the environment at call time: DQGP_POTRF_TRACE (diagnostic: time stamps of the Cholesky's leaf chain);
 *     DQGP_SV_NO_LC / DQGP_SV_FORCE_SHARED (test hooks: reach the two-fork / prefix-sharing simulator kernels at small sizes);
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef DQGP_H
#define DQGP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DQGP_VERSION 100

/* encoding circuits (reference ctor sites main.py:68-83, agent_riemannian.py:51-66) */
enum { DQGP_CHEBYSHEV = 0, DQGP_HUBREGTSEN = 1, DQGP_YZ_CX = 2, DQGP_KYRIIENKO = 3 };
/* outer kernels of the projected kernel (main.py:130-137, --outer-kernel main.py:1996-2013; sklearn RBF / Matern(1.5) /
 * ExpSineSquared / RationalQuadratic / DotProduct).  PairwiseKernel(metric="linear") is DOTPRODUCT with sigma_0 = 0. */
enum { DQGP_OUTER_GAUSSIAN = 0, DQGP_OUTER_MATERN15 = 1, DQGP_OUTER_EXPSINE2 = 2, DQGP_OUTER_RATQUAD = 3, DQGP_OUTER_DOTPRODUCT = 4 };
/* gate kinds / angle forms of the gate program (dqgp_circuit_describe) */
enum { DQGP_G_H = 0, DQGP_G_RX = 1, DQGP_G_RY = 2, DQGP_G_RZ = 3, DQGP_G_CX = 4, DQGP_G_CRZ = 5 };
enum { DQGP_A_NONE = 0, DQGP_A_P = 1, DQGP_A_X = 2, DQGP_A_P_PLUS_CX = 3, DQGP_A_P_TIMES_ACOS = 4, DQGP_A_C_TIMES_ACOS = 5 };

typedef struct dqgp_gate {
    int32_t kind;  /* DQGP_G_*                                   */
    int32_t q0;    /* target (1-qubit) or control (CX, CRZ)      */
    int32_t q1;    /* target of CX / CRZ, else -1                */
    int32_t form;  /* DQGP_A_*                                   */
    int32_t pidx;  /* parameter index or -1                      */
    int32_t fidx;  /* feature index or -1                        */
    double coef;   /* c in p + c*x  /  c*acos(x)                 */
} dqgp_gate;

typedef struct dqgp_circuit dqgp_circuit; /* immutable gate program resident on one device */
typedef struct dqgp_solver dqgp_solver;   /* workspace + task tables of the fp64 Cholesky / inverse */

int dqgp_version(void);
const char* dqgp_last_error(void);

/* ---- circuits: replaces squlearn ChebyshevPQC / HubregtsenEncodingCircuit / YZ_CX_EncodingCircuit /
 *      KyriienkoEncodingCircuit (num_qubits, num_features, num_layers); all other options at defaults. */
int dqgp_circuit_create(int encoding, int num_qubits, int num_features, int num_layers, dqgp_circuit** out);
void dqgp_circuit_destroy(dqgp_circuit* c);
int dqgp_circuit_num_parameters(const dqgp_circuit* c); /* = encoding_circuit.num_parameters (main.py:199) */
int dqgp_circuit_num_gates(const dqgp_circuit* c);
int dqgp_circuit_num_passes(const dqgp_circuit* c); /* shared-memory passes of the register-blocked simulator */
int dqgp_circuit_num_passes_cx_free(const dqgp_circuit* c); /* passes of the CX-free plan (CX gates absorbed into the index map);
                                                              0 when the circuit has CRZ gates or a parameter feeding several gates */
int dqgp_circuit_num_fused_ops(const dqgp_circuit* c); /* ops after fusing runs of 1-qubit gates (2x2 unitaries + CX/CRZ) */
/* executed simulator work per SAMPLE of dqgp_features_shifted / dqgp_states_shifted, in fused 2x2-unitary applications
 * (16 FMA = 32 flops per amplitude pair, 2^(q-1) pairs): bench.py's statevector roofline (SURVEY 8(d)).  Follows the CX-free plan
 * when the circuit has one (dqgp_circuit_num_passes_cx_free > 0), the CX-executing plan otherwise. */
long long dqgp_circuit_shifted_u2_applications(const dqgp_circuit* c);
int dqgp_circuit_describe(const dqgp_circuit* c, dqgp_gate* h_out, int capacity); /* host copy of the program */

/* ---- statevector simulation (what q_kernel.evaluate does per sample, agent_riemannian.py:118):
 *      d_X (n,d), d_Pm (S,P) parameter sets.  Features: d_F (S,n,3q) = [<X_k>],[<Y_k>],[<Z_k>];
 *      states: d_Psi (S,n,2^q) complex128. */
int dqgp_features(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int S, double* d_F, void* stream);
int dqgp_states(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int S, double* d_Psi, void* stream);

/* Same outputs for the 2P+1 central-difference sets of dqgp_shift_parameter_sets (d_Pm (2P+1,P): row 0 the base
 * set, rows 1+2i / 2+2i differing from it in parameter i only), computed with prefix sharing: the part of the circuit
 * that precedes the shifted gate is simulated once per sample.  Equal to dqgp_features / dqgp_states to rounding (2e-14): both
 * shifted sets of a rotation parameter are linear combinations of the base state and ONE forked state; features of circuits without
 * CRZ gates (yz_cx, kyriienko) run the CX-free plan (CX gates absorbed into a logical -> physical index map). */
int dqgp_features_shifted(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int P, double* d_F, void* stream);
int dqgp_states_shifted(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int P, double* d_Psi, void* stream);

/* ---- Gram matrices.  d_K (n1,n2) with leading dimension ldk (>= n2).
 *      projected: K = outer(f1_j, f2_k); hyp = {gamma} | {length_scale} | {length_scale, periodicity} |
 *      {length_scale, alpha} | {sigma_0} (NULL = all 1; ids as DQGP_OUTER_*) (ProjectedQuantumKernel.evaluate, main.py:130-137);
 *      fidelity: K = |<psi2_k|psi1_j>|^2 (FidelityKernel.evaluate, main.py:118-124). `same` != 0 promises the two operands are
 *      the same array so the diagonal of a stationary outer kernel is exactly outer(0) = 1 (the dot product's is
 *      sigma_0^2 + |f|^2, not overridden) and the mirror is exact; `same` == 2 (projected kernel) writes
 *      only the 64x64 tiles that intersect the lower triangle - all dqgp_potrf_solve_inv reads - and leaves
 *      the rest of d_K untouched.  Fidelity: dim = 2^q amplitudes with 1 <= q <= 12, and d_Psi1 / d_Psi2
 *      16-byte aligned (anything else returns < 0). */
int dqgp_gram_projected(int outer, const double* h_hyp, const double* d_F1, int n1, const double* d_F2, int n2, int m,
                        double* d_K, int ldk, int same, void* stream);
int dqgp_gram_fidelity(const double* d_Psi1, int n1, const double* d_Psi2, int n2, int dim, double* d_K, int ldk,
                       int same, void* stream);
/*      k(f_i, f_i) of the projected kernel for every row of d_F (n, m) -> d_out[n] (the predictive variance's prior term,
 *      main.py:1463): 1 for the stationary outer kernels (d_F is not read and may be NULL), sigma_0^2 + |f_i|^2 for the dot
 *      product (DotProduct.diag). */
int dqgp_projected_self_kernel(int outer, const double* h_hyp, const double* d_F, int n, int m, double* d_out, void* stream);

/* ---- fp64 Cholesky / solve / inverse (agent_riemannian.py:410-418, :442): for the SPD matrix
 *      A = K + sigma^2 I held in the solver (dqgp_solver_matrix, leading dimension dqgp_solver_ld):
 *      factor, alpha = A^-1 y, A^-1 (full symmetric, dqgp_solver_inverse), logdet(A).
 *      *d_info = 0 ok, j>0 = first non-positive pivot (1-based): the host then walks the reference's ladder
 *      (agent_riemannian.py:419-428) with dqgp_lu_solve_inv below.
 *      NOT computed here: the reference's `condition_number = np.linalg.cond(C)` (agent_riemannian.py:411), a 2-norm SVD of the
 *      UN-noised Gram used only in prints (main.py:2629-2642).  These Grams are numerically singular (cond ~ 1e17..1e19 in the
 *      golden files), so its value is rounding noise of that particular SVD; an estimate from this factorisation of C + sigma^2 I
 *      would be a different noise.  The Python layer returns NaN and offers a library SVD as a diagnostic opt-in. */
int dqgp_solver_create(int n, dqgp_solver** out);
/* outer_blocks: width of the outer Cholesky panel in 128-column blocks.  0 = default: 1 up to n = 6144 (bound by the leaf chain),
 * 4 above (rank-512 trailing updates: best throughput when several agents share a GPU); < 0 = width 4 while more than 28 block columns remain and 2
 * afterwards (one agent per GPU: wide while the trailing updates bound the factorisation, narrow once the leaf chain does). */
int dqgp_solver_create_ex(int n, int outer_blocks, dqgp_solver** out);
/* Lean solver for prediction / CV at full-train scale (main.py:1364-1596; SURVEY 8(f) row 1): ONE padded square (A, factored
 * in place) + the inverted 128x128 diagonal blocks + two rotating panel buffers, instead of three squares.  Supports
 * dqgp_potrf_solve_inv with want_inverse <= 0 (alpha by blocked substitution), dqgp_solver_apply_factor and
 * dqgp_solver_quadform_rows_inplace; no triangular inverse, no A^-1.  n = 117964 (config 5's training set) needs 112 GB. */
int dqgp_solver_create_lean(int n, int outer_blocks, dqgp_solver** out);
int dqgp_solver_is_lean(const dqgp_solver* s);
void dqgp_solver_destroy(dqgp_solver* s);
int dqgp_solver_n(const dqgp_solver* s);
int dqgp_solver_ld(const dqgp_solver* s);
double* dqgp_solver_matrix(dqgp_solver* s);  /* (n, ld): write A here (lower triangle is what is read) */
double* dqgp_solver_inverse(dqgp_solver* s); /* (n, ld): A^-1 after dqgp_potrf_solve_inv: want_inverse=1 fills the
                                              * lower 128x128 tiles (what the fused gradient reads), =2 the full matrix */
double* dqgp_solver_factor(dqgp_solver* s);  /* (n, ld): L (lower) after the call                      */
size_t dqgp_solver_bytes(const dqgp_solver* s);
int dqgp_solver_potrf_launches(const dqgp_solver* s); /* kernel launches of the Cholesky stage (bench launch accounting) */
int dqgp_add_diagonal(double* d_A, int n, int lda, double value, void* stream);
/* want_inverse: <0 factor only, 0 factor + alpha + logdet, 1 + A^-1 (lower tiles), 2 + A^-1 (full symmetric).
 * Enqueues on `stream` and on the solver's two internal high-priority streams (the leaf chain and the panel work of the
 * look-ahead schedule; both are forked from and joined back to `stream`, so the call is graph-capturable and ordered like
 * any other work on `stream`).  A lean solver accepts want_inverse <= 0 only. */
int dqgp_potrf_solve_inv(dqgp_solver* s, const double* d_y, double* d_alpha, double* d_logdet, int* d_info,
                         int want_inverse, void* stream);
/* want_inverse < 0 in dqgp_potrf_solve_inv = factor only (d_y, d_alpha may be NULL).
 * y = L x with the factor held by the solver: sampling from the GP prior (main.py:272-274). */
int dqgp_solver_apply_factor(dqgp_solver* s, const double* d_x, double* d_y, void* stream);
/* v = L^-1 B^T for B (nb, n): returns column sums of v^2 -> d_out[nb] (main.py:1462-1463) */
int dqgp_solver_quadform_rows(dqgp_solver* s, const double* d_B, int nb, int ldb, double* d_out, void* stream);

/* Same quantity by in-place blocked forward substitution (works on lean solvers): d_B (nb_pad, ldb) with nb_pad a multiple
 * of 128, ldb >= n_pad = dqgp_solver_ld() and even, 16-byte aligned, columns n..n_pad zero; rows are OVERWRITTEN by
 * (L^-1 b_i)^T, d_out[nb_pad] receives the squared norms.  Grows the solver's scratch on first use with a larger nb_pad
 * (synchronises `stream` then; not graph-capturable at that moment). */
int dqgp_solver_quadform_rows_inplace(dqgp_solver* s, double* d_B, int nb_pad, int ldb, double* d_out, void* stream);

/* ---- the reference's fallback ladder when np.linalg.cholesky raises (`info` > 0 above):
 *      agent step: scipy.linalg.lu_factor + lu_solve for alpha and for the explicit inverse against eye(n), then slogdet
 *      (agent_riemannian.py:419-425, :442); prediction: np.linalg.inv = getrf + getri (main.py:1479-1486).
 *      dqgp_lu_solve_inv factors d_A (n x n, row-major, leading dimension lda; BOTH triangles must be filled) in place as
 *      P A = L U with partial pivoting (LAPACK's pivot rule), and writes - each optional, pass NULL to skip -
 *      d_alpha = A^-1 y (by the two triangular solves, as lu_solve), d_Ainv = A^-1 (n x n, leading dimension ldi),
 *      d_slogdet[2] = {log|det A|, sign(det A)} (numpy.linalg.slogdet).  d_work: dqgp_lu_workspace_bytes(n) bytes.
 *      Stream-ordered, no host synchronisation, deterministic.  The third rung (np.linalg.pinv, :427-428) is only reached
 *      when LAPACK raises on non-finite input; non-finite input propagates NaN here instead.
 *      This is the exception path (e.g. ExpSineSquared Grams are indefinite): correct and O(n^3), not tuned to a roofline. */
size_t dqgp_lu_workspace_bytes(int n);
int dqgp_lu_solve_inv(double* d_A, int lda, int n, const double* d_y, double* d_alpha, double* d_Ainv, int ldi,
                      double* d_slogdet, void* d_work, void* stream);
/*      helpers of the prediction fallback (main.py:1482-1486: mean = K_st (A^-1 y), var = diag(K_ss - K_st A^-1 K_st^T)):
 *      C = beta C + alpha A B for row-major operands of any size; out[i] = <T[i,:], K[i,:]>. */
int dqgp_dgemm_general(int M, int N, int K, double alpha, const double* d_A, int lda, const double* d_B, int ldb,
                       double beta, double* d_C, int ldc, void* stream);
int dqgp_rowdot(const double* d_T, int ldt, const double* d_K, int ldk, int rows, int n, double* d_out, void* stream);

/* fp64 GEMM building block on the DMMA tensor path (used by the factorisation; exposed for tests):
 * C(MxN) = alpha*A*B + beta*C; A is [m][k] if a_k_contig else [k][m]; B is [n][k] if b_k_contig else [k][n].
 * M, N multiples of 128; K multiple of 16; even leading dimensions; 16-byte aligned pointers.
 * Test utility: allocates its one-entry task table with cudaMallocAsync and synchronises `stream` once. */
int dqgp_dgemm(int a_k_contig, int b_k_contig, int M, int N, int K, double alpha, const double* d_A, int lda,
               const double* d_B, int ldb, double beta, double* d_C, int ldc, void* stream);

/* ---- parameter sets of the central-difference ("parameter shift") rule
 *      (agent_riemannian.py:219,245-256 and the worker's wrap :41): d_Pm (2P+1, P). */
int dqgp_shift_parameter_sets(const double* d_z, int P, double h, double period, double* d_Pm, void* stream);

/* ---- fused gradient: grad_i = 1/2 sum_jk (A^-1 - alpha alpha^T)_jk (K(p+h e_i) - K(p-h e_i))_kj / (2h)
 *      (agent_riemannian.py:270-275 and :431-436) without materialising any shifted Gram.
 *      d_F: (2P+1, n, m) features / d_Psi: (2P+1, n, dim) states of the sets in dqgp_shift_parameter_sets
 *      order; d_Ainv (n, ld).  d_work: dqgp_grad_workspace_bytes(n, P) bytes.  d_grad[P] is UNROUNDED.
 *      Every outer kernel; the dot product's diagonal k(f_j, f_j) depends on the parameters and enters the sum.
 *      Fidelity: dim = 2^q amplitudes with 1 <= q <= 12, and d_Psi 16-byte aligned (anything else returns < 0). */
size_t dqgp_grad_workspace_bytes(int n, int P);
int dqgp_grad_projected(int outer, const double* h_hyp, const double* d_Ainv, int ld, const double* d_alpha,
                        const double* d_F, int n, int m, int P, double h, double* d_grad, void* d_work, void* stream);
int dqgp_grad_fidelity(const double* d_Ainv, int ld, const double* d_alpha, const double* d_Psi, int n, int dim, int P,
                       double h, double* d_grad, void* d_work, void* stream);

/* ---- analytic gradient (OPT-IN, SURVEY 8(f) row 3: the true derivative, not the reference's central difference with
 *      h = pi/8 - trajectories differ from the reference's; replaces the dead evaluate_derivatives branch,
 *      agent_riemannian.py:402-404).  dqgp_features_jacobian: d_F (n,3q) features at d_p (P) and d_J (P,n,3q) their exact
 *      derivatives, one extra suffix simulation per parameter (every parameter must feed exactly one gate).
 *      dqgp_grad_projected_analytic: every outer id (DQGP_OUTER_*), h_hyp as for dqgp_grad_projected ({gamma} | {length_scale} |
 *      {length_scale, periodicity} | {length_scale, alpha} | {sigma_0}); d_Ainv the FULL symmetric A^-1 (want_inverse = 2);
 *      m = 3q, q <= 12.  With B = A^-1 - alpha alpha^T, s = |f_j - f_k|^2 and d = sqrt(s), one pass over the n^2 entries
 *      (one outer-kernel derivative per entry instead of 2P kernels) gives
 *        stationary K = kappa(s): grad_i = 2 sum_j <J_i,j, G_j>, G_j = sum_k B_jk kappa'(s_jk) (f_j - f_k), with kappa'(s) =
 *          gaussian -gamma e^{-gamma s}; matern -(3/2) e^{-sqrt(3) d / l} / l^2;
 *          expsinesquared -(pi / (p l^2)) (sin(2 pi d / p) / d) K (limit -2 pi^2 / (p l)^2 at d = 0);
 *          rationalquadratic -(1 / (2 l^2)) (1 + s / (2 alpha l^2))^(-alpha-1);
 *        dotproduct K = sigma_0^2 + f_j.f_k: grad_i = sum_j <J_i,j, (B F)_j> (diagonal included; sigma_0 drops out).
 *      d_work: dqgp_grad_analytic_workspace_bytes(n, m). */
int dqgp_features_jacobian(const dqgp_circuit* c, const double* d_X, int n, const double* d_p, double* d_F, double* d_J, void* stream);
/* fidelity kernel: d_Psi (n,2^q) states at d_p and d_D (P,n,2^q) their derivatives d psi / dp_i (complex128);
 * dqgp_grad_fidelity_analytic: grad_i = 2 Re sum_j <G_j | d_i psi_j>, G_j = sum_k (A^-1 - alpha alpha^T)_jk <psi_k|psi_j> psi_k; d_Ainv
 *      the FULL symmetric A^-1 (want_inverse = 2); dim = 2^q, 1 <= q <= 12.  From dim = 128 on, d_Psi and d_work must be 16-byte
 *      aligned; d_work: dqgp_grad_fidelity_analytic_workspace_bytes(n, dim).  Deterministic: a second call gives the same bits. */
int dqgp_states_jacobian(const dqgp_circuit* c, const double* d_X, int n, const double* d_p, double* d_Psi, double* d_D, void* stream);
size_t dqgp_grad_fidelity_analytic_workspace_bytes(int n, int dim);
int dqgp_grad_fidelity_analytic(const double* d_Ainv, int ld, const double* d_alpha, const double* d_Psi, const double* d_D, int n,
                                int dim, int P, double* d_grad, void* d_work, void* stream);
size_t dqgp_grad_analytic_workspace_bytes(int n, int m);
int dqgp_grad_projected_analytic(int outer, const double* h_hyp, const double* d_Ainv, int ld, const double* d_alpha,
                                 const double* d_F, const double* d_J, int n, int m, int P, double* d_grad, void* d_work,
                                 void* stream);

/* ---- NLL gradient with respect to the outer kernel's hyper-parameters and the noise level (type-II maximum likelihood; the
 *      reference has none: it never applies outer-kernel hyper-parameters).  With A = K + sigma^2 I, alpha = A^-1 y,
 *      B = A^-1 - alpha alpha^T and NLL = 1/2 log det A + 1/2 y^T alpha:
 *        dNLL/dh = 1/2 sum_jk B_jk dK_jk/dh,   dNLL/dsigma = sigma tr(B),
 *      h the values exactly as given in h_hyp; the log-space gradient dNLL/dlog h is h times these.  With d = |f_j - f_k|, s = d^2:
 *        gaussian {gamma}: -s K;   matern (nu = 1.5) {length_scale}: k^2 e^{-k} / l, k = sqrt(3) d / l;
 *        expsinesquared {length_scale, periodicity}: (4 sin^2(pi d / p) / l^3) K ; (2 pi d / (l^2 p^2)) sin(2 pi d / p) K;
 *        rationalquadratic {length_scale, alpha}: 2 alpha u K / (l (1 + u)) ; K (u / (1 + u) - log1p(u)), u = s / (2 alpha l^2);
 *        dotproduct {sigma_0}: 2 sigma_0 (every entry, diagonal included).
 *      dqgp_grad_outer_hyperparameters: d_grad gets one entry per h_hyp value (1, 1, 2, 2, 1 by outer id), d_F (n, m) the
 *      features the Gram was built from, m <= 36.  Only A^-1[j][k] with j >= k is read (want_inverse = 1 or 2, or the LU rung);
 *      duplicates and the diagonal follow the Gram's s = 0 rules; NaN features give NaN (stationary kernels).
 *      d_work: dqgp_grad_outer_hyperparameters_workspace_bytes(n).  dqgp_grad_noise_std writes d_out[0] = sigma tr(B) for either
 *      kernel type.  Both only enqueue (no synchronisation, graph-capturable) and are deterministic: a second call gives the same bits. */
size_t dqgp_grad_outer_hyperparameters_workspace_bytes(int n);
int dqgp_grad_outer_hyperparameters(int outer, const double* h_hyp, const double* d_Ainv, int ld, const double* d_alpha,
                                    const double* d_F, int n, int m, double* d_grad, void* d_work, void* stream);
int dqgp_grad_noise_std(const double* d_Ainv, int ld, const double* d_alpha, int n, double noise_std, double* d_out, void* stream);

/* ---- NLL terms (agent_riemannian.py:441-452): d_out[4] = {1/2 logdet, 1/2 y^T alpha, n/2 log 2pi, total} */
int dqgp_nll_terms(const double* d_logdet, const double* d_y, const double* d_alpha, int n, double* d_out, void* stream);

/* ---- local ADMM update (agent_riemannian.py:438,479-486; riemannian_optimizer.py:324-368):
 *      g4 = round(grad,4); theta = (z - (g4+psi)/(rho+L)) mod period; psi' = psi + rho*((theta - z) mod period);
 *      outputs rounded to 4 decimals (psi' from the UNROUNDED theta).  z must already be wrapped. */
int dqgp_admm_local(const double* d_z, const double* d_grad, const double* d_psi, int P, double rho, double lipschitz,
                    double period, double* d_theta_out, double* d_psi_out, void* stream);
/* ---- consensus (riemannian_optimizer.py:302-322 -> :26-51; rounding main.py:2523):
 *      z = round(circular_mean(theta + psi/rho), 4) over A agents, summed in agent order. */
int dqgp_admm_consensus(const double* d_theta, const double* d_psi, int A, int P, double rho, double period,
                        double* d_z_out, void* stream);
/*      same, with agent a's rows at d_theta + a*row_stride and d_psi + a*row_stride (row_stride >= P doubles): the
 *      engine keeps theta_a and psi_a side by side in ONE (A, 2, P) buffer so that a single all-gather moves both
 *      (the only cross-agent exchange of the path, main.py:2550-2555). */
int dqgp_admm_consensus_strided(const double* d_theta, const double* d_psi, int A, int P, int row_stride, double rho,
                                double period, double* d_z_out, void* stream);

/* ---- GP prediction pieces (main.py:1458-1466, 1546-1552): mean = Kst alpha; var = max(diag - q, 1e-10);
 *      d_nlpd[0] = mean_i(0.5 log 2pi + 0.5 log var_i + 0.5 (y_i-mean_i)^2/var_i). */
/* mean only: d_mean[i] = sum_k Kst[i][k] alpha[k] (use before dqgp_solver_quadform_rows_inplace overwrites Kst; then call
 * dqgp_predict_finish with d_Kst = NULL, which keeps d_mean as given). */
int dqgp_predict_mean(const double* d_Kst, int nt, int n, int ldk, const double* d_alpha, double* d_mean, void* stream);
int dqgp_predict_finish(const double* d_Kst, int nt, int n, int ldk, const double* d_alpha, const double* d_kss_diag,
                        const double* d_quad, const double* d_ytest, double* d_mean, double* d_var, double* d_nlpd,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DQGP_H */
