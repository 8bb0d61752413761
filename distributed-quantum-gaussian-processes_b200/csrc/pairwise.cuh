// Pairwise tile machinery shared by the Gram kernels (gram.cu) and the fused gradient kernels (grad.cu).
//
// A CTA of 256 threads owns a 64x64 tile of (row sample j, column sample k) pairs; its 8 warps (4x2) each own a
// 16x32 sub-tile as 2x4 DMMA 8x8 blocks.  Sample rows live in shared memory [sample][feature] with pitch G2_PITCH.
#pragma once
#include "common.cuh"
#include "fastmath.cuh"

namespace dqgp {

constexpr int PW_TILE = 64;
constexpr int PW_THREADS = 256;
constexpr int PW_MAX_M = 3 * MAX_QUBITS;

struct OuterHyp {
    double a;   // gaussian: gamma        | matern: 1/length_scale | expsine2: 1/length_scale   | ratquad: 1/(2 alpha l^2) | dot: sigma_0^2
    double b;   //                                                  | expsine2: pi/periodicity   | ratquad: alpha
};

// the dot product is the one outer kernel that is not a function of f - g: no snap to zero, no diagonal override, B keeps its diagonal
__host__ __device__ constexpr bool outer_is_stationary(int outer) { return outer != DQGP_OUTER_DOTPRODUCT; }

static inline int make_outer_hyp(int outer, const double* h_hyp, OuterHyp* out) {
    const double pi = 3.14159265358979323846;
    switch (outer) {
        case DQGP_OUTER_GAUSSIAN:
            out->a = h_hyp ? h_hyp[0] : 1.0; out->b = 0.0;
            DQGP_REQUIRE(out->a > 0, "gaussian outer kernel: gamma must be > 0");
            return 0;
        case DQGP_OUTER_MATERN15: {
            const double l = h_hyp ? h_hyp[0] : 1.0;
            DQGP_REQUIRE(l > 0, "matern outer kernel: length_scale must be > 0");
            out->a = 1.0 / l; out->b = 0.0;
            return 0;
        }
        case DQGP_OUTER_EXPSINE2: {
            const double l = h_hyp ? h_hyp[0] : 1.0, per = h_hyp ? h_hyp[1] : 1.0;
            DQGP_REQUIRE(l > 0 && per > 0, "expsinesquared outer kernel: length_scale and periodicity must be > 0");
            out->a = 1.0 / l; out->b = pi / per;
            return 0;
        }
        case DQGP_OUTER_RATQUAD: {
            const double l = h_hyp ? h_hyp[0] : 1.0, alpha = h_hyp ? h_hyp[1] : 1.0;
            DQGP_REQUIRE(l > 0 && alpha > 0, "rationalquadratic outer kernel: length_scale and alpha must be > 0");
            out->a = 1.0 / (2.0 * alpha * l * l); out->b = alpha;
            return 0;
        }
        case DQGP_OUTER_DOTPRODUCT: {
            const double s0 = h_hyp ? h_hyp[0] : 1.0;
            DQGP_REQUIRE(s0 >= 0, "dotproduct outer kernel: sigma_0 must be >= 0");
            out->a = s0 * s0; out->b = 0.0;
            return 0;
        }
    }
    set_error("unknown outer kernel id %d (hot path covers gaussian, matern, expsinesquared, rationalquadratic, dotproduct)", outer);
    return -1;
}

// 1/x from the MUFU.RCP64H seed and one cubic Newton step y (1 + e + e^2), e = 1 - x y: 3 DFMA, no range branch.  Meant for
// x >= 1 (the rational quadratic's base): the seed's ~20 bits become ~60 before rounding, and x = 1 gives exactly 1.
__device__ __forceinline__ double fast_rcp_ge1(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x, y, 1.0);
    return fma(y, fma(e, e, e), y);
}

// RationalQuadratic (1 + d^2 / (2 alpha l^2))^-alpha from v = -d^2: a reciprocal at alpha = 1 (the only value the reference
// reaches, Q2), exp(-alpha log(base)) otherwise (uniform branch on a kernel argument)
__device__ __forceinline__ double ratquad_from_neg_d2(double v, const OuterHyp& h) {
    const double base = fma(-v, h.a, 1.0);
    return h.b == 1.0 ? fast_rcp_ge1(base) : exp(-h.b * log(base));
}

// Outer kernel from v = -gamma_eff * d^2 (gamma_eff = gamma for the Gaussian, 1 otherwise), as left in a DMMA
// accumulator by the Gram identity, with scikit-learn's formulas (sklearn/gaussian_process/kernels.py RBF /
// Matern(nu=1.5) / ExpSineSquared / RationalQuadratic, as used by squlearn's ProjectedQuantumKernel; reference main.py:130-137).
// The dot product's accumulator already holds sigma_0^2 + f.g, which passes through.
// Warp-collective: fast_exp_tab shuffles its table.
template <int OUTER>
__device__ __forceinline__ double outer_from_neg_gd2(double v, const OuterHyp& h, double tab) {
    // v = -gamma_eff * d^2 (gamma_eff = gamma for the Gaussian, 1 otherwise); warp-collective (table shuffle)
    if (OUTER == DQGP_OUTER_GAUSSIAN) {
        return fast_exp_tab(fmax(v, -700.0), tab);
    } else if (OUTER == DQGP_OUTER_MATERN15) {
        const double k = sqrt(fmax(-v, 0.0)) * h.a * 1.7320508075688772;
        return (1.0 + k) * fast_exp_tab(fmax(-k, -700.0), tab);
    } else if (OUTER == DQGP_OUTER_RATQUAD) {
        return ratquad_from_neg_d2(v, h);
    } else if (OUTER == DQGP_OUTER_DOTPRODUCT) {
        return v;
    } else {
        const double sn = sin(sqrt(fmax(-v, 0.0)) * h.b) * h.a;
        return fast_exp_tab(fmax(-2.0 * (sn * sn), -700.0), tab);
    }
}

// sqrt for the fused gradient's Matern / ExpSineSquared path: MUFU.RSQ64H seed (20 bits), one Newton step on y ~ 1/sqrt(x),
// one residual correction on s = x y: 8 FP64-pipe instructions, <= 1 ulp on normal x > 0, no range branch (libm's sqrt
// carries a slow-path call and measured 16 DFMA-equivalents in this loop, profiles/r01_fp64_peak.json).  The guard that keeps
// x away from zero / tiny negative rounding residue of the Gram identity is an INTEGER compare on the high word (ALU pipe,
// not the FP64 pipe that bounds the kernel); NaN passes through (np.sqrt(nan) = nan, as in the reference).
__device__ __forceinline__ double fast_sqrt_guarded(double x) {
    if (__double2hiint(x) < 0x01a56e1f) x = 1e-300;            // x < ~1e-300, zero, or negative -> sqrt ~ 1e-150 (= 0 for every use here)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double r = x * y;
    const double e = fma(-r, y, 1.0);
    y = fma(0.5 * y, e, y);
    double s = x * y;
    const double e2 = fma(-s, s, x);
    return fma(e2, 0.5 * y, s);
}

// The fused gradient's outer kernel from v = -gamma_eff d^2: same formulas as outer_from_neg_gd2, built for the FP64 pipe that
// bounds grad_projected_dmma_kernel: branch-free sqrt (above), degree-5 table exp (10 instructions), (1 + k) e^-k as one FMA,
// and no exponent clamp when the host has shown the argument cannot go below -700 (CLAMP = false; features lie in [-1, 1]).
// RationalQuadratic and DotProduct have no exponent (CLAMP is always false for them).
template <int OUTER, bool CLAMP>
__device__ __forceinline__ double outer_grad_from_neg_gd2(double v, const OuterHyp& h, double tab) {
    if (OUTER == DQGP_OUTER_GAUSSIAN) {
        // v arrives in units of ln2/32 (the kernel folds 32/ln2 into the DMMA operands): exact two-add range reduction
        return fast_exp_tab5_scaled(CLAMP ? fmax(v, -700.0 * DQGP_EXP_S32) : v, tab);
    } else if (OUTER == DQGP_OUTER_MATERN15) {
        const double nk = fast_sqrt_guarded(-v) * (-1.7320508075688772 * h.a);      // -sqrt(3) d / l
        const double e = fast_exp_tab5(CLAMP ? fmax(nk, -700.0) : nk, tab);
        return fma(-nk, e, e);
    } else if (OUTER == DQGP_OUTER_RATQUAD) {
        return ratquad_from_neg_d2(v, h);
    } else if (OUTER == DQGP_OUTER_DOTPRODUCT) {
        return v;
    } else {
        const double sn = sin(fast_sqrt_guarded(-v) * h.b) * h.a;
        const double x = -2.0 * (sn * sn);
        return fast_exp_tab5(CLAMP ? fmax(x, -700.0) : x, tab);
    }
}

// The analytic gradient's per-pair weight (grad_analytic_rows_kernel) from s = |f_j - f_k|^2, for a stationary outer kernel
// K = kappa(s): kappa'(s), with d = sqrt(s), a and b as in OuterHyp.  The Gaussian returns e^{-gamma s} and leaves -gamma to the
// contraction's scale.
//   Matern 1.5:        -(3/2) a^2 e^{-sqrt(3) a d}
//   ExpSineSquared:    -a^2 b (sin(2 b d) / d) kappa, kappa = e^{-2 a^2 sin^2(b d)}
//   RationalQuadratic: -alpha a base^{-alpha-1}, base = 1 + a s (alpha = 1: -a / base^2)
// A duplicate sample (s = 0) gets a finite weight: fast_sqrt_guarded never returns 0, and sin(b d) / d is then b exactly.  Matern,
// ExpSineSquared and RationalQuadratic clamp their exponents at -700 (a tiny length scale reaches it); the Gaussian's -gamma s is
// not clamped and stays inside fast_exp's range while gamma 4m < 708.  NaN features reach the gradient through f_j - f_k whatever
// the weight.  Not warp-collective: rows past n leave the column loop, so the table exp cannot be used.
// ALPHA1 (RationalQuadratic only): alpha = 1, chosen by the host per launch, so the pair loop carries no branch on alpha.
template <int OUTER, bool ALPHA1>
__device__ __forceinline__ double outer_analytic_weight(double s, const OuterHyp& h) {
    if (OUTER == DQGP_OUTER_GAUSSIAN) {
        return fast_exp(-h.a * s);
    } else if (OUTER == DQGP_OUTER_MATERN15) {
        const double nk = fast_sqrt_guarded(s) * (-1.7320508075688772 * h.a);      // -sqrt(3) d / l
        return (-1.5 * h.a * h.a) * fast_exp(fmax(nk, -700.0));
    } else if (OUTER == DQGP_OUTER_RATQUAD) {
        const double base = fma(s, h.a, 1.0);
        if (ALPHA1) {
            const double r = fast_rcp_ge1(base);
            return -h.a * (r * r);
        }
        return (-h.b * h.a) * fast_exp(fmax(-(h.b + 1.0) * log(base), -700.0));
    } else {
        const double d = fast_sqrt_guarded(s);
        double sn, cs;
        sincos(h.b * d, &sn, &cs);
        const double k = fast_exp(fmax(-2.0 * (h.a * h.a) * (sn * sn), -700.0));
        return (-2.0 * h.a * h.a * h.b) * (sn * cs / d) * k;
    }
}

// The hyper-parameter gradient's per-pair terms (grad_hyper_dmma_kernel) from s = |f_j - f_k|^2 >= 0: dK/dh_0 and dK/dh_1 up to
// per-kernel constants c_0, c_1 that the host folds into the tile sums (outer_hyper_scales), with d = sqrt(s), a and b as in OuterHyp.
//   Gaussian {gamma}:                        w0 = -s K                               c0 = 1
//   Matern 1.5 {l}, k = sqrt(3) a d:         w0 = k^2 e^{-k}                         c0 = a = 1/l
//   ExpSineSquared {l, p}, z = b d:          w0 = sin^2 z K,  w1 = d sin z cos z K   c0 = 4 a^3,  c1 = 4 a^2 b^2 / pi
//   RationalQuadratic {l, alpha}, u = a s:   w0 = u/(1+u) K,  w1 = (u/(1+u) - log1p u) K   c0 = 2 alpha / l,  c1 = 1
//   DotProduct {sigma_0}:                    w0 = 1                                  c0 = 2 sigma_0
// Every stationary term is exactly 0 at s = 0 (libm sqrt, no guard).  Exponents are clamped at -700.  Not warp-collective.
template <int OUTER>
__device__ __forceinline__ void outer_hyper_terms(double s, const OuterHyp& h, double& w0, double& w1) {
    w1 = 0.0;
    if (OUTER == DQGP_OUTER_GAUSSIAN) {
        w0 = -s * fast_exp(fmax(-h.a * s, -700.0));
    } else if (OUTER == DQGP_OUTER_MATERN15) {
        const double k = sqrt(s) * h.a * 1.7320508075688772;
        w0 = (k * k) * fast_exp(fmax(-k, -700.0));
    } else if (OUTER == DQGP_OUTER_EXPSINE2) {
        const double d = sqrt(s);
        double sn, cs;
        sincos(h.b * d, &sn, &cs);
        const double K = fast_exp(fmax(-2.0 * (h.a * h.a) * (sn * sn), -700.0));
        w0 = (sn * sn) * K;
        w1 = (d * sn * cs) * K;
    } else if (OUTER == DQGP_OUTER_RATQUAD) {
        const double u = s * h.a, lp = log1p(u), r = u / (1.0 + u);
        const double K = fast_exp(fmax(-h.b * lp, -700.0));
        w0 = r * K;
        w1 = (r - lp) * K;
    } else {
        w0 = 1.0;
    }
}

// out[row] = add (+ |F[row]|^2 when with_norm), rows of m features (gram.cu)
void launch_self_kernel(const double* F, long long rows, int m, double add, bool with_norm, double* out, cudaStream_t st);

// DMMA fidelity kernels (fid.cu)
int fidelity_gram_dmma(const double* Psi1, int n1, const double* Psi2, int n2, int dim, double* K, int ldk, cudaStream_t st);
int fidelity_grad_dmma(const double* Ainv, int ld, const double* alpha, const double* Psi, int n, int dim, int P, double* partial,
                       int tiles, cudaStream_t st);
// W = [B o Re S | B o Im S] (n_pad x 2 n_pad, every entry written), S_jk = <psi_k|psi_j>, B = A^-1 - alpha alpha^T
int fidelity_weights_dmma(const double* Ainv, int ld, const double* alpha, const double* Psi, int n, int dim, double* W, int n_pad,
                          cudaStream_t st);

constexpr int G2_PITCH = 36;   // doubles per staged sample row: = 4 (mod 16) -> conflict-free DMMA fragment loads

}  // namespace dqgp
