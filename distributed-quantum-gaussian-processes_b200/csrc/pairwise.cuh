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
    double a;   // gaussian: gamma        | matern: 1/length_scale | expsine2: 1/length_scale
    double b;   //                                                  | expsine2: pi/periodicity
};

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
    }
    set_error("unknown outer kernel id %d (hot path covers gaussian, matern, expsinesquared)", outer);
    return -1;
}

// Outer kernel from v = -gamma_eff * d^2 (gamma_eff = gamma for the Gaussian, 1 otherwise), as left in a DMMA
// accumulator by the Gram identity, with scikit-learn's formulas (sklearn/gaussian_process/kernels.py RBF /
// Matern(nu=1.5) / ExpSineSquared, as used by squlearn's ProjectedQuantumKernel; reference main.py:130-137).
// Warp-collective: fast_exp_tab shuffles its table.
template <int OUTER>
__device__ __forceinline__ double outer_from_neg_gd2(double v, const OuterHyp& h, double tab) {
    // v = -gamma_eff * d^2 (gamma_eff = gamma for the Gaussian, 1 otherwise); warp-collective (table shuffle)
    if (OUTER == DQGP_OUTER_GAUSSIAN) {
        return fast_exp_tab(fmax(v, -700.0), tab);
    } else if (OUTER == DQGP_OUTER_MATERN15) {
        const double k = sqrt(fmax(-v, 0.0)) * h.a * 1.7320508075688772;
        return (1.0 + k) * fast_exp_tab(fmax(-k, -700.0), tab);
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
template <int OUTER, bool CLAMP>
__device__ __forceinline__ double outer_grad_from_neg_gd2(double v, const OuterHyp& h, double tab) {
    if (OUTER == DQGP_OUTER_GAUSSIAN) {
        // v arrives in units of ln2/32 (the kernel folds 32/ln2 into the DMMA operands): exact two-add range reduction
        return fast_exp_tab5_scaled(CLAMP ? fmax(v, -700.0 * DQGP_EXP_S32) : v, tab);
    } else if (OUTER == DQGP_OUTER_MATERN15) {
        const double nk = fast_sqrt_guarded(-v) * (-1.7320508075688772 * h.a);      // -sqrt(3) d / l
        const double e = fast_exp_tab5(CLAMP ? fmax(nk, -700.0) : nk, tab);
        return fma(-nk, e, e);
    } else {
        const double sn = sin(fast_sqrt_guarded(-v) * h.b) * h.a;
        const double x = -2.0 * (sn * sn);
        return fast_exp_tab5(CLAMP ? fmax(x, -700.0) : x, tab);
    }
}

// DMMA fidelity kernels (fid.cu)
int fidelity_gram_dmma(const double* Psi1, int n1, const double* Psi2, int n2, int dim, double* K, int ldk, cudaStream_t st);
int fidelity_grad_dmma(const double* Ainv, int ld, const double* alpha, const double* Psi, int n, int dim, int P, double* partial,
                       int tiles, cudaStream_t st);

constexpr int G2_PITCH = 36;   // doubles per staged sample row: = 4 (mod 16) -> conflict-free DMMA fragment loads

}  // namespace dqgp
