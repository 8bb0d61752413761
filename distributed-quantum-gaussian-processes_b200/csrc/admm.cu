// O(P) kernels of the ADMM trajectory: shifted parameter sets, local update, consensus, NLL terms and the
// prediction epilogue.  They keep the whole iteration on the device (no host round trip between the
// Cholesky and the update) and reproduce NumPy's rounding: np.round(x,4) = rint(x*1e4)/1e4,
// np.mod(x,p) = fmod with the sign of p — evaluated with explicitly un-fused multiplies/adds so the
// 4-decimal grid points are the reference's (Q5).
#include "common.cuh"

namespace dqgp {

__device__ __forceinline__ double np_mod(double x, double p) {
    double r = fmod(x, p);
    if (r != 0.0) { if ((p < 0.0) != (r < 0.0)) r = __dadd_rn(r, p); }
    else r = copysign(0.0, p);
    return r;
}
__device__ __forceinline__ double np_round4(double x) { return __ddiv_rn(rint(__dmul_rn(x, 1e4)), 1e4); }

// agent_riemannian.py:219 (wrap p), :245-256 (p +- h e_i), worker wrap :41
__global__ void shift_sets_kernel(const double* __restrict__ z, int P, double h, double period, double* __restrict__ Pm) {
    const int s = blockIdx.x;   // 0 .. 2P
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
        double v = np_mod(z[k], period);
        if (s > 0) {
            const int i = (s - 1) >> 1;
            if (k == i) v = ((s - 1) & 1) ? __dsub_rn(v, h) : __dadd_rn(v, h);
        }
        Pm[(size_t)s * P + k] = np_mod(v, period);
    }
}

// agent_riemannian.py:438,479-486 with riemannian_optimizer.py:343-346,363-366
__global__ void admm_local_kernel(const double* __restrict__ z, const double* __restrict__ grad, const double* __restrict__ psi,
                                  int P, double rho, double lip, double period, double* __restrict__ theta_out,
                                  double* __restrict__ psi_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P) return;
    const double g4 = np_round4(grad[k]);
    const double step = __ddiv_rn(-__dadd_rn(g4, psi[k]), __dadd_rn(rho, lip));
    const double theta = np_mod(__dadd_rn(z[k], step), period);
    const double lg = np_mod(__dsub_rn(theta, z[k]), period);
    const double psi_new = __dadd_rn(psi[k], __dmul_rn(rho, lg));
    theta_out[k] = np_round4(theta);
    psi_out[k] = np_round4(psi_new);
}

// riemannian_optimizer.py:317-320 -> :42-49, rounding main.py:2523; agents summed in index order
__global__ void admm_consensus_kernel(const double* __restrict__ theta, const double* __restrict__ psi, int A, int P, int ld, double rho,
                                      double period, double* __restrict__ z_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P) return;
    const double two_pi = 6.283185307179586;
    double cs = 0.0, sn = 0.0;
    for (int a = 0; a < A; ++a) {
        const double xi = __dadd_rn(theta[(size_t)a * ld + k], __ddiv_rn(psi[(size_t)a * ld + k], rho));
        const double ang = __ddiv_rn(__dmul_rn(two_pi, xi), period);
        cs = __dadd_rn(cs, cos(ang));
        sn = __dadd_rn(sn, sin(ang));
    }
    const double mean = __ddiv_rn(__dmul_rn(atan2(sn, cs), period), two_pi);
    z_out[k] = np_round4(np_mod(mean, period));
}

// agent_riemannian.py:447-452
__global__ void nll_terms_kernel(const double* __restrict__ logdet, const double* __restrict__ y, const double* __restrict__ alpha,
                                 int n, double* __restrict__ out) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) acc = fma(y[i], alpha[i], acc);
    const double ya = block_sum_256(acc);
    if (threadIdx.x == 0) {
        const double ld = 0.5 * logdet[0], q = 0.5 * ya, c = 0.5 * n * log(6.283185307179586);
        out[0] = ld; out[1] = q; out[2] = c; out[3] = ld + q + c;
    }
}

// main.py:1458 (mean), :1463-1466 (variance clamp), :1546-1552 (NLPD)
__global__ void predict_finish_kernel(const double* __restrict__ Kst, int nt, int n, int ldk, const double* __restrict__ alpha,
                                      const double* __restrict__ kss, const double* __restrict__ quad,
                                      const double* __restrict__ ytest, double* __restrict__ mean, double* __restrict__ var,
                                      double* __restrict__ nlpd_terms) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= nt) return;
    double acc = 0.0;
    if (Kst != nullptr) {
        for (int k = lane; k < n; k += 32) acc = fma(Kst[(size_t)row * ldk + k], alpha[k], acc);
        acc = warp_sum(acc);
    } else {
        acc = mean[row];                  // precomputed by dqgp_predict_mean
    }
    if (lane == 0) {
        if (kss == nullptr) { mean[row] = acc; return; }     // mean-only launch
        const double t = kss[row] - quad[row];
        const double v = (t != t) ? t : fmax(t, 1e-10);     // np.maximum (main.py:1466) propagates NaN; CUDA's fmax would drop it
        mean[row] = acc;
        var[row] = v;
        if (nlpd_terms) {
            const double r = ytest[row] - acc;
            nlpd_terms[row] = 0.5 * log(6.283185307179586) + 0.5 * log(v) + 0.5 * (r * r / v);
        }
    }
}
__global__ void mean_kernel(const double* __restrict__ v, int n, double* __restrict__ out) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) acc += v[i];
    const double sum = block_sum_256(acc);
    if (threadIdx.x == 0) out[0] = sum / n;
}

}  // namespace dqgp

extern "C" {

int dqgp_shift_parameter_sets(const double* d_z, int P, double h, double period, double* d_Pm, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_z && d_Pm && P >= 1 && period > 0, "dqgp_shift_parameter_sets: bad arguments");
    shift_sets_kernel<<<2 * P + 1, 128, 0, as_stream(stream)>>>(d_z, P, h, period, d_Pm);
    DQGP_LAUNCH_CHECK("shift_sets_kernel");
    return 0;
}

int dqgp_admm_local(const double* d_z, const double* d_grad, const double* d_psi, int P, double rho, double lipschitz,
                    double period, double* d_theta_out, double* d_psi_out, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_z && d_grad && d_psi && d_theta_out && d_psi_out && P >= 1, "dqgp_admm_local: bad arguments");
    admm_local_kernel<<<(P + 127) / 128, 128, 0, as_stream(stream)>>>(d_z, d_grad, d_psi, P, rho, lipschitz, period, d_theta_out, d_psi_out);
    DQGP_LAUNCH_CHECK("admm_local_kernel");
    return 0;
}

int dqgp_admm_consensus(const double* d_theta, const double* d_psi, int A, int P, double rho, double period, double* d_z_out,
                        void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_theta && d_psi && d_z_out && A >= 1 && P >= 1 && rho != 0.0, "dqgp_admm_consensus: bad arguments");
    admm_consensus_kernel<<<(P + 127) / 128, 128, 0, as_stream(stream)>>>(d_theta, d_psi, A, P, P, rho, period, d_z_out);
    DQGP_LAUNCH_CHECK("admm_consensus_kernel");
    return 0;
}

int dqgp_admm_consensus_strided(const double* d_theta, const double* d_psi, int A, int P, int row_stride, double rho, double period,
                                double* d_z_out, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_theta && d_psi && d_z_out && A >= 1 && P >= 1 && row_stride >= P && rho != 0.0, "dqgp_admm_consensus_strided: bad arguments");
    admm_consensus_kernel<<<(P + 127) / 128, 128, 0, as_stream(stream)>>>(d_theta, d_psi, A, P, row_stride, rho, period, d_z_out);
    DQGP_LAUNCH_CHECK("admm_consensus_kernel");
    return 0;
}

int dqgp_nll_terms(const double* d_logdet, const double* d_y, const double* d_alpha, int n, double* d_out, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_logdet && d_y && d_alpha && d_out && n >= 1, "dqgp_nll_terms: bad arguments");
    nll_terms_kernel<<<1, 256, 0, as_stream(stream)>>>(d_logdet, d_y, d_alpha, n, d_out);
    DQGP_LAUNCH_CHECK("nll_terms_kernel");
    return 0;
}

int dqgp_predict_mean(const double* d_Kst, int nt, int n, int ldk, const double* d_alpha, double* d_mean, void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_Kst && d_alpha && d_mean && nt >= 1 && n >= 1 && ldk >= n, "dqgp_predict_mean: bad arguments");
    predict_finish_kernel<<<(nt + 7) / 8, 256, 0, as_stream(stream)>>>(d_Kst, nt, n, ldk, d_alpha, nullptr, nullptr, nullptr, d_mean, nullptr, nullptr);
    DQGP_LAUNCH_CHECK("predict_mean kernel");
    return 0;
}

int dqgp_predict_finish(const double* d_Kst, int nt, int n, int ldk, const double* d_alpha, const double* d_kss_diag,
                        const double* d_quad, const double* d_ytest, double* d_mean, double* d_var, double* d_nlpd,
                        void* stream) {
    using namespace dqgp;
    DQGP_REQUIRE(d_alpha && d_kss_diag && d_quad && d_mean && d_var && nt >= 1 && n >= 1 && (d_Kst == nullptr || ldk >= n), "dqgp_predict_finish: bad arguments");
    DQGP_REQUIRE((d_nlpd == nullptr) == (d_ytest == nullptr), "dqgp_predict_finish: d_ytest and d_nlpd go together");
    cudaStream_t st = as_stream(stream);
    double* terms = d_nlpd ? d_nlpd + 1 : nullptr;   // d_nlpd: [mean NLPD, per-point terms ...] (1 + nt doubles)
    predict_finish_kernel<<<(nt + 7) / 8, 256, 0, st>>>(d_Kst, nt, n, ldk, d_alpha, d_kss_diag, d_quad, d_ytest, d_mean, d_var, terms);
    if (d_nlpd) mean_kernel<<<1, 256, 0, st>>>(terms, nt, d_nlpd);
    DQGP_LAUNCH_CHECK("predict_finish kernels");
    return 0;
}
}
