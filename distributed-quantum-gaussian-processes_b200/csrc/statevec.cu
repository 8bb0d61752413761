// Batched statevector simulation of the encoding circuits + Pauli-XYZ features (sm_100a).
//
// Replaces what squlearn does behind q_kernel.evaluate for every sample and parameter set
// (reference call site agent_riemannian.py:118; S = 2P+1 sets built at :245-256).
//
// Mapping: one warp owns one state (2^q complex128 amplitudes in shared memory, never in HBM); for q <= 7 a
// warp is split into lane groups, one state per group, so no lane idles.  The gate list is executed as
// REGISTER-BLOCKED PASSES (plan built on the host, circuit.cu): a pass names <= 3 block qubits; a lane loads the
// 2^3 amplitudes of one block into registers, applies every gate of the pass whose target is a block qubit
// (runs of rotations / H on one qubit fused into a general 2x2 unitary composed per state; CX / CRZ with the
// control read from the index or from the block) and stores them back — one
// shared-memory round trip for ~15 gates instead of one per gate (v1: 59 round trips for config 4, 16.6 ms;
// ncu profiles/r01_v1_statevec: LSU-wavefront bound, 27% bank conflicts).  All sin/cos of a state's gate
// angles are computed once, cooperatively, into a per-state table; arccos(x) once per sample.  Only
// __syncwarp separates passes.  The epilogue reduces <X_k>,<Y_k>,<Z_k> three qubits at a time from registers
// with group-local shuffles, or streams the state to HBM for the fidelity kernel.
#include <cstdlib>
#include "common.cuh"

namespace dqgp {

__device__ __forceinline__ int insert_zero_bit(int k, int t) {
    const int lo = k & ((1 << t) - 1);
    return ((k >> t) << (t + 1)) | lo;
}

// Shared-memory placement of amplitude i: XOR the low three index bits with bits 3..5.  A lane's register block
// is 8 amplitudes; when the block qubits are {0,1,2} consecutive lanes would otherwise sit 128 bytes apart and
// every LDS.128 of a quarter-warp would hit the same four banks (32-way conflict, measured: v2 without the
// swizzle was still 12.9 ms).  With it those accesses, and the {3,4,5} blocks, are conflict-free.
__device__ __forceinline__ int sv_phys(int i) { return i ^ ((i >> 3) & 7); }

template <int Q>
struct SvGeom {
    static constexpr int DIM = 1 << Q;
    static constexpr int BMAX = Q < 3 ? Q : 3;
    static constexpr int GROUPS = DIM >> BMAX;                    // register blocks per state (full-size pass)
    static constexpr int LPS = GROUPS >= 32 ? 32 : GROUPS;        // lanes per state
    static constexpr int SPW = 32 / LPS;                          // states per warp
};

// ---- ops on the register block, target = local bit L (compile time) ------------------------------------------
// general 2x2 complex unitary u = {u00,u01,u10,u11} on every pair along bit L: 16 FP64 instructions per pair
template <int N, int L>
__device__ __forceinline__ void apply_u2(double2 (&r)[N], const double2 u00, const double2 u01, const double2 u10, const double2 u11) {
    constexpr int BIT = 1 << L;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        if (j & BIT) continue;
        const double2 a = r[j], b = r[j | BIT];
        double2 na, nb;
        na.x = fma(u01.x, b.x, fma(-u01.y, b.y, fma(u00.x, a.x, -u00.y * a.y)));
        na.y = fma(u01.x, b.y, fma(u01.y, b.x, fma(u00.x, a.y, u00.y * a.x)));
        nb.x = fma(u11.x, b.x, fma(-u11.y, b.y, fma(u10.x, a.x, -u10.y * a.y)));
        nb.y = fma(u11.x, b.y, fma(u11.y, b.x, fma(u10.x, a.y, u10.y * a.x)));
        r[j] = na;
        r[j | BIT] = nb;
    }
}
// CX (swap) / CRZ (phases e^{-+ i theta/2}) on the pairs whose control bit is set
template <int N, int L>
__device__ __forceinline__ void apply_controlled(double2 (&r)[N], int kind, int cloc, bool ext, double c, double s, bool zero_off = false) {
    constexpr int BIT = 1 << L;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        if (j & BIT) continue;
        const bool on = cloc >= 0 ? (((j >> cloc) & 1) != 0) : ext;
        const double2 a = r[j], b = r[j | BIT];
        double2 na, nb;
        if (kind == SV_CX) {
            na = b;
            nb = a;
        } else {
            na = make_double2(fma(c, a.x, s * a.y), fma(c, a.y, -s * a.x));
            nb = make_double2(fma(c, b.x, -s * b.y), fma(c, b.y, s * b.x));
        }
        const double2 zero = make_double2(0.0, 0.0);
        r[j] = on ? na : (zero_off ? zero : a);
        r[j | BIT] = on ? nb : (zero_off ? zero : b);
    }
}

// one shifted parameter: either a replacement for fused matrix `mat`, or replacement cos/sin for CRZ gate `gate`
struct SvAlt {
    int mat;            // fused-matrix index replaced by u[0..3], or -1
    int gate;           // CRZ gate index whose (cos, sin) is u[0], or -1
    const double2* u;
    int zero_off;       // that CRZ also ZEROES the amplitudes whose control bit is clear (derivative fork: dCRZ/dtheta = P1 x RZ(theta+pi)/2)
};

template <int N, int L>
__device__ __forceinline__ void apply_op(double2 (&r)[N], const SvOp op, int base, const double2* __restrict__ mats,
                                         const double2* __restrict__ trig, const SvAlt& alt) {
    if (op.kind == SV_U2) {
        const double2* u = (op.idx == alt.mat) ? alt.u : mats + 4 * op.idx;
        apply_u2<N, L>(r, u[0], u[1], u[2], u[3]);
    } else {
        const bool ext = (op.cq >= 0) ? (((base >> op.cq) & 1) != 0) : false;
        const bool is_alt = op.kind == SV_CRZ && op.idx == alt.gate;
        const double2 cs = (op.kind == SV_CRZ) ? (is_alt ? alt.u[0] : trig[op.idx]) : make_double2(1.0, 0.0);
        apply_controlled<N, L>(r, op.kind, op.cloc, ext, cs.x, cs.y, is_alt && alt.zero_off != 0);
    }
}

template <int B>
__device__ __forceinline__ void run_pass(double2* __restrict__ amp, const SvPass& ps, const SvOp* __restrict__ ops,
                                         const double2* __restrict__ mats, const double2* __restrict__ trig, int lig, int lps,
                                         int groups, const SvAlt alt = SvAlt{-1, -1, nullptr, 0}) {
    constexpr int N = 1 << B;
    const int q0 = ps.q[0], q1 = ps.q[1], q2 = ps.q[2];
    int off[N];
#pragma unroll
    for (int j = 0; j < N; ++j) off[j] = ((j & 1) ? (1 << q0) : 0) + ((B > 1 && (j & 2)) ? (1 << q1) : 0) + ((B > 2 && (j & 4)) ? (1 << q2) : 0);
    for (int gi = lig; gi < groups; gi += lps) {
        int base = insert_zero_bit(gi, q0);
        if (B > 1) base = insert_zero_bit(base, q1);
        if (B > 2) base = insert_zero_bit(base, q2);
        double2 r[N];
#pragma unroll
        for (int j = 0; j < N; ++j) r[j] = amp[sv_phys(base + off[j])];
#pragma unroll 1
        for (int o = ps.op_begin; o < ps.op_end; ++o) {
            const SvOp op = ops[o];
            if (op.lbit == 0) apply_op<N, 0>(r, op, base, mats, trig, alt);
            else if (B > 1 && op.lbit == 1) apply_op<N, (B > 1 ? 1 : 0)>(r, op, base, mats, trig, alt);
            else if (B > 2) apply_op<N, (B > 2 ? 2 : 0)>(r, op, base, mats, trig, alt);
        }
#pragma unroll
        for (int j = 0; j < N; ++j) amp[sv_phys(base + off[j])] = r[j];
    }
}

// matrix of one original gate from its (cos, sin) of the half angle
__device__ __forceinline__ void gate_matrix(int kind, double c, double s, double2 (&g)[4]) {
    const double r2 = 0.70710678118654752440;
    switch (kind) {
        case DQGP_G_H: g[0] = make_double2(r2, 0); g[1] = make_double2(r2, 0); g[2] = make_double2(r2, 0); g[3] = make_double2(-r2, 0); break;
        case DQGP_G_RX: g[0] = make_double2(c, 0); g[1] = make_double2(0, -s); g[2] = make_double2(0, -s); g[3] = make_double2(c, 0); break;
        case DQGP_G_RY: g[0] = make_double2(c, 0); g[1] = make_double2(-s, 0); g[2] = make_double2(s, 0); g[3] = make_double2(c, 0); break;
        default: g[0] = make_double2(c, -s); g[1] = make_double2(0, 0); g[2] = make_double2(0, 0); g[3] = make_double2(c, s); break;   // RZ
    }
}
__device__ __forceinline__ double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }

// <X>,<Y>,<Z> of qubits k0 .. k0+B-1 from register blocks; group-local shuffle reduction; lane 0 of the state writes
template <int B, int Q>
__device__ __forceinline__ void features_block(const double2* __restrict__ amp, int k0, int lig, int lps, bool live,
                                               double* __restrict__ dst, double* __restrict__ red = nullptr) {
    constexpr int N = 1 << B;
    const int groups = (1 << Q) >> B;
    double fx[B], fy[B], fz[B];
#pragma unroll
    for (int l = 0; l < B; ++l) fx[l] = fy[l] = fz[l] = 0.0;
    for (int gi = lig; gi < groups; gi += lps) {
        int base = gi;
#pragma unroll
        for (int l = 0; l < B; ++l) base = insert_zero_bit(base, k0 + l);
        double2 r[N];
#pragma unroll
        for (int j = 0; j < N; ++j) {
            int o = 0;
#pragma unroll
            for (int l = 0; l < B; ++l) o += ((j >> l) & 1) << (k0 + l);
            r[j] = amp[sv_phys(base + o)];
        }
#pragma unroll
        for (int l = 0; l < B; ++l)
#pragma unroll
            for (int j = 0; j < N; ++j) {
                if (j & (1 << l)) continue;
                const double2 a = r[j], b = r[j | (1 << l)];
                fx[l] += a.x * b.x + a.y * b.y;
                fy[l] += a.x * b.y - a.y * b.x;
                fz[l] += (a.x * a.x + a.y * a.y) - (b.x * b.x + b.y * b.y);
            }
    }
    if (lps <= 32) {
#pragma unroll
        for (int l = 0; l < B; ++l) {
            for (int o = lps >> 1; o > 0; o >>= 1) {
                fx[l] += __shfl_xor_sync(0xffffffffu, fx[l], o);
                fy[l] += __shfl_xor_sync(0xffffffffu, fy[l], o);
                fz[l] += __shfl_xor_sync(0xffffffffu, fz[l], o);
            }
            if (live && lig == 0) {
                dst[k0 + l] = 2.0 * fx[l];
                dst[Q + k0 + l] = 2.0 * fy[l];
                dst[2 * Q + k0 + l] = fz[l];
            }
        }
    } else {
        // team = whole block (several warps per state): warp shuffle, then a fixed-order sum over warps in shared memory
        const int warp = lig >> 5, nw = lps >> 5;
#pragma unroll
        for (int l = 0; l < B; ++l) {
            fx[l] = warp_sum(fx[l]); fy[l] = warp_sum(fy[l]); fz[l] = warp_sum(fz[l]);
            if ((lig & 31) == 0) { red[(warp * 3 + 0) * 3 + l] = fx[l]; red[(warp * 3 + 1) * 3 + l] = fy[l]; red[(warp * 3 + 2) * 3 + l] = fz[l]; }
        }
        __syncthreads();
        if (lig < 3 * B) {
            const int which = lig / B, l = lig - which * B;
            double t = 0.0;
            for (int w = 0; w < nw; ++w) t += red[(w * 3 + which) * 3 + l];
            if (live) dst[which * Q + k0 + l] = (which == 2) ? t : 2.0 * t;
        }
        __syncthreads();
    }
}

// Re<psi|O|phi> for O = X_k, Y_k, Z_k, k = k0 .. k0+B-1, of two states held side by side (same layout as features_block;
// psi = phi gives <X>, <Y>, <Z>).  Used by the linear-combination form of the central-difference sets (statevec_lc_kernel).
template <int B, int Q>
__device__ __forceinline__ void features_cross_block(const double2* __restrict__ amp1, const double2* __restrict__ amp2, int k0, int lig,
                                                     int lps, double* __restrict__ dst, double* __restrict__ red = nullptr) {
    constexpr int N = 1 << B;
    const int groups = (1 << Q) >> B;
    double fx[B], fy[B], fz[B];
#pragma unroll
    for (int l = 0; l < B; ++l) fx[l] = fy[l] = fz[l] = 0.0;
    for (int gi = lig; gi < groups; gi += lps) {
        int base = gi;
#pragma unroll
        for (int l = 0; l < B; ++l) base = insert_zero_bit(base, k0 + l);
        double2 r[N], s[N];
#pragma unroll
        for (int j = 0; j < N; ++j) {
            int o = 0;
#pragma unroll
            for (int l = 0; l < B; ++l) o += ((j >> l) & 1) << (k0 + l);
            r[j] = amp1[sv_phys(base + o)];
            s[j] = amp2[sv_phys(base + o)];
        }
#pragma unroll
        for (int l = 0; l < B; ++l)
#pragma unroll
            for (int j = 0; j < N; ++j) {
                if (j & (1 << l)) continue;
                const double2 a = r[j], b = r[j | (1 << l)], a2 = s[j], b2 = s[j | (1 << l)];
                fx[l] += (a.x * b2.x + a.y * b2.y) + (b.x * a2.x + b.y * a2.y);
                fy[l] += (a.x * b2.y - a.y * b2.x) - (b.x * a2.y - b.y * a2.x);
                fz[l] += (a.x * a2.x + a.y * a2.y) - (b.x * b2.x + b.y * b2.y);
            }
    }
    if (lps <= 32) {
#pragma unroll
        for (int l = 0; l < B; ++l) {
            for (int o = lps >> 1; o > 0; o >>= 1) {
                fx[l] += __shfl_xor_sync(0xffffffffu, fx[l], o);
                fy[l] += __shfl_xor_sync(0xffffffffu, fy[l], o);
                fz[l] += __shfl_xor_sync(0xffffffffu, fz[l], o);
            }
            if (lig == 0) {
                dst[k0 + l] = fx[l];
                dst[Q + k0 + l] = fy[l];
                dst[2 * Q + k0 + l] = fz[l];
            }
        }
    } else {
        const int warp = lig >> 5, nw = lps >> 5;
#pragma unroll
        for (int l = 0; l < B; ++l) {
            fx[l] = warp_sum(fx[l]); fy[l] = warp_sum(fy[l]); fz[l] = warp_sum(fz[l]);
            if ((lig & 31) == 0) { red[(warp * 3 + 0) * 3 + l] = fx[l]; red[(warp * 3 + 1) * 3 + l] = fy[l]; red[(warp * 3 + 2) * 3 + l] = fz[l]; }
        }
        __syncthreads();
        if (lig < 3 * B) {
            const int which = lig / B, l = lig - which * B;
            double t = 0.0;
            for (int w = 0; w < nw; ++w) t += red[(w * 3 + which) * 3 + l];
            dst[which * Q + k0 + l] = t;
        }
        __syncthreads();
    }
}

template <int Q, bool WANT_STATES>
__global__ void __launch_bounds__(128) statevec_kernel(const dqgp_gate* __restrict__ gates, int n_gates,
                                                        const SvPass* __restrict__ passes, int n_passes,
                                                        const SvOp* __restrict__ ops, const SvMat* __restrict__ mats,
                                                        int n_mats, const int* __restrict__ mat_gates, int n_mat_gates, int d, int P,
                                                        int uses_acos,
                                                        const double* __restrict__ X, int n, const double* __restrict__ Pm,
                                                        int S, double* __restrict__ out) {
    using G = SvGeom<Q>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // block layout: [gate program][passes][ops][mats][mat_gates][per warp: SPW x (DIM amp | n_gates trig | n_mats x 4 u2 | d acos)]
    const size_t gate_bytes = (sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15);
    const size_t pass_bytes = (sizeof(SvPass) * n_passes + 15) & ~size_t(15);
    const size_t op_bytes = (sizeof(SvOp) * n_gates + 15) & ~size_t(15);
    const size_t mat_bytes = (sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15);
    dqgp_gate* s_gates = reinterpret_cast<dqgp_gate*>(smem_raw);
    SvPass* s_passes = reinterpret_cast<SvPass*>(smem_raw + gate_bytes);
    SvOp* s_ops = reinterpret_cast<SvOp*>(smem_raw + gate_bytes + pass_bytes);
    SvMat* s_mats = reinterpret_cast<SvMat*>(smem_raw + gate_bytes + pass_bytes + op_bytes);
    int* s_mat_gates = reinterpret_cast<int*>(s_mats + n_mats);
    const int warps = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t state_bytes = sizeof(double2) * (G::DIM + n_gates + 4 * n_mats) + ((sizeof(double) * d + 15) & ~size_t(15));
    for (int i = threadIdx.x; i < n_gates; i += blockDim.x) { s_gates[i] = gates[i]; s_ops[i] = ops[i]; }   // #ops <= #gates
    for (int i = threadIdx.x; i < n_passes; i += blockDim.x) s_passes[i] = passes[i];
    for (int i = threadIdx.x; i < n_mats; i += blockDim.x) s_mats[i] = mats[i];
    for (int i = threadIdx.x; i < n_mat_gates; i += blockDim.x) s_mat_gates[i] = mat_gates[i];
    __syncthreads();

    const int sub = lane / G::LPS;   // which state of this warp
    const int lig = lane % G::LPS;   // lane in group
    unsigned char* my = smem_raw + gate_bytes + pass_bytes + op_bytes + mat_bytes + state_bytes * (size_t(warp) * G::SPW + sub);
    double2* amp = reinterpret_cast<double2*>(my);
    double2* trig = amp + G::DIM;
    double2* u2 = trig + n_gates;
    double* acx = reinterpret_cast<double*>(u2 + 4 * n_mats);

    const long long total = (long long)S * n;
    const long long n_groups = (total + G::SPW - 1) / G::SPW;
    const int m = 3 * Q;
    for (long long grp = (long long)blockIdx.x * warps + warp; grp < n_groups; grp += (long long)gridDim.x * warps) {
        long long st = grp * G::SPW + sub;
        const bool live = st < total;
        if (!live) st = total - 1;
        const int s = int(st / n), j = int(st % n);
        const double* x = X + (size_t)j * d;
        const double* p = Pm + (size_t)s * P;

        if (uses_acos) {
            for (int f = lig; f < d; f += G::LPS) acx[f] = acos(x[f]);
            __syncwarp();
        }
        for (int g = lig; g < n_gates; g += G::LPS) {
            const dqgp_gate gt = s_gates[g];
            if (gt.form == DQGP_A_NONE) continue;   // H, CX carry no angle
            double ang = 0.0;
            switch (gt.form) {
                case DQGP_A_P: ang = p[gt.pidx]; break;
                case DQGP_A_X: ang = x[gt.fidx]; break;
                case DQGP_A_P_PLUS_CX: ang = p[gt.pidx] + gt.coef * x[gt.fidx]; break;
                case DQGP_A_P_TIMES_ACOS: ang = p[gt.pidx] * acx[gt.fidx]; break;
                case DQGP_A_C_TIMES_ACOS: ang = gt.coef * acx[gt.fidx]; break;
                default: break;
            }
            double sn, cs;
            sincos(0.5 * ang, &sn, &cs);
            trig[g] = make_double2(cs, sn);
        }
        for (int i = lig; i < G::DIM; i += G::LPS) amp[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);   // sv_phys(0) == 0
        __syncwarp();
        // compose the fused 2x2 unitaries of this state: M = G_last ... G_first
        for (int f = lig; f < n_mats; f += G::LPS) {
            const SvMat mt = s_mats[f];
            double2 mm[4];
            {
                const int g0 = s_mat_gates[mt.g_begin];
                const double2 cs = trig[g0];
                gate_matrix(s_gates[g0].kind, cs.x, cs.y, mm);
            }
            for (int e = mt.g_begin + 1; e < mt.g_end; ++e) {
                const int g = s_mat_gates[e];
                const double2 cs = trig[g];
                double2 gg[4];
                gate_matrix(s_gates[g].kind, cs.x, cs.y, gg);
                const double2 n0 = cadd(cmul(gg[0], mm[0]), cmul(gg[1], mm[2]));
                const double2 n1 = cadd(cmul(gg[0], mm[1]), cmul(gg[1], mm[3]));
                const double2 n2 = cadd(cmul(gg[2], mm[0]), cmul(gg[3], mm[2]));
                const double2 n3 = cadd(cmul(gg[2], mm[1]), cmul(gg[3], mm[3]));
                mm[0] = n0; mm[1] = n1; mm[2] = n2; mm[3] = n3;
            }
            u2[4 * f + 0] = mm[0]; u2[4 * f + 1] = mm[1]; u2[4 * f + 2] = mm[2]; u2[4 * f + 3] = mm[3];
        }
        __syncwarp();

        for (int ip = 0; ip < n_passes; ++ip) {
            const SvPass ps = s_passes[ip];
            if (ps.nq == 3) run_pass<(Q >= 3 ? 3 : 1)>(amp, ps, s_ops, u2, trig, lig, G::LPS, G::DIM >> 3);
            else if (ps.nq == 2) run_pass<(Q >= 2 ? 2 : 1)>(amp, ps, s_ops, u2, trig, lig, G::LPS, G::DIM >> 2);
            else run_pass<1>(amp, ps, s_ops, u2, trig, lig, G::LPS, G::DIM >> 1);
            __syncwarp();
        }

        if (WANT_STATES) {
            if (live) {
                double2* dst = reinterpret_cast<double2*>(out) + (size_t)st * G::DIM;
                for (int i = lig; i < G::DIM; i += G::LPS) dst[i] = amp[sv_phys(i)];
            }
        } else {
            double* dst = out + (size_t)st * m;
            constexpr int FULL = Q / 3, REM = Q % 3;
#pragma unroll 1
            for (int b = 0; b < FULL; ++b) features_block<(Q >= 3 ? 3 : 1), Q>(amp, 3 * b, lig, G::LPS, live, dst);
            if (REM == 2) features_block<(Q >= 2 ? 2 : 1), Q>(amp, 3 * FULL, lig, G::LPS, live, dst);
            if (REM == 1) features_block<1, Q>(amp, 3 * FULL, lig, G::LPS, live, dst);
        }
        __syncwarp();
    }
}

// ---- q >= 9: one state per CTA (2^(q-3) threads: 64 .. 512), so the 16 KB+ of amplitudes per state buy
// 2..16 warps of parallelism instead of one (q=10 warp-per-state ran at 8 warps/SM: 139 ms per agent at config 5).
template <int Q, bool WANT_STATES>
__global__ void __launch_bounds__(((1 << Q) >> 3)) statevec_block_kernel(const dqgp_gate* __restrict__ gates, int n_gates,
                                                                          const SvPass* __restrict__ passes, int n_passes,
                                                                          const SvOp* __restrict__ ops, const SvMat* __restrict__ mats,
                                                                          int n_mats, const int* __restrict__ mat_gates,
                                                                          int n_mat_gates, int d, int P, int uses_acos,
                                                                          const double* __restrict__ X, int n,
                                                                          const double* __restrict__ Pm, int S, double* __restrict__ out) {
    constexpr int DIM = 1 << Q;
    constexpr int TEAM = DIM >> 3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const size_t gate_bytes = (sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15);
    const size_t pass_bytes = (sizeof(SvPass) * n_passes + 15) & ~size_t(15);
    const size_t op_bytes = (sizeof(SvOp) * n_gates + 15) & ~size_t(15);
    const size_t mat_bytes = (sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15);
    dqgp_gate* s_gates = reinterpret_cast<dqgp_gate*>(smem_raw);
    SvPass* s_passes = reinterpret_cast<SvPass*>(smem_raw + gate_bytes);
    SvOp* s_ops = reinterpret_cast<SvOp*>(smem_raw + gate_bytes + pass_bytes);
    SvMat* s_mats = reinterpret_cast<SvMat*>(smem_raw + gate_bytes + pass_bytes + op_bytes);
    int* s_mat_gates = reinterpret_cast<int*>(s_mats + n_mats);
    double2* amp = reinterpret_cast<double2*>(smem_raw + gate_bytes + pass_bytes + op_bytes + mat_bytes);
    double2* trig = amp + DIM;
    double2* u2 = trig + n_gates;
    double* acx = reinterpret_cast<double*>(u2 + 4 * n_mats);
    double* red = acx + ((d + 1) & ~1);
    const int tid = threadIdx.x;
    for (int i = tid; i < n_gates; i += TEAM) { s_gates[i] = gates[i]; s_ops[i] = ops[i]; }
    for (int i = tid; i < n_passes; i += TEAM) s_passes[i] = passes[i];
    for (int i = tid; i < n_mats; i += TEAM) s_mats[i] = mats[i];
    for (int i = tid; i < n_mat_gates; i += TEAM) s_mat_gates[i] = mat_gates[i];
    __syncthreads();
    const long long total = (long long)S * n;
    const int m = 3 * Q;
    for (long long st = blockIdx.x; st < total; st += gridDim.x) {
        const int s = int(st / n), j = int(st % n);
        const double* x = X + (size_t)j * d;
        const double* p = Pm + (size_t)s * P;
        if (uses_acos) {
            for (int f = tid; f < d; f += TEAM) acx[f] = acos(x[f]);
            __syncthreads();
        }
        for (int g = tid; g < n_gates; g += TEAM) {
            const dqgp_gate gt = s_gates[g];
            if (gt.form == DQGP_A_NONE) continue;
            double ang = 0.0;
            switch (gt.form) {
                case DQGP_A_P: ang = p[gt.pidx]; break;
                case DQGP_A_X: ang = x[gt.fidx]; break;
                case DQGP_A_P_PLUS_CX: ang = p[gt.pidx] + gt.coef * x[gt.fidx]; break;
                case DQGP_A_P_TIMES_ACOS: ang = p[gt.pidx] * acx[gt.fidx]; break;
                case DQGP_A_C_TIMES_ACOS: ang = gt.coef * acx[gt.fidx]; break;
                default: break;
            }
            double sn, cs;
            sincos(0.5 * ang, &sn, &cs);
            trig[g] = make_double2(cs, sn);
        }
        for (int i = tid; i < DIM; i += TEAM) amp[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);
        __syncthreads();
        for (int f = tid; f < n_mats; f += TEAM) {
            const SvMat mt = s_mats[f];
            double2 mm[4];
            {
                const int g0 = s_mat_gates[mt.g_begin];
                const double2 cs = trig[g0];
                gate_matrix(s_gates[g0].kind, cs.x, cs.y, mm);
            }
            for (int e = mt.g_begin + 1; e < mt.g_end; ++e) {
                const int g = s_mat_gates[e];
                const double2 cs = trig[g];
                double2 gg[4];
                gate_matrix(s_gates[g].kind, cs.x, cs.y, gg);
                const double2 n0 = cadd(cmul(gg[0], mm[0]), cmul(gg[1], mm[2]));
                const double2 n1 = cadd(cmul(gg[0], mm[1]), cmul(gg[1], mm[3]));
                const double2 n2 = cadd(cmul(gg[2], mm[0]), cmul(gg[3], mm[2]));
                const double2 n3 = cadd(cmul(gg[2], mm[1]), cmul(gg[3], mm[3]));
                mm[0] = n0; mm[1] = n1; mm[2] = n2; mm[3] = n3;
            }
            u2[4 * f + 0] = mm[0]; u2[4 * f + 1] = mm[1]; u2[4 * f + 2] = mm[2]; u2[4 * f + 3] = mm[3];
        }
        __syncthreads();
        for (int ip = 0; ip < n_passes; ++ip) {
            const SvPass ps = s_passes[ip];
            if (ps.nq == 3) run_pass<3>(amp, ps, s_ops, u2, trig, tid, TEAM, DIM >> 3);
            else if (ps.nq == 2) run_pass<2>(amp, ps, s_ops, u2, trig, tid, TEAM, DIM >> 2);
            else run_pass<1>(amp, ps, s_ops, u2, trig, tid, TEAM, DIM >> 1);
            __syncthreads();
        }
        if (WANT_STATES) {
            double2* dst = reinterpret_cast<double2*>(out) + (size_t)st * DIM;
            for (int i = tid; i < DIM; i += TEAM) dst[i] = amp[sv_phys(i)];
        } else {
            double* dst = out + (size_t)st * m;
            constexpr int FULL = Q / 3, REM = Q % 3;
#pragma unroll 1
            for (int b = 0; b < FULL; ++b) features_block<3, Q>(amp, 3 * b, tid, TEAM, true, dst, red);
            if (REM == 2) features_block<2, Q>(amp, 3 * FULL, tid, TEAM, true, dst, red);
            if (REM == 1) features_block<1, Q>(amp, 3 * FULL, tid, TEAM, true, dst, red);
        }
        __syncthreads();
    }
}

// ---- all 2P+1 central-difference parameter sets of one sample with PREFIX SHARING ---------------------------------
// Set s = 1+2i+sg differs from the base set only in parameter i, i.e. in ONE fused matrix (or one CRZ angle) of the
// plan.  A team (lane group / warp for q <= 8, CTA for q >= 9) owns one sample: it advances the base state pass by pass
// and, before executing pass p, forks every parameter whose op lives in pass p: copy base -> scratch, run passes p..end
// with the replaced matrix, reduce the features.  Work drops from (2P+1) full circuits to 1 + sum_i 2*(suffix of i):
// ~1.6x fewer pass executions for config 4, ~1.8x for config 5 — and results are bit-identical to the per-set kernel.
__device__ __forceinline__ double np_mod_d(double x, double p) {
    double r = fmod(x, p);
    if (r != 0.0) { if ((p < 0.0) != (r < 0.0)) r += p; } else r = copysign(0.0, p);
    return r;
}

__device__ __forceinline__ double gate_angle(const dqgp_gate& gt, double pval, const double* __restrict__ x, const double* __restrict__ acx) {
    switch (gt.form) {
        case DQGP_A_P: return pval;
        case DQGP_A_X: return x[gt.fidx];
        case DQGP_A_P_PLUS_CX: return pval + gt.coef * x[gt.fidx];
        case DQGP_A_P_TIMES_ACOS: return pval * acx[gt.fidx];
        case DQGP_A_C_TIMES_ACOS: return gt.coef * acx[gt.fidx];
        default: return 0.0;
    }
}

// compose fused matrix f from the cos/sin table, with gate `g_alt` (if >= 0) using `cs_alt` instead of its table entry
__device__ __forceinline__ void compose_matrix(const SvMat mt, const int* __restrict__ s_mat_gates, const dqgp_gate* __restrict__ s_gates,
                                               const double2* __restrict__ trig, int g_alt, double2 cs_alt, double2* __restrict__ dst) {
    double2 mm[4];
    {
        const int g0 = s_mat_gates[mt.g_begin];
        const double2 cs = (g0 == g_alt) ? cs_alt : trig[g0];
        gate_matrix(s_gates[g0].kind, cs.x, cs.y, mm);
    }
    for (int e = mt.g_begin + 1; e < mt.g_end; ++e) {
        const int g = s_mat_gates[e];
        const double2 cs = (g == g_alt) ? cs_alt : trig[g];
        double2 gg[4];
        gate_matrix(s_gates[g].kind, cs.x, cs.y, gg);
        const double2 n0 = cadd(cmul(gg[0], mm[0]), cmul(gg[1], mm[2]));
        const double2 n1 = cadd(cmul(gg[0], mm[1]), cmul(gg[1], mm[3]));
        const double2 n2 = cadd(cmul(gg[2], mm[0]), cmul(gg[3], mm[2]));
        const double2 n3 = cadd(cmul(gg[2], mm[1]), cmul(gg[3], mm[3]));
        mm[0] = n0; mm[1] = n1; mm[2] = n2; mm[3] = n3;
    }
    dst[0] = mm[0]; dst[1] = mm[1]; dst[2] = mm[2]; dst[3] = mm[3];
}

template <int Q>
struct SvTeam {
    static constexpr bool BLOCK = Q >= 9;
    static constexpr int DIM = 1 << Q;
    static constexpr int SIZE = BLOCK ? (DIM >> 3) : SvGeom<Q>::LPS;      // threads cooperating on one sample
    static constexpr int PER_WARP = BLOCK ? 1 : SvGeom<Q>::SPW;           // samples per warp (lane-group teams)
    static constexpr int SLOTS = SIZE < 32 ? SIZE : 32;                   // forks whose matrices are prepared together
    static constexpr int THREADS = BLOCK ? SIZE : 128;
    __device__ static __forceinline__ void sync() { if (BLOCK) __syncthreads(); else __syncwarp(); }
};

template <int Q, bool WANT_STATES>
__device__ __forceinline__ void sv_emit(const double2* __restrict__ amp, int lig, bool live, double* __restrict__ out, long long row,
                                        double* __restrict__ red) {
    using T = SvTeam<Q>;
    if (WANT_STATES) {
        if (live) {
            double2* dst = reinterpret_cast<double2*>(out) + (size_t)row * T::DIM;
            for (int i = lig; i < T::DIM; i += T::SIZE) dst[i] = amp[sv_phys(i)];
        }
    } else {
        double* dst = out + (size_t)row * (3 * Q);
        constexpr int FULL = Q / 3, REM = Q % 3;
#pragma unroll 1
        for (int b = 0; b < FULL; ++b) features_block<(Q >= 3 ? 3 : 1), Q>(amp, 3 * b, lig, T::SIZE, live, dst, red);
        if (REM == 2) features_block<(Q >= 2 ? 2 : 1), Q>(amp, 3 * FULL, lig, T::SIZE, live, dst, red);
        if (REM == 1) features_block<1, Q>(amp, 3 * FULL, lig, T::SIZE, live, dst, red);
    }
}

template <int Q>
__device__ __forceinline__ void sv_run_passes(double2* __restrict__ amp, const SvPass* __restrict__ s_passes, int p_from, int n_passes,
                                              const SvOp* __restrict__ s_ops, const double2* __restrict__ u2, const double2* __restrict__ trig,
                                              int lig, const SvAlt alt, int only_one) {
    using T = SvTeam<Q>;
    const int p_to = only_one ? p_from + 1 : n_passes;
    for (int ip = p_from; ip < p_to; ++ip) {
        const SvPass ps = s_passes[ip];
        if (ps.nq == 3) run_pass<(Q >= 3 ? 3 : 1)>(amp, ps, s_ops, u2, trig, lig, T::SIZE, T::DIM >> 3, alt);
        else if (ps.nq == 2) run_pass<(Q >= 2 ? 2 : 1)>(amp, ps, s_ops, u2, trig, lig, T::SIZE, T::DIM >> 2, alt);
        else run_pass<1>(amp, ps, s_ops, u2, trig, lig, T::SIZE, T::DIM >> 1, alt);
        T::sync();
    }
}

template <int Q, bool WANT_STATES>
__global__ void __launch_bounds__(SvTeam<Q>::THREADS) statevec_shared_kernel(
    const dqgp_gate* __restrict__ gates, int n_gates, const SvPass* __restrict__ passes, int n_passes, const SvOp* __restrict__ ops,
    const SvMat* __restrict__ mats, int n_mats, const int* __restrict__ mat_gates, int n_mat_gates, const int* __restrict__ share,
    int d, int P, int uses_acos, const double* __restrict__ X, int n, const double* __restrict__ Pm, double* __restrict__ out) {
    using T = SvTeam<Q>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const size_t gate_bytes = (sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15);
    const size_t pass_bytes = (sizeof(SvPass) * n_passes + 15) & ~size_t(15);
    const size_t op_bytes = (sizeof(SvOp) * n_gates + 15) & ~size_t(15);
    const size_t mat_bytes = (sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15);
    const int n_share = 2 * P + n_passes + 1 + P;
    const size_t share_bytes = (sizeof(int) * n_share + 15) & ~size_t(15);
    dqgp_gate* s_gates = reinterpret_cast<dqgp_gate*>(smem_raw);
    SvPass* s_passes = reinterpret_cast<SvPass*>(smem_raw + gate_bytes);
    SvOp* s_ops = reinterpret_cast<SvOp*>(smem_raw + gate_bytes + pass_bytes);
    SvMat* s_mats = reinterpret_cast<SvMat*>(smem_raw + gate_bytes + pass_bytes + op_bytes);
    int* s_mat_gates = reinterpret_cast<int*>(s_mats + n_mats);
    int* s_share = reinterpret_cast<int*>(smem_raw + gate_bytes + pass_bytes + op_bytes + mat_bytes);
    const int* par_gate = s_share;
    const int* par_mat = s_share + P;
    const int* pass_par_begin = s_share + 2 * P;
    const int* pass_params = s_share + 2 * P + n_passes + 1;
    for (int i = threadIdx.x; i < n_gates; i += blockDim.x) { s_gates[i] = gates[i]; s_ops[i] = ops[i]; }
    for (int i = threadIdx.x; i < n_passes; i += blockDim.x) s_passes[i] = passes[i];
    for (int i = threadIdx.x; i < n_mats; i += blockDim.x) s_mats[i] = mats[i];
    for (int i = threadIdx.x; i < n_mat_gates; i += blockDim.x) s_mat_gates[i] = mat_gates[i];
    for (int i = threadIdx.x; i < n_share; i += blockDim.x) s_share[i] = share[i];
    __syncthreads();

    // per-team storage: base amplitudes | scratch amplitudes | cos/sin table | fused matrices | fork matrices | acos | reduction
    const size_t team_bytes = sizeof(double2) * (2 * T::DIM + n_gates + 4 * n_mats + 4 * T::SLOTS) +
                              sizeof(double) * (((d + 1) & ~1) + (T::BLOCK ? 9 * (T::SIZE / 32) + 1 : 0));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int team_in_block = T::BLOCK ? 0 : warp * T::PER_WARP + lane / T::SIZE;
    const int lig = T::BLOCK ? threadIdx.x : lane % T::SIZE;
    const int teams_per_block = T::BLOCK ? 1 : (blockDim.x >> 5) * T::PER_WARP;
    unsigned char* my = smem_raw + gate_bytes + pass_bytes + op_bytes + mat_bytes + share_bytes + team_bytes * team_in_block;
    double2* base = reinterpret_cast<double2*>(my);
    double2* scr = base + T::DIM;
    double2* trig = scr + T::DIM;
    double2* u2 = trig + n_gates;
    double2* altm = u2 + 4 * n_mats;
    double* acx = reinterpret_cast<double*>(altm + 4 * T::SLOTS);
    double* red = acx + ((d + 1) & ~1);
    const SvAlt no_alt = SvAlt{-1, -1, nullptr, 0};

    // lane-group teams of one warp must iterate together (the plan is identical, only the data differ)
    const long long n_rounds = (n + (long long)gridDim.x * teams_per_block - 1) / ((long long)gridDim.x * teams_per_block);
    for (long long round = 0; round < n_rounds; ++round) {
        long long j = (round * gridDim.x + blockIdx.x) * teams_per_block + team_in_block;
        const bool live = j < n;
        if (!live) j = n - 1;
        const double* x = X + (size_t)j * d;
        if (uses_acos) {
            for (int f = lig; f < d; f += T::SIZE) acx[f] = acos(x[f]);
            T::sync();
        }
        for (int g = lig; g < n_gates; g += T::SIZE) {
            const dqgp_gate gt = s_gates[g];
            if (gt.form == DQGP_A_NONE) continue;
            double sn, cs;
            sincos(0.5 * gate_angle(gt, gt.pidx >= 0 ? Pm[gt.pidx] : 0.0, x, acx), &sn, &cs);
            trig[g] = make_double2(cs, sn);
        }
        for (int i = lig; i < T::DIM; i += T::SIZE) base[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0);
        T::sync();
        for (int f = lig; f < n_mats; f += T::SIZE) compose_matrix(s_mats[f], s_mat_gates, s_gates, trig, -1, make_double2(0, 0), u2 + 4 * f);
        T::sync();

        for (int ip = 0; ip < n_passes; ++ip) {
            const int pb = pass_par_begin[ip], pe = pass_par_begin[ip + 1];
            for (int f0 = 2 * pb; f0 < 2 * pe; f0 += T::SLOTS) {          // forks: (parameter, sign) pairs of this pass
                const int cnt = min(T::SLOTS, 2 * pe - f0);
                if (lig < cnt) {
                    const int fk = f0 + lig, i = pass_params[fk >> 1], sg = fk & 1;
                    const int g = par_gate[i];
                    double sn, cs;
                    sincos(0.5 * gate_angle(s_gates[g], Pm[(size_t)(1 + 2 * i + sg) * P + i], x, acx), &sn, &cs);
                    if (par_mat[i] >= 0) compose_matrix(s_mats[par_mat[i]], s_mat_gates, s_gates, trig, g, make_double2(cs, sn), altm + 4 * lig);
                    else altm[4 * lig] = make_double2(cs, sn);
                }
                T::sync();
                for (int t = 0; t < cnt; ++t) {
                    const int fk = f0 + t, i = pass_params[fk >> 1], sg = fk & 1;
                    for (int a = lig; a < T::DIM; a += T::SIZE) scr[a] = base[a];
                    T::sync();
                    const SvAlt alt = SvAlt{par_mat[i], par_mat[i] >= 0 ? -1 : par_gate[i], altm + 4 * t, 0};
                    sv_run_passes<Q>(scr, s_passes, ip, n_passes, s_ops, u2, trig, lig, alt, 0);
                    sv_emit<Q, WANT_STATES>(scr, lig, live, out, (long long)(1 + 2 * i + sg) * n + j, red);
                    T::sync();
                }
            }
            sv_run_passes<Q>(base, s_passes, ip, n_passes, s_ops, u2, trig, lig, no_alt, 1);
        }
        sv_emit<Q, WANT_STATES>(base, lig, live, out, j, red);
        T::sync();
    }
}

// ---- central-difference sets by LINEAR COMBINATION --------------------------------------------------------------------
// For a parameter that enters through ONE rotation R(theta) = exp(-i theta sigma / 2) (RX / RY / RZ: every parameter of yz_cx and
// kyriienko, the non-CRZ ones of chebyshev and hubregtsen), R(theta + D) = cos(D/2) R(theta) + sin(D/2) R(theta + pi), and the rest
// of the circuit is linear, so BOTH shifted states of that parameter are combinations of the base state psi and one extra state
// phi (the circuit with that gate's angle advanced by pi):   psi(D) = cos(D/2) psi + sin(D/2) phi,
//     <O>(D) = cos^2(D/2) <psi|O|psi> + sin^2(D/2) <phi|O|phi> + sin(D) Re<psi|O|phi>.
// One fork per parameter instead of two: P suffix simulations instead of 2P (D+ and D- are whatever the wrapped parameter sets of
// dqgp_shift_parameter_sets give for this sample: they need not be symmetric).  CRZ parameters keep the two-fork path.  Results
// equal the per-set simulation to rounding (1e-15), not bit for bit.
// JAC: instead of the two shifted sets, emit the exact feature Jacobian  d<O_k>/dp_i = (dtheta/dp_i) Re<psi|O_k|phi>  (the sin D
// coefficient above is the derivative at D = 0): out = base features (n, 3q), jac = (P, n, 3q); Pm is the single base row.
template <int Q, bool WANT_STATES, bool JAC = false>
__global__ void __launch_bounds__(SvTeam<Q>::THREADS) statevec_lc_kernel(
    const dqgp_gate* __restrict__ gates, int n_gates, const SvPass* __restrict__ passes, int n_passes, const SvOp* __restrict__ ops,
    const SvMat* __restrict__ mats, int n_mats, const int* __restrict__ mat_gates, int n_mat_gates, const int* __restrict__ share,
    int d, int P, int uses_acos, const double* __restrict__ X, int n, const double* __restrict__ Pm, double* __restrict__ out,
    double* __restrict__ jac = nullptr) {
    using T = SvTeam<Q>;
    constexpr int M3 = 3 * Q, M3P = (M3 + 1) & ~1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const size_t gate_bytes = (sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15);
    const size_t pass_bytes = (sizeof(SvPass) * n_passes + 15) & ~size_t(15);
    const size_t op_bytes = (sizeof(SvOp) * n_gates + 15) & ~size_t(15);
    const size_t mat_bytes = (sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15);
    const int n_share = 2 * P + n_passes + 1 + P;
    const size_t share_bytes = (sizeof(int) * n_share + 15) & ~size_t(15);
    dqgp_gate* s_gates = reinterpret_cast<dqgp_gate*>(smem_raw);
    SvPass* s_passes = reinterpret_cast<SvPass*>(smem_raw + gate_bytes);
    SvOp* s_ops = reinterpret_cast<SvOp*>(smem_raw + gate_bytes + pass_bytes);
    SvMat* s_mats = reinterpret_cast<SvMat*>(smem_raw + gate_bytes + pass_bytes + op_bytes);
    int* s_mat_gates = reinterpret_cast<int*>(s_mats + n_mats);
    int* s_share = reinterpret_cast<int*>(smem_raw + gate_bytes + pass_bytes + op_bytes + mat_bytes);
    const int* par_gate = s_share;
    const int* par_mat = s_share + P;
    const int* pass_par_begin = s_share + 2 * P;
    const int* pass_params = s_share + 2 * P + n_passes + 1;
    for (int i = threadIdx.x; i < n_gates; i += blockDim.x) { s_gates[i] = gates[i]; s_ops[i] = ops[i]; }
    for (int i = threadIdx.x; i < n_passes; i += blockDim.x) s_passes[i] = passes[i];
    for (int i = threadIdx.x; i < n_mats; i += blockDim.x) s_mats[i] = mats[i];
    for (int i = threadIdx.x; i < n_mat_gates; i += blockDim.x) s_mat_gates[i] = mat_gates[i];
    for (int i = threadIdx.x; i < n_share; i += blockDim.x) s_share[i] = share[i];
    __syncthreads();

    // per-team storage: base | scratch | final base state | cos/sin table | fused matrices | fork matrices | acos | reduction | A,B,C
    const size_t team_bytes = sizeof(double2) * (3 * T::DIM + n_gates + 4 * n_mats + 4 * T::SLOTS) +
                              sizeof(double) * (((d + 1) & ~1) + (T::BLOCK ? 9 * (T::SIZE / 32) + 1 : 0) + 3 * M3P);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int team_in_block = T::BLOCK ? 0 : warp * T::PER_WARP + lane / T::SIZE;
    const int lig = T::BLOCK ? threadIdx.x : lane % T::SIZE;
    const int teams_per_block = T::BLOCK ? 1 : (blockDim.x >> 5) * T::PER_WARP;
    unsigned char* my = smem_raw + gate_bytes + pass_bytes + op_bytes + mat_bytes + share_bytes + team_bytes * team_in_block;
    double2* base = reinterpret_cast<double2*>(my);
    double2* scr = base + T::DIM;
    double2* fin = scr + T::DIM;
    double2* trig = fin + T::DIM;
    double2* u2 = trig + n_gates;
    double2* altm = u2 + 4 * n_mats;
    double* acx = reinterpret_cast<double*>(altm + 4 * T::SLOTS);
    double* red = acx + ((d + 1) & ~1);
    double* featA = red + (T::BLOCK ? 9 * (T::SIZE / 32) + 1 : 0);
    double* featB = featA + M3P;
    double* featC = featB + M3P;
    const SvAlt no_alt = SvAlt{-1, -1, nullptr, 0};
    constexpr int FULL = Q / 3, REM = Q % 3;

    const long long n_rounds = (n + (long long)gridDim.x * teams_per_block - 1) / ((long long)gridDim.x * teams_per_block);
    for (long long round = 0; round < n_rounds; ++round) {
        long long j = (round * gridDim.x + blockIdx.x) * teams_per_block + team_in_block;
        const bool live = j < n;
        if (!live) j = n - 1;
        const double* x = X + (size_t)j * d;
        if (uses_acos) {
            for (int f = lig; f < d; f += T::SIZE) acx[f] = acos(x[f]);
            T::sync();
        }
        for (int g = lig; g < n_gates; g += T::SIZE) {
            const dqgp_gate gt = s_gates[g];
            if (gt.form == DQGP_A_NONE) continue;
            double sn, cs;
            sincos(0.5 * gate_angle(gt, gt.pidx >= 0 ? Pm[gt.pidx] : 0.0, x, acx), &sn, &cs);
            trig[g] = make_double2(cs, sn);
        }
        for (int i = lig; i < T::DIM; i += T::SIZE) { base[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0); fin[i] = base[i]; }
        T::sync();
        for (int f = lig; f < n_mats; f += T::SIZE) compose_matrix(s_mats[f], s_mat_gates, s_gates, trig, -1, make_double2(0, 0), u2 + 4 * f);
        T::sync();

        // sweep 1: the final base state (kept for the cross terms) and the base set's output
        sv_run_passes<Q>(fin, s_passes, 0, n_passes, s_ops, u2, trig, lig, no_alt, 0);
        if (WANT_STATES) {
            sv_emit<Q, true>(fin, lig, live, out, j, red);
        } else {
#pragma unroll 1
            for (int b = 0; b < FULL; ++b) features_block<(Q >= 3 ? 3 : 1), Q>(fin, 3 * b, lig, T::SIZE, true, featA, red);
            if (REM == 2) features_block<(Q >= 2 ? 2 : 1), Q>(fin, 3 * FULL, lig, T::SIZE, true, featA, red);
            if (REM == 1) features_block<1, Q>(fin, 3 * FULL, lig, T::SIZE, true, featA, red);
            T::sync();
            if (live)
                for (int k = lig; k < M3; k += T::SIZE) out[(size_t)j * M3 + k] = featA[k];
        }
        T::sync();

        // sweep 2: advance the base pass by pass; fork every parameter whose op lives in the pass about to run
        for (int ip = 0; ip < n_passes; ++ip) {
            const int pb = pass_par_begin[ip], pe = pass_par_begin[ip + 1];
            for (int f0 = 2 * pb; f0 < 2 * pe; f0 += T::SLOTS) {
                const int cnt = min(T::SLOTS, 2 * pe - f0);
                if (lig < cnt) {
                    const int fk = f0 + lig, i = pass_params[fk >> 1], sg = fk & 1;
                    const int g = par_gate[i];
                    if (par_mat[i] >= 0) {
                        // rotation: one fork with the gate's angle advanced by pi: (cos, sin)(theta/2 + pi/2) = (-sin, cos)(theta/2)
                        if (sg == 0) compose_matrix(s_mats[par_mat[i]], s_mat_gates, s_gates, trig, g, make_double2(-trig[g].y, trig[g].x), altm + 4 * lig);
                    } else if (!JAC) {
                        double sn, cs;
                        sincos(0.5 * gate_angle(s_gates[g], Pm[(size_t)(1 + 2 * i + sg) * P + i], x, acx), &sn, &cs);
                        altm[4 * lig] = make_double2(cs, sn);
                    } else if (sg == 0) {
                        altm[4 * lig] = make_double2(-trig[g].y, trig[g].x);     // CRZ derivative fork: RZ(theta + pi) on the control-on pairs
                    }
                }
                T::sync();
                for (int t = 0; t < cnt; ++t) {
                    const int fk = f0 + t, i = pass_params[fk >> 1], sg = fk & 1;
                    const bool rot = par_mat[i] >= 0;
                    if ((rot || JAC) && sg == 1) continue;        // both signs (or the derivative) come out of the sg = 0 fork
                    for (int a = lig; a < T::DIM; a += T::SIZE) scr[a] = base[a];
                    T::sync();
                    const SvAlt alt = SvAlt{par_mat[i], rot ? -1 : par_gate[i], altm + 4 * t, (JAC && !rot) ? 1 : 0};
                    sv_run_passes<Q>(scr, s_passes, ip, n_passes, s_ops, u2, trig, lig, alt, 0);
                    if (!rot && !JAC) {
                        sv_emit<Q, WANT_STATES>(scr, lig, live, out, (long long)(1 + 2 * i + sg) * n + j, red);
                    } else if (JAC) {
                        // d<O>/dtheta = Re<psi|O|phi> (phi: the gate's angle advanced by pi; for a CRZ also projected on control = 1);
                        // dtheta/dp = 1 (p, p + c x) or arccos(x) (p arccos x)
                        const dqgp_gate gt = s_gates[par_gate[i]];
                        const double dth = (gt.form == DQGP_A_P_TIMES_ACOS) ? acx[gt.fidx] : 1.0;
                        if (WANT_STATES) {
                            // d psi / dp = (dtheta/dp) phi / 2
                            if (live) {
                                double2* dst = reinterpret_cast<double2*>(jac) + ((size_t)i * n + j) * T::DIM;
                                for (int a = lig; a < T::DIM; a += T::SIZE) {
                                    const double2 v = scr[sv_phys(a)];
                                    dst[a] = make_double2(0.5 * dth * v.x, 0.5 * dth * v.y);
                                }
                            }
                        } else {
#pragma unroll 1
                            for (int b = 0; b < FULL; ++b) features_cross_block<(Q >= 3 ? 3 : 1), Q>(fin, scr, 3 * b, lig, T::SIZE, featC, red);
                            if (REM == 2) features_cross_block<(Q >= 2 ? 2 : 1), Q>(fin, scr, 3 * FULL, lig, T::SIZE, featC, red);
                            if (REM == 1) features_cross_block<1, Q>(fin, scr, 3 * FULL, lig, T::SIZE, featC, red);
                            T::sync();
                            if (live)
                                for (int k = lig; k < M3; k += T::SIZE) jac[((size_t)i * n + j) * M3 + k] = dth * featC[k];
                        }
                    } else {
                        const dqgp_gate gt = s_gates[par_gate[i]];
                        const double th0 = gate_angle(gt, Pm[i], x, acx);
                        double c[2], sn[2];
#pragma unroll
                        for (int e = 0; e < 2; ++e)
                            sincos(0.5 * (gate_angle(gt, Pm[(size_t)(1 + 2 * i + e) * P + i], x, acx) - th0), &sn[e], &c[e]);
                        if (WANT_STATES) {
                            if (live) {
#pragma unroll
                                for (int e = 0; e < 2; ++e) {
                                    double2* dst = reinterpret_cast<double2*>(out) + ((size_t)(1 + 2 * i + e) * n + j) * T::DIM;
                                    for (int a = lig; a < T::DIM; a += T::SIZE) {
                                        const double2 u = fin[sv_phys(a)], v = scr[sv_phys(a)];
                                        dst[a] = make_double2(fma(c[e], u.x, sn[e] * v.x), fma(c[e], u.y, sn[e] * v.y));
                                    }
                                }
                            }
                        } else {
#pragma unroll 1
                            for (int b = 0; b < FULL; ++b) {
                                features_block<(Q >= 3 ? 3 : 1), Q>(scr, 3 * b, lig, T::SIZE, true, featB, red);
                                features_cross_block<(Q >= 3 ? 3 : 1), Q>(fin, scr, 3 * b, lig, T::SIZE, featC, red);
                            }
                            if (REM == 2) {
                                features_block<(Q >= 2 ? 2 : 1), Q>(scr, 3 * FULL, lig, T::SIZE, true, featB, red);
                                features_cross_block<(Q >= 2 ? 2 : 1), Q>(fin, scr, 3 * FULL, lig, T::SIZE, featC, red);
                            }
                            if (REM == 1) {
                                features_block<1, Q>(scr, 3 * FULL, lig, T::SIZE, true, featB, red);
                                features_cross_block<1, Q>(fin, scr, 3 * FULL, lig, T::SIZE, featC, red);
                            }
                            T::sync();
                            if (live) {
                                for (int k = lig; k < M3; k += T::SIZE) {
                                    const double A = featA[k], B = featB[k], C = featC[k];
#pragma unroll
                                    for (int e = 0; e < 2; ++e)
                                        out[((size_t)(1 + 2 * i + e) * n + j) * M3 + k] =
                                            fma(c[e] * c[e], A, fma(sn[e] * sn[e], B, 2.0 * sn[e] * c[e] * C));
                                }
                            }
                        }
                    }
                    T::sync();
                }
            }
            sv_run_passes<Q>(base, s_passes, ip, n_passes, s_ops, u2, trig, lig, no_alt, 1);
        }
        T::sync();
    }
}

// ---- lc2: the linear-combination form, rebuilt around what ncu showed in round 2 (profiles/r02_sv_q10_before.txt: FP64 pipe
// 33%, issue slots 52%, 68% of all instructions are not FP64) -------------------------------------------------------------------
// For circuits whose parameters ALL enter through one RX / RY / RZ (yz_cx, kyriienko: BASELINE configs 4 and 5), features only.
//  * TWO forks advance together through every pass (run_pass3<Q, B, 2>): the op decode, address arithmetic and
//    fused-matrix loads of a pass are paid once for two states, and every thread carries two independent FP64 chains;
//  * the first pass of a fork reads the base state and writes the fork's scratch (no copy);
//  * ONE epilogue sweep per fork gives <phi|O|phi> and Re<psi|O|phi> together (each scratch amplitude is loaded once per qubit
//    group instead of twice), the Z observables come from elementwise products in a single layout (they need no pairing);
//  * team reductions halve the data with every shuffle step (team_reduce) instead of all-reducing every value: 85 shuffle steps
//    per fork instead of 300 - SHFL issues once per cycle per SM, it was 14% of the kernel's time;
//  * the gate program is read from global memory (uniform, L1-resident) instead of being copied into every CTA's shared memory.
// __noinline__: one copy of each instantiation for all call sites (the inlined version stalled 14% of the time on instruction
// fetch, profiles/r02_sv_q10_lc2_v1.txt).
// ---- CX-free passes (SvPass3): the coset a thread owns is selected by the bits of its index through the pass's rest masks; register j
// holds the amplitude whose logical block bits are j.  Only fused 2x2 unitaries are executed: CX gates live in the index map.
template <int NREST>
__device__ __forceinline__ int coset_base(const int* __restrict__ rest, int gi) {
    int p0 = 0;
#pragma unroll
    for (int i = 0; i < NREST; ++i) p0 ^= (-((gi >> i) & 1)) & rest[i];
    return p0;
}

template <int Q, int B, int NS, bool ALT>
__device__ __noinline__ void run_pass3(const double2* __restrict__ src0, const double2* __restrict__ src1, double2* __restrict__ dst0,
                                       double2* __restrict__ dst1, const SvPass3* __restrict__ pass, const SvOp* __restrict__ ops,
                                       const double2* __restrict__ mats, int lig, int lps, int alt_mat0, const double2* __restrict__ alt_u0,
                                       int alt_mat1, const double2* __restrict__ alt_u1) {
    constexpr int N = 1 << B, GROUPS = (1 << Q) >> B;
    const int m0 = pass->bm[0], m1 = pass->bm[1], m2 = pass->bm[2];
    const int op_begin = pass->op_begin, op_end = pass->op_end;
    int comb[N];
#pragma unroll
    for (int j = 0; j < N; ++j) comb[j] = ((j & 1) ? m0 : 0) ^ ((B > 1 && (j & 2)) ? m1 : 0) ^ ((B > 2 && (j & 4)) ? m2 : 0);
    for (int gi = lig; gi < GROUPS; gi += lps) {
        const int p0 = coset_base<Q - B>(pass->rest, gi);
        int addr[N];
        double2 r0[N], r1[N];      // r1 is dead code for NS == 1
#pragma unroll
        for (int j = 0; j < N; ++j) {
            addr[j] = sv_phys(p0 ^ comb[j]);
            r0[j] = src0[addr[j]];
            if (NS == 2) r1[j] = src1[addr[j]];
        }
        SvOp nxt = ops[op_begin];
#pragma unroll 1
        for (int o = op_begin; o < op_end; ++o) {
            const SvOp op = nxt;
            if (o + 1 < op_end) nxt = ops[o + 1];
            const double2* u0 = mats + 4 * op.idx;
            const double2* u1 = u0;
            if (ALT) {
                if (op.idx == alt_mat0) u0 = alt_u0;
                if (NS == 2 && op.idx == alt_mat1) u1 = alt_u1;
            }
            double2 a = u0[0], b = u0[1], c = u0[2], d = u0[3];
            if (op.lbit == 0) apply_u2<N, 0>(r0, a, b, c, d);
            else if (B > 1 && op.lbit == 1) apply_u2<N, (B > 1 ? 1 : 0)>(r0, a, b, c, d);
            else if (B > 2) apply_u2<N, (B > 2 ? 2 : 0)>(r0, a, b, c, d);
            if (NS == 2) {
                if (ALT && u1 != u0) { a = u1[0]; b = u1[1]; c = u1[2]; d = u1[3]; }
                if (op.lbit == 0) apply_u2<N, 0>(r1, a, b, c, d);
                else if (B > 1 && op.lbit == 1) apply_u2<N, (B > 1 ? 1 : 0)>(r1, a, b, c, d);
                else if (B > 2) apply_u2<N, (B > 2 ? 2 : 0)>(r1, a, b, c, d);
            }
        }
#pragma unroll
        for (int j = 0; j < N; ++j) {
            dst0[addr[j]] = r0[j];
            if (NS == 2) dst1[addr[j]] = r1[j];
        }
    }
}

template <int Q, int NS, bool ALT>
__device__ __forceinline__ void sv_pass3(const double2* src0, const double2* src1, double2* dst0, double2* dst1, const SvPass3* ps_ptr,
                                         const SvOp* __restrict__ ops, const double2* __restrict__ u2, int lig, int am0, const double2* au0,
                                         int am1, const double2* au1) {
    using T = SvTeam<Q>;
    const int nq = ps_ptr->nq;
    if (nq == 3) run_pass3<Q, (Q >= 3 ? 3 : 1), NS, ALT>(src0, src1, dst0, dst1, ps_ptr, ops, u2, lig, T::SIZE, am0, au0, am1, au1);
    else if (nq == 2) run_pass3<Q, (Q >= 2 ? 2 : 1), NS, ALT>(src0, src1, dst0, dst1, ps_ptr, ops, u2, lig, T::SIZE, am0, au0, am1, au1);
    else run_pass3<Q, 1, NS, ALT>(src0, src1, dst0, dst1, ps_ptr, ops, u2, lig, T::SIZE, am0, au0, am1, au1);
    T::sync();
}

// Sum v[0..N) over the W (power of two, <= 32, aligned) lanes of a team, halving the data with every shuffle step: a lane
// whose bit m is set keeps the upper half and sends the lower one.  Afterwards slots [0, max(1, N/W)) of every lane hold the team
// totals of the original indices idx_base + slot; when N < W the remaining steps all-reduce and `writer` marks one lane per index.
template <int N, int W>
__device__ __forceinline__ void team_reduce(double (&v)[N], int lane_in_team, int& idx_base, bool& writer) {
    idx_base = 0;
    writer = true;
    int n = N;
#pragma unroll
    for (int m = W >> 1; m >= 1; m >>= 1) {
        const bool hi = (lane_in_team & m) != 0;
        if (n > 1) {
            const int half = n >> 1;
#pragma unroll
            for (int j = 0; j < N / 2; ++j) {
                if (j < half) {
                    const double send = hi ? v[j] : v[j + half];
                    const double keep = hi ? v[j + half] : v[j];
                    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, m);
                }
            }
            idx_base += hi ? half : 0;
            n = half;
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], m);
            writer = writer && !hi;
        }
    }
}
template <int N, int W>
struct TeamReduceLeft { static constexpr int value = (N / W) > 1 ? (N / W) : 1; };

// value ids of one fork in the reduction buffer: [Bx | By | Bz | Cx | Cy | Cz] x Q, B = <phi|O|phi> (X, Y without their factor 2),
// C = Re<psi|O|phi>; red[id * NW + warp]
// positions through the final index map of the CX-free plan (`grp`: the group's block / rest masks)
template <int Q, int B>
__device__ __forceinline__ void lc2_group_xy(const double2* __restrict__ fin, const double2* __restrict__ scr, int k0, int lig, int warp,
                                             double* __restrict__ red, const SvPass3* __restrict__ grp) {
    using T = SvTeam<Q>;
    constexpr int N = 1 << B, NV = 16, W = T::SIZE < 32 ? T::SIZE : 32, NW = T::BLOCK ? T::SIZE / 32 : 1;
    const int groups = T::DIM >> B;
    double v[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = 0.0;
    int comb[N];
#pragma unroll
    for (int j = 0; j < N; ++j) comb[j] = ((j & 1) ? grp->bm[0] : 0) ^ ((B > 1 && (j & 2)) ? grp->bm[1] : 0) ^ ((B > 2 && (j & 4)) ? grp->bm[2] : 0);
    for (int gi = lig; gi < groups; gi += T::SIZE) {
        const int base = coset_base<Q - B>(grp->rest, gi);
        double2 p[N], s[N];
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const int a = sv_phys(base ^ comb[j]);
            p[j] = fin[a];
            s[j] = scr[a];
        }
#pragma unroll
        for (int l = 0; l < B; ++l)
#pragma unroll
            for (int j = 0; j < N; ++j) {
                if (j & (1 << l)) continue;
                const double2 a = s[j], b = s[j | (1 << l)], pa = p[j], pb = p[j | (1 << l)];
                v[0 * B + l] = fma(a.x, b.x, fma(a.y, b.y, v[0 * B + l]));                                   // Re conj(phi_a) phi_b
                v[1 * B + l] = fma(a.x, b.y, fma(-a.y, b.x, v[1 * B + l]));                                  // Im conj(phi_a) phi_b
                v[2 * B + l] = fma(pa.x, b.x, fma(pa.y, b.y, fma(pb.x, a.x, fma(pb.y, a.y, v[2 * B + l]))));    // Re<psi|X|phi>
                v[3 * B + l] = fma(pa.x, b.y, fma(-pa.y, b.x, fma(-pb.x, a.y, fma(pb.y, a.x, v[3 * B + l]))));  // Re<psi|Y|phi>
            }
    }
    int idx;
    bool writer;
    team_reduce<NV, W>(v, lig & (W - 1), idx, writer);
    constexpr int LEFT = TeamReduceLeft<NV, W>::value;
    if (writer) {
#pragma unroll
        for (int j = 0; j < LEFT; ++j) {
            const int e = idx + j;                 // slot = kind4 * B + l
            if (e < 4 * B) {
                const int kind4 = e / B, l = e - kind4 * B;
                const int id = (kind4 < 2 ? kind4 : kind4 + 1) * Q + k0 + l;      // Bx, By, Cx, Cy -> rows 0, 1, 3, 4
                red[id * NW + warp] = v[j];
            }
        }
    }
}

// Z observables of a fork from ONE layout (block qubits 0, 1, 2): <phi|Z_k|phi> = sum_a (+-)|phi_a|^2, Re<psi|Z_k|phi> likewise
template <int Q>
__device__ __forceinline__ void lc2_group_z(const double2* __restrict__ fin, const double2* __restrict__ scr, int lig, int warp,
                                            double* __restrict__ red, const SvPass3* __restrict__ grp) {
    using T = SvTeam<Q>;
    constexpr int NZ = (2 * Q <= 16) ? 16 : 32, W = T::SIZE < 32 ? T::SIZE : 32, NW = T::BLOCK ? T::SIZE / 32 : 1;
    double v[NZ];
#pragma unroll
    for (int i = 0; i < NZ; ++i) v[i] = 0.0;
    int comb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) comb[j] = ((j & 1) ? grp->bm[0] : 0) ^ ((j & 2) ? grp->bm[1] : 0) ^ ((j & 4) ? grp->bm[2] : 0);
    for (int gi = lig; gi < (T::DIM >> 3); gi += T::SIZE) {
        const int base = coset_base<(Q >= 3 ? Q - 3 : 0)>(grp->rest, gi);
        double pp[8], ww[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int a = sv_phys(base ^ comb[j]);
            const double2 ps = fin[a], ph = scr[a];
            pp[j] = fma(ph.x, ph.x, ph.y * ph.y);
            ww[j] = fma(ps.x, ph.x, ps.y * ph.y);
        }
        // block qubits: signed sums over the 8 slots; outside qubits: the slot total with the sign of the group's index bit
        const double p01 = pp[0] + pp[1], p23 = pp[2] + pp[3], p45 = pp[4] + pp[5], p67 = pp[6] + pp[7];
        const double w01 = ww[0] + ww[1], w23 = ww[2] + ww[3], w45 = ww[4] + ww[5], w67 = ww[6] + ww[7];
        v[0] += ((pp[0] - pp[1]) + (pp[2] - pp[3])) + ((pp[4] - pp[5]) + (pp[6] - pp[7]));
        v[Q + 0] += ((ww[0] - ww[1]) + (ww[2] - ww[3])) + ((ww[4] - ww[5]) + (ww[6] - ww[7]));
        v[1] += (p01 - p23) + (p45 - p67);
        v[Q + 1] += (w01 - w23) + (w45 - w67);
        const double plo = p01 + p23, phi_ = p45 + p67, wlo = w01 + w23, whi = w45 + w67;
        v[2] += plo - phi_;
        v[Q + 2] += wlo - whi;
        const double pt = plo + phi_, wt = wlo + whi;
#pragma unroll
        for (int k = 3; k < Q; ++k) {
            const bool neg = ((gi >> (k - 3)) & 1) != 0;
            v[k] += neg ? -pt : pt;
            v[Q + k] += neg ? -wt : wt;
        }
    }
    int idx;
    bool writer;
    team_reduce<NZ, W>(v, lig & (W - 1), idx, writer);
    constexpr int LEFT = TeamReduceLeft<NZ, W>::value;
    if (writer) {
#pragma unroll
        for (int j = 0; j < LEFT; ++j) {
            const int e = idx + j;                 // slot = z2 * Q + k
            if (e < 2 * Q) {
                const int z2 = e / Q, k = e - z2 * Q;
                red[((z2 ? 5 : 2) * Q + k) * NW + warp] = v[j];
            }
        }
    }
}

// one fork's epilogue: both central-difference sets of parameter i from A = <psi|O|psi> (featA), B, C
// all partial sums of one fork into `red` (no synchronisation); `grps`: the epilogue groups of the CX-free plan
template <int Q>
__device__ __forceinline__ void lc2_collect(const double2* __restrict__ fin, const double2* __restrict__ scr, double* __restrict__ red, int lig,
                                            const SvPass3* __restrict__ grps) {
    using T = SvTeam<Q>;
    constexpr int FULL = Q / 3, REM = Q % 3;
    const int warp = T::BLOCK ? (lig >> 5) : 0;
    lc2_group_z<Q>(fin, scr, lig, warp, red, grps);
#pragma unroll 1
    for (int b = 0; b < FULL; ++b) lc2_group_xy<Q, 3>(fin, scr, 3 * b, lig, warp, red, grps + b);
    if (REM == 2) lc2_group_xy<Q, 2>(fin, scr, 3 * FULL, lig, warp, red, grps + FULL);
    if (REM == 1) lc2_group_xy<Q, 1>(fin, scr, 3 * FULL, lig, warp, red, grps + FULL);
}

template <int Q>
__device__ __forceinline__ void lc2_emit(const double2* __restrict__ fin, const double2* __restrict__ scr, const double* __restrict__ featA,
                                         double* __restrict__ red, int lig, bool live, double c0, double s0, double c1, double s1,
                                         double* __restrict__ out_plus, double* __restrict__ out_minus, const SvPass3* __restrict__ grps) {
    using T = SvTeam<Q>;
    constexpr int NW = T::BLOCK ? T::SIZE / 32 : 1, M3 = 3 * Q;
    lc2_collect<Q>(fin, scr, red, lig, grps);
    T::sync();
    if (live) {
        for (int k = lig; k < M3; k += T::SIZE) {
            double Bv = 0.0, Cv = 0.0;
#pragma unroll
            for (int w = 0; w < NW; ++w) { Bv += red[k * NW + w]; Cv += red[(M3 + k) * NW + w]; }
            if (k < 2 * Q) Bv *= 2.0;            // X, Y: every pair was counted once
            const double A = featA[k];
            out_plus[k] = fma(c0 * c0, A, fma(s0 * s0, Bv, 2.0 * s0 * c0 * Cv));
            out_minus[k] = fma(c1 * c1, A, fma(s1 * s1, Bv, 2.0 * s1 * c1 * Cv));
        }
    }
    T::sync();
}

// Runs the CX-free plan (SvPass3 passes; CX gates absorbed into the logical -> physical index map, Pauli features read through the
// final map).  PAIR: where a CTA owns the state (q >= 9) two forks advance together through every pass (four state copies); a
// lane-group team (q <= 8) takes one fork at a time with three state copies (no second scratch).
// Resident CTAs the register allocation must allow: CTA-per-state teams up to q = 10 three CTAs (73 KB each).  Without the bound the
// q = 10 kernel takes 174 registers and drops to two CTAs per SM (39.8 ms at config 5 against 36.3 ms).  (An unpaired CTA-per-state
// variant - three copies, the plan read from global memory, four CTAs per SM - measured 37.3 ms there and was removed.)
template <int Q>
constexpr int LC2_MIN_BLOCKS = (SvTeam<Q>::BLOCK && Q <= 10) ? 3 : 0;      // 0 = unspecified
template <int Q>
__global__ void __launch_bounds__(SvTeam<Q>::THREADS, LC2_MIN_BLOCKS<Q>) statevec_lc2_kernel(
    const dqgp_gate* __restrict__ g_gates, int n_gates, const SvPass3* __restrict__ g_passes, int n_passes, const SvOp* __restrict__ g_ops,
    const SvMat* __restrict__ g_mats, int n_mats, const int* __restrict__ g_mat_gates, const int* __restrict__ g_share, int d, int P,
    int uses_acos, const double* __restrict__ X, int n, const double* __restrict__ Pm, double* __restrict__ out) {
    using T = SvTeam<Q>;
    using PassT = SvPass3;
    constexpr bool PAIR = T::BLOCK;
    constexpr int M3 = 3 * Q, M3P = (M3 + 1) & ~1, NW = T::BLOCK ? T::SIZE / 32 : 1;
    constexpr int N_EPI = (Q + 2) / 3;        // epilogue group entries stored after the real passes
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int* par_gate = g_share;
    const int* par_mat = g_share + P;
    const int* pass_par_begin = g_share + 2 * P;
    const int* pass_params = g_share + 2 * P + n_passes + 1;
    // per CTA: the op list and the pass table (read in every pass; the rest of the gate program stays in global memory)
    const size_t op_bytes = (sizeof(SvOp) * n_gates + 15) & ~size_t(15);
    const size_t pass_bytes = (sizeof(PassT) * (n_passes + N_EPI) + 15) & ~size_t(15);
    SvOp* s_ops = reinterpret_cast<SvOp*>(smem_raw);
    PassT* s_passes = reinterpret_cast<PassT*>(smem_raw + op_bytes);
    for (int i = threadIdx.x; i < n_gates; i += blockDim.x) s_ops[i] = g_ops[i];        // #ops <= #gates
    for (int i = threadIdx.x; i < n_passes + N_EPI; i += blockDim.x) s_passes[i] = g_passes[i];
    const SvPass3* epi = s_passes + n_passes;
    __syncthreads();
    // per-team storage: base | scratch 0 | scratch 1 | final base state | cos/sin table | fused matrices | 2 fork matrices | acos | red | A
    const size_t team_bytes = sizeof(double2) * ((PAIR ? 4 : 3) * T::DIM + n_gates + 4 * n_mats + 8) + sizeof(double) * (((d + 1) & ~1) + 2 * M3 * NW + M3P + 8);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int team_in_block = T::BLOCK ? 0 : warp * T::PER_WARP + lane / T::SIZE;
    const int lig = T::BLOCK ? threadIdx.x : lane % T::SIZE;
    const int teams_per_block = T::BLOCK ? 1 : (blockDim.x >> 5) * T::PER_WARP;
    unsigned char* my = smem_raw + op_bytes + pass_bytes + team_bytes * team_in_block;
    double2* base = reinterpret_cast<double2*>(my);
    double2* scr0 = base + T::DIM;
    double2* scr1 = PAIR ? scr0 + T::DIM : scr0;
    double2* fin = scr0 + (PAIR ? 2 : 1) * T::DIM;
    double2* trig = fin + T::DIM;
    double2* u2 = trig + n_gates;
    double2* altm = u2 + 4 * n_mats;
    double* acx = reinterpret_cast<double*>(altm + 8);
    double* red = acx + ((d + 1) & ~1);
    double* featA = red + 2 * M3 * NW;
    double* coef = featA + M3P;

    const long long n_rounds = (n + (long long)gridDim.x * teams_per_block - 1) / ((long long)gridDim.x * teams_per_block);
    for (long long round = 0; round < n_rounds; ++round) {
        long long j = (round * gridDim.x + blockIdx.x) * teams_per_block + team_in_block;
        const bool live = j < n;
        if (!live) j = n - 1;
        const double* x = X + (size_t)j * d;
        if (uses_acos) {
            for (int f = lig; f < d; f += T::SIZE) acx[f] = acos(x[f]);
            T::sync();
        }
        for (int g = lig; g < n_gates; g += T::SIZE) {
            const dqgp_gate gt = g_gates[g];
            if (gt.form == DQGP_A_NONE) continue;
            double sn, cs;
            sincos(0.5 * gate_angle(gt, gt.pidx >= 0 ? Pm[gt.pidx] : 0.0, x, acx), &sn, &cs);
            trig[g] = make_double2(cs, sn);
        }
        for (int i = lig; i < T::DIM; i += T::SIZE) { base[i] = make_double2(i == 0 ? 1.0 : 0.0, 0.0); fin[i] = base[i]; }
        T::sync();
        for (int f = lig; f < n_mats; f += T::SIZE) compose_matrix(g_mats[f], g_mat_gates, g_gates, trig, -1, make_double2(0, 0), u2 + 4 * f);
        T::sync();

        // sweep 1: the final base state (kept for the cross terms) and the base set's features A
        for (int ip = 0; ip < n_passes; ++ip) sv_pass3<Q, 1, false>(fin, fin, fin, fin, s_passes + ip, s_ops, u2, lig, -1, nullptr, -1, nullptr);
        // A = <psi|O|psi> through the final index map: the fork epilogue's own sums with phi = psi
        lc2_collect<Q>(fin, fin, red, lig, epi);
        T::sync();
        for (int k = lig; k < M3; k += T::SIZE) {
            double Bv = 0.0;
#pragma unroll
            for (int w = 0; w < NW; ++w) Bv += red[k * NW + w];
            featA[k] = (k < 2 * Q) ? 2.0 * Bv : Bv;
        }
        T::sync();
        if (live)
            for (int k = lig; k < M3; k += T::SIZE) out[(size_t)j * M3 + k] = featA[k];
        T::sync();

        // sweep 2: advance the base pass by pass; before pass ip runs, fork every parameter whose rotation lives in it
        for (int ip = 0; ip < n_passes; ++ip) {
            const int pb = pass_par_begin[ip], pe = pass_par_begin[ip + 1];
            const PassT* ps0 = s_passes + ip;
            for (int f0 = pb; f0 < pe; f0 += (PAIR ? 2 : 1)) {
                const int i0 = pass_params[f0];
                const int i1 = (PAIR && f0 + 1 < pe) ? pass_params[f0 + 1] : -1;
                // fork matrices: the parameter's rotation with its angle advanced by pi: (cos, sin)(theta/2 + pi/2) = (-sin, cos)(theta/2)
                // and the linear-combination coefficients cos / sin of half the two angle differences (once per fork, not per thread)
                for (int e = lig; e < 2; e += T::SIZE) {
                    const int i = e == 0 ? i0 : i1;
                    if (i >= 0) {
                        const int g = par_gate[i];
                        compose_matrix(g_mats[par_mat[i]], g_mat_gates, g_gates, trig, g, make_double2(-trig[g].y, trig[g].x), altm + 4 * e);
                        const dqgp_gate gt = g_gates[g];
                        const double th0 = gate_angle(gt, Pm[i], x, acx);
                        sincos(0.5 * (gate_angle(gt, Pm[(size_t)(1 + 2 * i) * P + i], x, acx) - th0), &coef[4 * e + 1], &coef[4 * e + 0]);
                        sincos(0.5 * (gate_angle(gt, Pm[(size_t)(2 + 2 * i) * P + i], x, acx) - th0), &coef[4 * e + 3], &coef[4 * e + 2]);
                    }
                }
                T::sync();
                if (PAIR && i1 >= 0) {
                    sv_pass3<Q, (PAIR ? 2 : 1), true>(base, base, scr0, scr1, ps0, s_ops, u2, lig, par_mat[i0], altm, par_mat[i1], altm + 4);
                    for (int kp = ip + 1; kp < n_passes; ++kp)
                        sv_pass3<Q, (PAIR ? 2 : 1), false>(scr0, scr1, scr0, scr1, s_passes + kp, s_ops, u2, lig, -1, nullptr, -1, nullptr);
                } else {
                    sv_pass3<Q, 1, true>(base, base, scr0, scr0, ps0, s_ops, u2, lig, par_mat[i0], altm, -1, nullptr);
                    for (int kp = ip + 1; kp < n_passes; ++kp)
                        sv_pass3<Q, 1, false>(scr0, scr0, scr0, scr0, s_passes + kp, s_ops, u2, lig, -1, nullptr, -1, nullptr);
                }
#pragma unroll 1
                for (int e = 0; e < 2; ++e) {
                    const int i = e == 0 ? i0 : i1;
                    if (i < 0) break;
                    lc2_emit<Q>(fin, e == 0 ? scr0 : scr1, featA, red, lig, live, coef[4 * e], coef[4 * e + 1], coef[4 * e + 2], coef[4 * e + 3],
                                        out + ((size_t)(1 + 2 * i) * n + j) * M3, out + ((size_t)(2 + 2 * i) * n + j) * M3, epi);
                }
            }
            sv_pass3<Q, 1, false>(base, base, base, base, ps0, s_ops, u2, lig, -1, nullptr, -1, nullptr);
        }
        T::sync();
    }
}

template <int Q>
static int launch_sv_lc2(const dqgp_circuit* c, const double* X, int n, const double* Pm, double* out, cudaStream_t st) {
    using T = SvTeam<Q>;
    constexpr bool PAIR = T::BLOCK;
    const int n_gates = (int)c->gates.size();
    const int n_passes = c->n_passes3, n_mats = (int)c->mats3.size();
    const int n_epi = (Q + 2) / 3;
    constexpr int M3 = 3 * Q, M3P = (M3 + 1) & ~1, NW = T::BLOCK ? T::SIZE / 32 : 1;
    const size_t team_bytes = sizeof(double2) * ((PAIR ? 4 : 3) * T::DIM + n_gates + 4 * n_mats + 8) + sizeof(double) * (((c->d + 1) & ~1) + 2 * M3 * NW + M3P + 8);
    const size_t fixed = ((sizeof(SvOp) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvPass3) * (n_passes + n_epi) + 15) & ~size_t(15));
    int warps = T::BLOCK ? T::SIZE / 32 : 4;
    if (!T::BLOCK) {
        // CTA size that keeps the most warps resident under the shared-memory limit
        int best = 0;
        for (int w = 4; w >= 1; --w) {
            const size_t bytes = fixed + team_bytes * w * T::PER_WARP + 1024;
            const int resident = bytes <= 228 * 1024 ? (int)((228 * 1024) / bytes) * w : 0;
            if (resident > best) { best = resident; warps = w; }
        }
    }
    const int teams = T::BLOCK ? 1 : warps * T::PER_WARP;
    const size_t smem = fixed + team_bytes * teams;
    if (smem > 227 * 1024) return 1;          // caller falls back to the one-fork kernel
    auto kern = statevec_lc2_kernel<Q>;
    DQGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    DQGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
    if (per_sm < 1) per_sm = 1;
    long long blocks = ((long long)n + teams - 1) / teams;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) return 0;
    kern<<<(unsigned)blocks, warps * 32, smem, st>>>(c->d_gates, n_gates, c->d_passes3, n_passes, c->d_ops3, c->d_mats3, n_mats, c->d_mat_gates3,
                                                    c->d_share3, c->d, c->P, c->uses_acos ? 1 : 0, X, n, Pm, out);
    DQGP_LAUNCH_CHECK("statevec_lc2_kernel");
    return 0;
}

template <int Q, bool WANT_STATES>
static int launch_sv_shared(const dqgp_circuit* c, const double* X, int n, const double* Pm, double* out, cudaStream_t st) {
    using T = SvTeam<Q>;
    const int n_gates = (int)c->gates.size(), n_passes = (int)c->passes.size();
    const int n_mats = (int)c->mats.size(), n_mat_gates = (int)c->mat_gates.size();
    const int n_share = 2 * c->P + n_passes + 1 + c->P;
    const size_t fixed = ((sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvPass) * n_passes + 15) & ~size_t(15)) +
                         ((sizeof(SvOp) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15)) +
                         ((sizeof(int) * n_share + 15) & ~size_t(15));
    // linear-combination form (statevec_lc_kernel) unless its third copy of the state does not fit in shared memory (q = 12 with a long
    // gate list) or DQGP_SV_NO_LC is set: a test hook, the only way to reach the two-fork kernel (statevec_shared_kernel) at small q
    bool use_lc = getenv("DQGP_SV_NO_LC") == nullptr;
    // lc2 (fused epilogue, halving reductions; two forks per pass where a CTA owns the state) for circuits with the CX-free plan (no CRZ
    // in the circuit, so every parameter sits on a rotation: yz_cx, kyriienko): CX gates cost nothing and the pass loop shrinks to fused
    // 2x2 unitaries.  Config 5's shard 60 -> 36 ms, config 4's 3.9 -> 3.1 ms.  Circuits with a CRZ take statevec_lc_kernel below.
    if (!WANT_STATES && Q >= 3 && use_lc && c->has_plan3) {
        const int rc = launch_sv_lc2<(Q >= 3 ? Q : 3)>(c, X, n, Pm, out, st);
        if (rc <= 0) return rc;          // 1 = does not fit in shared memory: the one-fork kernel below
    }
    auto team_size = [&](bool lc) {
        return sizeof(double2) * ((lc ? 3 : 2) * T::DIM + n_gates + 4 * n_mats + 4 * T::SLOTS) +
               sizeof(double) * (((c->d + 1) & ~1) + (T::BLOCK ? 9 * (T::SIZE / 32) + 1 : 0) + (lc ? 3 * ((3 * Q + 1) & ~1) : 0));
    };
    if (use_lc && T::BLOCK && fixed + team_size(true) > 227 * 1024) use_lc = false;
    const size_t team_bytes = team_size(use_lc);
    int warps = T::BLOCK ? T::SIZE / 32 : 4;
    int teams = T::BLOCK ? 1 : warps * T::PER_WARP;
    while (!T::BLOCK && warps > 1 && fixed + team_bytes * teams > 100 * 1024) { warps >>= 1; teams = warps * T::PER_WARP; }
    const size_t smem = fixed + team_bytes * teams;
    DQGP_REQUIRE(smem <= 227 * 1024, "statevector kernel needs %zu bytes of shared memory (q=%d, %d gates)", smem, Q, n_gates);
    auto lc_kern = statevec_lc_kernel<Q, WANT_STATES, false>;
    auto fork_kern = statevec_shared_kernel<Q, WANT_STATES>;
    int per_sm = 0;
    if (use_lc) {
        DQGP_CUDA(cudaFuncSetAttribute(lc_kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DQGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lc_kern, warps * 32, smem));
    } else {
        DQGP_CUDA(cudaFuncSetAttribute(fork_kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DQGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fork_kern, warps * 32, smem));
    }
    if (per_sm < 1) per_sm = 1;
    long long blocks = ((long long)n + teams - 1) / teams;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) return 0;
    if (use_lc)
        lc_kern<<<(unsigned)blocks, warps * 32, smem, st>>>(c->d_gates, n_gates, c->d_passes, n_passes, c->d_ops, c->d_mats, n_mats, c->d_mat_gates,
                                                            n_mat_gates, c->d_share, c->d, c->P, c->uses_acos ? 1 : 0, X, n, Pm, out, nullptr);
    else
        fork_kern<<<(unsigned)blocks, warps * 32, smem, st>>>(c->d_gates, n_gates, c->d_passes, n_passes, c->d_ops, c->d_mats, n_mats,
                                                              c->d_mat_gates, n_mat_gates, c->d_share, c->d, c->P, c->uses_acos ? 1 : 0, X, n, Pm, out);
    DQGP_LAUNCH_CHECK("statevec_shared_kernel");
    return 0;
}

template <int Q, bool WANT_STATES>
static int launch_sv_block(const dqgp_circuit* c, const double* X, int n, const double* Pm, int S, double* out, cudaStream_t st) {
    constexpr int DIM = 1 << Q, TEAM = DIM >> 3;
    const int n_gates = (int)c->gates.size(), n_passes = (int)c->passes.size();
    const int n_mats = (int)c->mats.size(), n_mat_gates = (int)c->mat_gates.size();
    const size_t fixed = ((sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvPass) * n_passes + 15) & ~size_t(15)) +
                         ((sizeof(SvOp) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15));
    const size_t smem = fixed + sizeof(double2) * (DIM + n_gates + 4 * n_mats) + sizeof(double) * (((c->d + 1) & ~1) + 9 * (TEAM / 32));
    DQGP_REQUIRE(smem <= 227 * 1024, "statevector kernel needs %zu bytes of shared memory (q=%d, %d gates)", smem, Q, n_gates);
    auto kern = statevec_block_kernel<Q, WANT_STATES>;
    DQGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    DQGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TEAM, smem));
    if (per_sm < 1) per_sm = 1;
    long long blocks = (long long)S * n;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) return 0;
    kern<<<(unsigned)blocks, TEAM, smem, st>>>(c->d_gates, n_gates, c->d_passes, n_passes, c->d_ops, c->d_mats, n_mats, c->d_mat_gates,
                                              n_mat_gates, c->d, c->P, c->uses_acos ? 1 : 0, X, n, Pm, S, out);
    DQGP_LAUNCH_CHECK("statevec_block_kernel");
    return 0;
}

template <int Q, bool WANT_STATES>
static int launch_sv(const dqgp_circuit* c, const double* X, int n, const double* Pm, int S, double* out, cudaStream_t st) {
    using G = SvGeom<Q>;
    const int n_gates = (int)c->gates.size(), n_passes = (int)c->passes.size();
    const size_t gate_bytes = (sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15);
    const size_t pass_bytes = (sizeof(SvPass) * n_passes + 15) & ~size_t(15);
    const size_t op_bytes = (sizeof(SvOp) * n_gates + 15) & ~size_t(15);
    const int n_mats = (int)c->mats.size(), n_mat_gates = (int)c->mat_gates.size();
    const size_t mat_bytes = (sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15);
    const size_t fixed = gate_bytes + pass_bytes + op_bytes + mat_bytes;
    const size_t state_bytes = sizeof(double2) * (G::DIM + n_gates + 4 * n_mats) + ((sizeof(double) * c->d + 15) & ~size_t(15));
    int warps = 4;
    while (warps > 1 && fixed + state_bytes * G::SPW * warps > 100 * 1024) warps >>= 1;
    const size_t smem = fixed + state_bytes * G::SPW * warps;
    DQGP_REQUIRE(smem <= 227 * 1024, "statevector kernel needs %zu bytes of shared memory (q=%d, %d gates)", smem, Q, n_gates);
    auto kern = statevec_kernel<Q, WANT_STATES>;
    DQGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    DQGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
    if (per_sm < 1) per_sm = 1;
    const long long total = (long long)S * n;
    const long long n_groups = (total + G::SPW - 1) / G::SPW;
    long long blocks = (n_groups + warps - 1) / warps;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) return 0;
    kern<<<(unsigned)blocks, warps * 32, smem, st>>>(c->d_gates, n_gates, c->d_passes, n_passes, c->d_ops, c->d_mats, n_mats,
                                                     c->d_mat_gates, n_mat_gates, c->d, c->P, c->uses_acos ? 1 : 0, X, n, Pm, S, out);
    DQGP_LAUNCH_CHECK("statevec_kernel");
    return 0;
}

template <int Q, bool WANT_STATES>
static int launch_sv_jac(const dqgp_circuit* c, const double* X, int n, const double* p, double* F, double* J, cudaStream_t st) {
    using T = SvTeam<Q>;
    const int n_gates = (int)c->gates.size(), n_passes = (int)c->passes.size();
    const int n_mats = (int)c->mats.size(), n_mat_gates = (int)c->mat_gates.size();
    const int n_share = 2 * c->P + n_passes + 1 + c->P;
    const size_t fixed = ((sizeof(dqgp_gate) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvPass) * n_passes + 15) & ~size_t(15)) +
                         ((sizeof(SvOp) * n_gates + 15) & ~size_t(15)) + ((sizeof(SvMat) * n_mats + sizeof(int) * n_mat_gates + 15) & ~size_t(15)) +
                         ((sizeof(int) * n_share + 15) & ~size_t(15));
    const size_t team_bytes = sizeof(double2) * (3 * T::DIM + n_gates + 4 * n_mats + 4 * T::SLOTS) +
                              sizeof(double) * (((c->d + 1) & ~1) + (T::BLOCK ? 9 * (T::SIZE / 32) + 1 : 0) + 3 * ((3 * Q + 1) & ~1));
    int warps = T::BLOCK ? T::SIZE / 32 : 4;
    int teams = T::BLOCK ? 1 : warps * T::PER_WARP;
    while (!T::BLOCK && warps > 1 && fixed + team_bytes * teams > 100 * 1024) { warps >>= 1; teams = warps * T::PER_WARP; }
    const size_t smem = fixed + team_bytes * teams;
    DQGP_REQUIRE(smem <= 227 * 1024, "statevector kernel needs %zu bytes of shared memory (q=%d, %d gates)", smem, Q, n_gates);
    auto kern = statevec_lc_kernel<Q, WANT_STATES, true>;
    DQGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    DQGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
    if (per_sm < 1) per_sm = 1;
    long long blocks = ((long long)n + teams - 1) / teams;
    const long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) return 0;
    kern<<<(unsigned)blocks, warps * 32, smem, st>>>(c->d_gates, n_gates, c->d_passes, n_passes, c->d_ops, c->d_mats, n_mats, c->d_mat_gates,
                                                     n_mat_gates, c->d_share, c->d, c->P, c->uses_acos ? 1 : 0, X, n, p, F, J);
    DQGP_LAUNCH_CHECK("statevec_lc_kernel (jacobian)");
    return 0;
}

template <bool WANT_STATES>
static int dispatch_sv(const dqgp_circuit* c, const double* X, int n, const double* Pm, int S, double* out, void* stream) {
    DQGP_REQUIRE(n >= 0 && S >= 0, "statevector: negative size");
    if (n == 0 || S == 0) return 0;      // empty input: nothing to do (pointers may be NULL)
    DQGP_REQUIRE(c && X && Pm && out, "statevector: NULL argument");
    int rc = circuit_on_device(c);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    switch (c->q) {
#define DQGP_SV_CASE(QQ) case QQ: return launch_sv<QQ, WANT_STATES>(c, X, n, Pm, S, out, st);
        DQGP_SV_CASE(1) DQGP_SV_CASE(2) DQGP_SV_CASE(3) DQGP_SV_CASE(4) DQGP_SV_CASE(5) DQGP_SV_CASE(6)
        DQGP_SV_CASE(7) DQGP_SV_CASE(8)
#undef DQGP_SV_CASE
#define DQGP_SV_CASE(QQ) case QQ: return launch_sv_block<QQ, WANT_STATES>(c, X, n, Pm, S, out, st);
        DQGP_SV_CASE(9) DQGP_SV_CASE(10) DQGP_SV_CASE(11) DQGP_SV_CASE(12)
#undef DQGP_SV_CASE
    }
    set_error("statevector: unsupported qubit count %d", c->q);
    return -1;
}

template <bool WANT_STATES>
static int dispatch_sv_shared(const dqgp_circuit* c, const double* X, int n, const double* Pm, int P, double* out, void* stream) {
    DQGP_REQUIRE(n >= 0, "statevector: negative size");
    if (n == 0) return 0;
    DQGP_REQUIRE(c && X && Pm && out, "statevector: NULL argument");
    DQGP_REQUIRE(P == c->P, "statevector: circuit has %d parameters, got %d", c->P, P);
    // prefix sharing parallelises over samples only: with few samples (or a parameter feeding several gates) the
    // per-set kernel, which parallelises over samples x sets, fills the machine better
    const long long teams = c->q >= 9 ? n : (long long)n * (c->q > 3 ? (1 << (c->q - 3)) : 1) / 32;
    // DQGP_SV_FORCE_SHARED: a test hook that reaches the prefix-sharing kernels at small n
    if (!c->shareable || (teams < (c->q >= 9 ? 600 : 1200) && getenv("DQGP_SV_FORCE_SHARED") == nullptr))
        return WANT_STATES ? dqgp_states(c, X, n, Pm, 2 * P + 1, out, stream) : dqgp_features(c, X, n, Pm, 2 * P + 1, out, stream);
    int rc = circuit_on_device(c);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    switch (c->q) {
#define DQGP_SV_CASE(QQ) case QQ: return launch_sv_shared<QQ, WANT_STATES>(c, X, n, Pm, out, st);
        DQGP_SV_CASE(1) DQGP_SV_CASE(2) DQGP_SV_CASE(3) DQGP_SV_CASE(4) DQGP_SV_CASE(5) DQGP_SV_CASE(6)
        DQGP_SV_CASE(7) DQGP_SV_CASE(8) DQGP_SV_CASE(9) DQGP_SV_CASE(10) DQGP_SV_CASE(11) DQGP_SV_CASE(12)
#undef DQGP_SV_CASE
    }
    set_error("statevector: unsupported qubit count %d", c->q);
    return -1;
}


template <bool WANT_STATES>
static int dispatch_sv_jac(const dqgp_circuit* c, const double* X, int n, const double* p, double* out, double* jac, void* stream) {
    DQGP_REQUIRE(n >= 0, "jacobian: negative size");
    if (n == 0) return 0;
    DQGP_REQUIRE(c && X && p && out && jac, "jacobian: NULL argument");
    DQGP_REQUIRE(c->shareable, "jacobian: a parameter of this circuit feeds several gates");
    int rc = circuit_on_device(c);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    switch (c->q) {
#define DQGP_SV_CASE(QQ) case QQ: return launch_sv_jac<QQ, WANT_STATES>(c, X, n, p, out, jac, st);
        DQGP_SV_CASE(1) DQGP_SV_CASE(2) DQGP_SV_CASE(3) DQGP_SV_CASE(4) DQGP_SV_CASE(5) DQGP_SV_CASE(6)
        DQGP_SV_CASE(7) DQGP_SV_CASE(8) DQGP_SV_CASE(9) DQGP_SV_CASE(10) DQGP_SV_CASE(11) DQGP_SV_CASE(12)
#undef DQGP_SV_CASE
    }
    set_error("statevector: unsupported qubit count %d", c->q);
    return -1;
}

}  // namespace dqgp

// This file is compiled five times (build.py: -DDQGP_SV_PART=1..5), one group of entry points per object, so the twelve qubit
// counts x kernel variants compile in parallel (one translation unit took 2.6 minutes).
#ifndef DQGP_SV_PART
#define DQGP_SV_PART 0      // 0 = everything in one object
#endif
extern "C" {
#if DQGP_SV_PART == 0 || DQGP_SV_PART == 5
int dqgp_features_jacobian(const dqgp_circuit* c, const double* d_X, int n, const double* d_p, double* d_F, double* d_J, void* stream) {
    return dqgp::dispatch_sv_jac<false>(c, d_X, n, d_p, d_F, d_J, stream);
}
int dqgp_states_jacobian(const dqgp_circuit* c, const double* d_X, int n, const double* d_p, double* d_Psi, double* d_D, void* stream) {
    return dqgp::dispatch_sv_jac<true>(c, d_X, n, d_p, d_Psi, d_D, stream);
}
#endif
#if DQGP_SV_PART == 0 || DQGP_SV_PART == 3
int dqgp_features_shifted(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int P, double* d_F, void* stream) {
    return dqgp::dispatch_sv_shared<false>(c, d_X, n, d_Pm, P, d_F, stream);
}
#endif
#if DQGP_SV_PART == 0 || DQGP_SV_PART == 4
int dqgp_states_shifted(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int P, double* d_Psi, void* stream) {
    return dqgp::dispatch_sv_shared<true>(c, d_X, n, d_Pm, P, d_Psi, stream);
}
#endif
#if DQGP_SV_PART == 0 || DQGP_SV_PART == 1
int dqgp_features(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int S, double* d_F, void* stream) {
    return dqgp::dispatch_sv<false>(c, d_X, n, d_Pm, S, d_F, stream);
}
#endif
#if DQGP_SV_PART == 0 || DQGP_SV_PART == 2
int dqgp_states(const dqgp_circuit* c, const double* d_X, int n, const double* d_Pm, int S, double* d_Psi, void* stream) {
    return dqgp::dispatch_sv<true>(c, d_X, n, d_Pm, S, d_Psi, stream);
}
#endif
}
