// Shared internals of libdqgp (sm_100a).  Not part of the public ABI (see include/dqgp.h).
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <cstdint>
#include <vector>
#include "../../include/dqgp.h"

struct dqgp_circuit;

namespace dqgp {

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define DQGP_CUDA(call)                                                     \
    do {                                                                    \
        cudaError_t e__ = (call);                                           \
        if (e__ != cudaSuccess) return ::dqgp::cuda_fail(e__, #call);       \
    } while (0)
#define DQGP_LAUNCH_CHECK(name)                                             \
    do {                                                                    \
        cudaError_t e__ = cudaGetLastError();                               \
        if (e__ != cudaSuccess) return ::dqgp::cuda_fail(e__, name);        \
    } while (0)
#define DQGP_REQUIRE(cond, ...)                                             \
    do {                                                                    \
        if (!(cond)) { ::dqgp::set_error(__VA_ARGS__); return -1; }         \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Raise KERNEL's dynamic shared memory limit to `bytes`.  The attribute belongs to the device, so it is set once per device
// (on every call for a device id of 64 or more).
template <auto KERNEL>
int set_max_dynamic_smem(int bytes) {
    static bool done[64] = {false};
    int dev = 0;
    DQGP_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && done[dev]) return 0;
    DQGP_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    if (dev >= 0 && dev < 64) done[dev] = true;
    return 0;
}

int sm_count();
int circuit_on_device(const dqgp_circuit* c);  // uploads the gate program on first use

constexpr int MAX_QUBITS = 12;

// fp64 mma.sync m8n8k4: A 8x4 (row), B 4x8 (col), C 8x8.  Fragment ownership (lane = 4*g + t):
//   a = A[g][t], b = B[t][g], c0 = C[g][2t], c1 = C[g][2t+1].   SASS: DMMA.8x8x4
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }

// ---- 1-D bulk async copies (the TMA engine without a tensor map: cp.async.bulk, SASS UBLKCP) + mbarrier completion ----------
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    const unsigned a = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(a), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    const unsigned a = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    const unsigned a = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    unsigned ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}
// bytes: multiple of 16; smem and gmem 16-byte aligned
__device__ __forceinline__ void bulk_copy_g2s(void* smem, const void* gmem, unsigned bytes, unsigned long long* bar) {
    const unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    const unsigned b = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(d), "l"(gmem), "r"(bytes), "r"(b) : "memory");
}
// one box of a 3-D tensor map (TMA proper, SASS UTMALDG): coordinates innermost first; elements outside the tensor arrive as zeros
// and count towards the transaction bytes.  smem 128-byte aligned; `tmap` = address of a __grid_constant__ CUtensorMap parameter.
__device__ __forceinline__ void tensor_copy_3d_g2s(void* smem, const void* tmap, int c0, int c1, int c2, unsigned long long* bar) {
    const unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    const unsigned b = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n"
                 ::"r"(d), "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(b) : "memory");
}
__device__ __forceinline__ void tensor_copy_2d_g2s(void* smem, const void* tmap, int c0, int c1, unsigned long long* bar) {
    const unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    const unsigned b = static_cast<unsigned>(__cvta_generic_to_shared(bar));
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
                 ::"r"(d), "l"(tmap), "r"(c0), "r"(c1), "r"(b) : "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Fixed-order sum over a block of 256 threads, each holding `acc` (its strided partial sum): a halving tree through shared memory,
// so the result is bit-reproducible run to run.  Every thread gets the sum; call it from all 256 threads.
__device__ __forceinline__ double block_sum_256(double acc) {
    __shared__ double s[256];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    return s[0];
}

}  // namespace dqgp

// Execution plan of the statevector kernel: the gate list regrouped into passes over <= 3 "block" qubits.
// Within a pass every op's TARGET is a block qubit, so a lane holding the 2^b amplitudes of one block in
// registers applies all of them back to back; controls may be any qubit (read-only index bits).  Runs of
// single-qubit gates on one qubit are fused into one general 2x2 unitary (SV_U2) whose matrix is composed
// per state from the cos/sin table (its constituents are mat_gates[g_begin, g_end) in application order).
enum { SV_U2 = 0, SV_CX = 1, SV_CRZ = 2 };
struct SvOp {
    int8_t kind;    // SV_*
    int8_t lbit;    // target as a local bit of the pass block (0..2)
    int8_t cloc;    // control as a local bit of the block, or -1
    int8_t cq;      // control as a global qubit (when not in the block), or -1
    int16_t idx;    // SV_U2: matrix index; SV_CRZ: original gate index (selects the cos/sin pair)
    int16_t pad;
};
struct SvMat {
    int g_begin, g_end;   // range in mat_gates
};
struct SvPass {
    int nq;         // block size 1..3
    int q[3];       // block qubits, ascending
    int op_begin, op_end;
    // ops [op_begin, lead_end) and [trail_begin, op_end) are CX gates whose control lies OUTSIDE the block: a thread's groups
    // see a fixed control bit, so these are XORs of the target bit into the LOAD / STORE address of the pass (statevec_lc2_kernel);
    // kernels that ignore the two fields execute them as ordinary ops
    int lead_end, trail_begin;
};

// Plan of the CX-free simulator (statevec_lc2_kernel): circuits made of 1-qubit gates and CX only.  A CX is never
// executed: amplitudes stay where they are and the map from LOGICAL basis index x to PHYSICAL position p = M x (M over GF(2), one
// column mask per logical qubit) absorbs it - CX(c -> t) replaces the control's mask m_c by m_c ^ m_t.  A pass applies the fused 2x2
// unitaries of <= 3 logical qubits: a thread owns the coset of span{bm} selected by the bits of its index (bit i <-> rest[i]),
// register j holds the amplitude whose logical block bits are j, at position p0 ^ comb(j).  Entries past the real passes describe
// the Pauli-feature epilogue's qubit groups under the FINAL map.
struct SvPass3 {
    int nq;                              // block size 1..3
    int bm[3];                           // masks of the block's logical qubits (register bit l <-> bm[l])
    int rest[dqgp::MAX_QUBITS];          // masks of the other logical qubits, ascending logical index: coset bit i <-> rest[i]
    int op_begin, op_end;                // ops3 range (SV_U2 only: lbit, idx = fused matrix)
};

struct dqgp_circuit {
    int encoding, q, d, layers, P;
    bool uses_acos;
    std::vector<dqgp_gate> gates;  // host copy
    std::vector<SvPass> passes;
    std::vector<SvOp> ops;
    std::vector<SvMat> mats;
    std::vector<int> mat_gates;
    // prefix sharing across the 2P+1 central-difference sets: where each parameter enters the plan
    bool shareable;                 // every parameter is used by exactly one gate
    std::vector<int> par_gate;      // [P] gate using parameter i
    std::vector<int> par_mat;       // [P] fused matrix containing that gate, or -1 (CRZ)
    std::vector<int> pass_par_begin;// [n_passes+1] ranges into pass_params
    std::vector<int> pass_params;   // [P] parameters ordered by the pass their op belongs to
    // CX-free plan (has_plan3: no CRZ in the circuit, every parameter on one rotation)
    bool has_plan3;
    int n_passes3;                  // real passes; passes3 holds n_passes3 + ceil(q/3) entries (epilogue groups at the end)
    std::vector<SvPass3> passes3;
    std::vector<SvOp> ops3;
    std::vector<SvMat> mats3;
    std::vector<int> mat_gates3, par_mat3, pass_par_begin3, pass_params3;
    SvPass3* d_passes3;
    SvOp* d_ops3;
    SvMat* d_mats3;
    int* d_mat_gates3;
    int* d_share3;                  // par_gate | par_mat3 | pass_par_begin3 | pass_params3
    int* d_share;                   // device copy: par_gate | par_mat | pass_par_begin | pass_params
    dqgp_gate* d_gates;            // device copies
    SvPass* d_passes;
    SvOp* d_ops;
    SvMat* d_mats;
    int* d_mat_gates;
    int device;
};
