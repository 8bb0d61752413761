// Host side of the TMA tensor maps (cuTensorMapEncodeTiled through the runtime's driver entry point: libdqgp.so does not link libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

namespace dqgp {

// A = [sets][n][inner] doubles (row stride inner * 8 bytes, a multiple of 16) as a 3-D tensor map whose box is (1, box_rows, box_inner).
// box_inner may exceed `inner` and a box may hang over the last row: what lies outside the tensor arrives as zeros.
// false when the driver entry point is missing or refuses the map.
static inline bool make_rows_tensor_map(CUtensorMap* out, const double* base, int inner, int n, int sets, int box_inner, int box_rows) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    static bool looked = false;
    if (!looked) {
        looked = true;
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            encode = reinterpret_cast<EncodeFn>(fn);
        else
            cudaGetLastError();
    }
    if (!encode || (inner & 1) || (reinterpret_cast<uintptr_t>(base) & 15)) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)n, (cuuint64_t)sets};
    const cuuint64_t strides[2] = {(cuuint64_t)inner * sizeof(double), (cuuint64_t)n * inner * sizeof(double)};      // bytes, dimensions 1 and 2
    const cuuint32_t box[3] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// A row-major matrix view [outer][inner] doubles with row stride ld (doubles, even) as a 2-D tensor map with a (box_outer, box_inner) box.
static inline bool make_matrix_tensor_map(CUtensorMap* out, const double* base, long long inner, long long outer, long long ld, int box_inner,
                                          int box_outer) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    static bool looked = false;
    if (!looked) {
        looked = true;
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            encode = reinterpret_cast<EncodeFn>(fn);
        else
            cudaGetLastError();
    }
    if (!encode || (ld & 1) || (reinterpret_cast<uintptr_t>(base) & 15)) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(double)};
    const cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
    const cuuint32_t estr[2] = {1u, 1u};
    return encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace dqgp
