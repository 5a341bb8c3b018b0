// Host-only: the TMA tensor maps of the tcgen05 kernels.  cuTensorMapEncodeTiled is a driver entry point, resolved
// through the runtime at first use, so the library links no libcuda and loads on a machine without a GPU driver.
#include "common.cuh"

namespace triad {

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmapEncodeTiled get_encode_fn() {
    static PFN_tmapEncodeTiled fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = (PFN_tmapEncodeTiled)p;
    return fn;
}

int encode_tmap(CUtensorMap* map, CUtensorMapDataType type, const void* base, int rank, const cuuint64_t* dims,
                const cuuint64_t* strides, const cuuint32_t* box, Swizzle swizzle) {
    PFN_tmapEncodeTiled fn = get_encode_fn();
    if (!fn) return fail_msg(TRIAD_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(map, type, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE,
                          swizzle == Swizzle::k128B ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        const char* elt = type == CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 ? "bf16" : type == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? "fp32" : "uint8";
        char buf[96];
        snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled (%s) failed (CUresult %d)", elt, (int)r);
        return fail_msg(TRIAD_ERR_CUDA, buf);
    }
    return TRIAD_OK;
}

}  // namespace triad
