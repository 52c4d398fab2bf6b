// api.cu -- version / error strings / launch counter of libofb200.so, and the tensor-map encoder of the TMA kernels.
#include <cudaTypedefs.h>

#include "sm100.cuh"

int64_t g_ofb_launches = 0;

bool ofb::encode_tiled(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims,
                       const cuuint64_t* strides_bytes, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                       CUtensorMapL2promotion l2_promotion) {
    // the driver entry point is looked up once; a function-local static is initialised thread-safely
    static const PFN_cuTensorMapEncodeTiled_v12000 enc = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
                        qres == cudaDriverEntryPointSuccess;
        return ok ? reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p) : nullptr;
    }();
    if (!enc) return false;
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    return enc(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2_promotion, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

OFB_API int ofb_version(void) { return OFB_VERSION; }

OFB_API int64_t ofb_launch_count(void) { return __atomic_load_n(&g_ofb_launches, __ATOMIC_RELAXED); }

OFB_API const char* ofb_strerror(int code) {
    switch (code) {
        case OFB_OK: return "ok";
        case OFB_EINVAL: return "invalid argument (null pointer, negative size or unknown enum value)";
        case OFB_EUNSUPPORTED: return "request not supported by this kernel build";
        case OFB_EALIGN: return "pointer, pitch or stride not aligned as the kernel requires";
        case OFB_EDRIVER: return "cuTensorMapEncodeTiled unavailable or rejected the tensor map";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown ofb200 error";
}
