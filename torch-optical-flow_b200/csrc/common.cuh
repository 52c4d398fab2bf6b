// common.cuh -- shared device helpers for the ofb200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "../../include/ofb200.h"

#define OFB_API extern "C" __attribute__((visibility("default")))

extern int64_t g_ofb_launches;  // api.cu

#define OFB_LAUNCH_CHECK()                         \
    do {                                           \
        __atomic_add_fetch(&g_ofb_launches, 1, __ATOMIC_RELAXED); \
        cudaError_t e__ = cudaGetLastError();      \
        if (e__ != cudaSuccess) return (int)e__;   \
    } while (0)

#define OFB_CUDA(...)  /* variadic: the call may contain template-argument commas */ \
    do {                                           \
        cudaError_t e__ = (__VA_ARGS__);           \
        if (e__ != cudaSuccess) return (int)e__;   \
    } while (0)

// Function attributes and the SM count belong to a device: cache them per device, so a process that drives several
// GPUs (not the one-process-per-GPU model of the bench, but legal for a library) configures each of them.
constexpr int OFB_MAX_DEVICES = 64;
static inline int ofb_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return (dev >= 0 && dev < OFB_MAX_DEVICES) ? dev : 0;
}

static inline int ofb_num_sms() {
    static int sms[OFB_MAX_DEVICES] = {0};
    const int dev = ofb_device();
    if (!sms[dev]) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        sms[dev] = n > 0 ? n : 148;
    }
    return sms[dev];
}

// Raises Kernel's dynamic shared-memory limit to `bytes`, the first time it is called on each device.
template <auto Kernel>
static inline cudaError_t ofb_smem_once(int bytes) {
    static bool configured[OFB_MAX_DEVICES] = {false};
    const int dev = ofb_device();
    if (!configured[dev]) {
        const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
        configured[dev] = true;
    }
    return cudaSuccess;
}

namespace ofb {

// torch.linspace(-1, 1, n)[i] in fp32: step = 2/(n-1); symmetric halves, one fused op each
// (same expression ATen's CPU and CUDA range factories evaluate; reference call sites
// optical_flow/operator/operator.py:49-50).
// a single-element linspace is its start value, -1 (torch.linspace(-1, 1, 1) == [-1])
__device__ __forceinline__ float linspace_m1_p1(int i, int n, float step) {
    return (i < n / 2 || n == 1) ? __fmaf_rn(step, (float)i, -1.0f) : __fmaf_rn(-step, (float)(n - 1 - i), 1.0f);
}
__host__ __device__ __forceinline__ float linspace_step(int n) { return n > 1 ? 2.0f / (float)(n - 1) : 0.0f; }

// grid_sample coordinate pipeline (ATen GridSampler.h:26-36,57-59,88-107,143-160).
template <bool AC>
__device__ __forceinline__ float unnormalize(float g, int size) {
    if (AC) return __fmul_rn(__fdiv_rn(__fadd_rn(g, 1.0f), 2.0f), (float)(size - 1));
    return __fmaf_rn(__fadd_rn(g, 1.0f), 0.5f * (float)size, -0.5f);
}
__device__ __forceinline__ float clip_coord(float x, int size) { return fminf((float)(size - 1), fmaxf(x, 0.0f)); }
__device__ __forceinline__ float reflect_coord(float in, int twice_low, int twice_high) {
    if (twice_low == twice_high) return 0.0f;
    float mn = (float)twice_low / 2.0f;
    float span = (float)(twice_high - twice_low) / 2.0f;
    in = fabsf(in - mn);
    float extra = fmodf(in, span);
    int flips = (int)floorf(in / span);
    return (flips % 2 == 0) ? (extra + mn) : (span - extra + mn);
}
template <int PAD, bool AC>
__device__ __forceinline__ float source_index(float g, int size) {
    float x = unnormalize<AC>(g, size);
    if (PAD == OFB_PAD_BORDER) {
        x = clip_coord(x, size);
    } else if (PAD == OFB_PAD_REFLECTION) {
        x = AC ? reflect_coord(x, 0, 2 * (size - 1)) : reflect_coord(x, -1, 2 * size - 1);
        x = clip_coord(x, size);
    }
    return x;
}

__device__ __forceinline__ float ld_nc(const float* p) { return __ldg(p); }

// input element -> fp32: feature maps and mask logits arrive in fp32, or in half precision from an autocast caller
__device__ __forceinline__ float ld_f32(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_f32(const __nv_bfloat16* p) {
    return __uint_as_float((unsigned)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}
__device__ __forceinline__ float ld_f32(const __half* p) {
    return __half2float(__ushort_as_half(__ldg(reinterpret_cast<const unsigned short*>(p))));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace ofb
