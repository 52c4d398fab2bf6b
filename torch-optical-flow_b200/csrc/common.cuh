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

// One tap of the correlation lookup's window (CorrBlock.__call__ + bilinear_sampler, methods/raft/model/corr.py:56-77,
// utils.py:64-80).  Bit-exactness contract (SURVEY.md 8c): the fp32 coordinate sequence is replayed operation by
// operation with round-to-nearest intrinsics so nvcc cannot contract it, and the floor indices and validity masks match
// the reference bit for bit.  `center` is the level-scaled coordinate c = coord / 2^l (corr.py:68, exact):
//     x  = c + (t - r)                       (corr.py:70; window TRANSPOSED: the x taps move the output channel's i)
//     g  = 2*x/(size-1) - 1                  (utils.py:70-71)
//     ix = ((g + 1) * 0.5) * (size-1)        (ATen GridSampler.h:30, align_corners=True; (g+1)/2 == (g+1)*0.5 exactly)
//     fl = floor(ix); valid = -1 < g < 1     (utils.py:77)
// Every lookup kernel (forward, backward, on-demand) takes its taps from here; each decides what an out-of-guard tap
// contributes.
struct LookupTap {
    float fl;          // floor of the un-normalised coordinate (what the idx output reports)
    float w0, w1;      // bilinear weights of columns fl and fl + 1
    bool valid;        // utils.py:77 predicate
    bool in_guard;     // fl in [-32768, 70000]: (int)fl is exact, and fp32 resolves ix to better than 1/64.  Level sizes
                       // are <= 65536 and a window spans 2r+1 <= 9 taps, so a tap outside the guard means every tap of
                       // its axis is outside the image.  NaN / inf coordinates are outside it.
};
__device__ __forceinline__ LookupTap lookup_tap(float center, int t, int radius, int size) {
    const float pos = __fadd_rn(center, (float)(t - radius));
    const float sm1 = (float)(size - 1);
    const float g = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, pos), sm1), 1.0f);
    const float ic = __fmul_rn(__fmul_rn(__fadd_rn(g, 1.0f), 0.5f), sm1);
    LookupTap tp;
    tp.fl = floorf(ic);
    tp.w1 = __fsub_rn(ic, tp.fl);
    tp.w0 = __fsub_rn(__fadd_rn(tp.fl, 1.0f), ic);
    tp.valid = (g > -1.0f) && (g < 1.0f);
    tp.in_guard = tp.fl >= -32768.0f && tp.fl <= 70000.0f;
    return tp;
}
constexpr int TAP_FAR = -1000000;   // floor index given to an out-of-guard tap whose weights are zeroed

// Warp-level window of the generic and the on-demand lookup: one warp handles one (query, level).  Lane t < 16 holds
// x tap t, lane 16 + t holds y tap t (taps t >= 2r+1 are computed and unused); the samples are read from a PD x PD
// shared-memory patch that covers every tap.
constexpr int PD = 12;       // patch rows / cols: 2r+3 <= 11 taps, plus one when the x origin is rounded down to even
constexpr int MAX_D = 9;     // 2*radius+1, radius <= 4

struct WarpWindow {
    float fl;                // this lane's tap: floor index
    int valid;               //   utils.py:77 predicate
    int i0;                  //   floor index, TAP_FAR outside the guard
    float w0, w1;            //   weights, zero outside the guard
    int px0, py0;            // patch origin: first x (EVEN_X: rounded down to even) and y tap
    int cols, rows;          // patch extent covering every tap and its + 1 neighbour
    bool patch_ok;           // warp-uniform: the extent fits PD x PD
};

// Step 1: this lane's tap and the patch geometry.  cx0, cy0: the query's level-0 coordinates; inv = 1 / 2^l.
template <bool EVEN_X>
__device__ __forceinline__ WarpWindow warp_window(float cx0, float cy0, float inv, int radius, int Wl, int Hl, int lane) {
    const int t = lane & 15, isy = lane >> 4, D = 2 * radius + 1;
    const LookupTap tp = lookup_tap(__fmul_rn(isy ? cy0 : cx0, inv), t, radius, isy ? Hl : Wl);
    WarpWindow w;
    w.fl = tp.fl;
    w.valid = tp.valid;
    w.i0 = tp.in_guard ? (int)tp.fl : TAP_FAR;
    w.w0 = tp.w0;
    w.w1 = tp.w1;
    if (w.i0 == TAP_FAR) { w.w0 = 0.0f; w.w1 = 0.0f; }
    const int x_first = __shfl_sync(0xffffffffu, w.i0, 0), x_last = __shfl_sync(0xffffffffu, w.i0, D - 1);
    const int y_first = __shfl_sync(0xffffffffu, w.i0, 16), y_last = __shfl_sync(0xffffffffu, w.i0, 16 + D - 1);
    w.px0 = EVEN_X ? (x_first & ~1) : x_first;
    w.py0 = y_first;
    w.cols = x_last + 2 - w.px0;
    w.rows = y_last + 2 - w.py0;
    w.patch_ok = w.cols <= PD && w.rows <= PD && w.cols > 0 && w.rows > 0;
    return w;
}

__device__ __forceinline__ float bilinear(float v00, float v01, float v10, float v11, float wx0, float wx1, float wy0,
                                          float wy1) {
    float acc = __fmul_rn(v00, __fmul_rn(wx0, wy0));
    acc = __fmaf_rn(v01, __fmul_rn(wx1, wy0), acc);
    acc = __fmaf_rn(v10, __fmul_rn(wx0, wy1), acc);
    return __fmaf_rn(v11, __fmul_rn(wx1, wy1), acc);
}

// Step 3: the (2r+1)^2 bilinear samples, 3 per lane, each tap's floor index and weights fetched from its owning lane.
// Sample k = i*D + j (i moves x: corr.py:64-70) is read from the patch when w.patch_ok, else it is
// outside(x0, y0, wx0, wx1, wy0, wy1); emit(k, i, j, value) stores it.
template <typename Outside, typename Emit>
__device__ __forceinline__ void warp_window_samples(const WarpWindow& w, const float* patch, int radius, int lane,
                                                    Outside outside, Emit emit) {
    const int D = 2 * radius + 1, DD = D * D;
#pragma unroll
    for (int kk = 0; kk < (MAX_D * MAX_D + 31) / 32; ++kk) {
        const int k = kk * 32 + lane;
        const bool active = k < DD;
        const int i = active ? k / D : 0, j = active ? k - (k / D) * D : 0;
        const int x0 = __shfl_sync(0xffffffffu, w.i0, i), y0 = __shfl_sync(0xffffffffu, w.i0, 16 + j);
        const float wx0 = __shfl_sync(0xffffffffu, w.w0, i), wx1 = __shfl_sync(0xffffffffu, w.w1, i);
        const float wy0 = __shfl_sync(0xffffffffu, w.w0, 16 + j), wy1 = __shfl_sync(0xffffffffu, w.w1, 16 + j);
        if (!active) continue;
        float acc;
        if (w.patch_ok) {
            const float* s = patch + (y0 - w.py0) * PD + (x0 - w.px0);
            acc = bilinear(s[0], s[1], s[PD], s[PD + 1], wx0, wx1, wy0, wy1);
        } else {
            acc = outside(x0, y0, wx0, wx1, wy0, wy1);
        }
        emit(k, i, j, acc);
    }
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
// half-word `hi` (0: low, 1: high) of a 4-byte word of two bf16 / fp16 elements -> fp32
template <typename T> __device__ __forceinline__ float widen16(unsigned wd, int hi);
template <> __device__ __forceinline__ float widen16<__nv_bfloat16>(unsigned wd, int hi) {
    return __uint_as_float(hi ? (wd & 0xffff0000u) : (wd << 16));
}
template <> __device__ __forceinline__ float widen16<__half>(unsigned wd, int hi) {
    return __half2float(__ushort_as_half((unsigned short)(hi ? (wd >> 16) : (wd & 0xffffu))));
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

// An ofb_pyramid's level geometry as the lookup kernels receive it (strides in elements, unused levels zeroed)
struct PyramidLevels {
    void* base[OFB_MAX_LEVELS];
    long long q_stride[OFB_MAX_LEVELS];
    int pitch[OFB_MAX_LEVELS];
    int lh[OFB_MAX_LEVELS];
    int lw[OFB_MAX_LEVELS];
};

// Copies pyr's levels into lv and checks them: 1 .. OFB_MAX_LEVELS levels, each with a base pointer, a positive size
// and a row pitch no smaller than its width.
inline int unpack_levels(const ofb_pyramid& pyr, PyramidLevels& lv) {
    if (pyr.levels < 1 || pyr.levels > OFB_MAX_LEVELS) return OFB_EINVAL;
    for (int l = 0; l < OFB_MAX_LEVELS; ++l) {
        const bool on = l < pyr.levels;
        lv.base[l] = on ? pyr.base[l] : nullptr;
        lv.q_stride[l] = on ? pyr.q_stride[l] : 0;
        lv.pitch[l] = on ? pyr.row_pitch[l] : 0;
        lv.lh[l] = on ? pyr.lvl_h[l] : 0;
        lv.lw[l] = on ? pyr.lvl_w[l] : 0;
        if (on && (!lv.base[l] || lv.lh[l] <= 0 || lv.lw[l] <= 0 || lv.pitch[l] < lv.lw[l])) return OFB_EINVAL;
    }
    return OFB_OK;
}

}  // namespace ofb
