// common.cuh -- shared device helpers for the ofb200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include <climits>
#include <type_traits>

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

// Returns f(pad, ac) with both as std::integral_constant, so f can name a kernel template instance: pad is one of the
// OFB_PAD_* modes and ac is 0 or 1, anything else is OFB_EINVAL.
template <typename F>
static inline int ofb_dispatch_pad_ac(int pad, int ac, F f) {
    auto with_pad = [&](auto p) -> int {
        if (ac == 0) return f(p, std::false_type{});
        if (ac == 1) return f(p, std::true_type{});
        return OFB_EINVAL;
    };
    switch (pad) {
        case OFB_PAD_ZEROS: return with_pad(std::integral_constant<int, OFB_PAD_ZEROS>{});
        case OFB_PAD_BORDER: return with_pad(std::integral_constant<int, OFB_PAD_BORDER>{});
        case OFB_PAD_REFLECTION: return with_pad(std::integral_constant<int, OFB_PAD_REFLECTION>{});
        default: return OFB_EINVAL;
    }
}

// The floating-point element types of correlation pyramids and of the lookup's output and its gradient
static inline bool ofb_float_dtype(int dtype) {
    return dtype == OFB_DTYPE_F32 || dtype == OFB_DTYPE_F16 || dtype == OFB_DTYPE_BF16;
}
// Returns f(T{}) for the element type of dtype OFB_DTYPE_F32 / F16 / BF16 (float, __half, __nv_bfloat16), so f can name
// a kernel template instance; any other dtype is OFB_EINVAL.
template <typename F>
static inline int ofb_dispatch_dtype(int dtype, F f) {
    switch (dtype) {
        case OFB_DTYPE_F32: return f(float{});
        case OFB_DTYPE_F16: return f(__half{});
        case OFB_DTYPE_BF16: return f(__nv_bfloat16{});
        default: return OFB_EINVAL;
    }
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
// reflect_coordinates(_set_grad) (GridSampler.h:88-107,110-140); *dsign receives d(result)/d(in): +-1, or 0 for a
// one-pixel span
__device__ __forceinline__ float reflect_coord(float in, int twice_low, int twice_high, float* dsign = nullptr) {
    if (twice_low == twice_high) {
        if (dsign) *dsign = 0.0f;
        return 0.0f;
    }
    const float mn = (float)twice_low / 2.0f;
    const float span = (float)(twice_high - twice_low) / 2.0f;
    const float d = in - mn;
    in = fabsf(d);
    const float extra = fmodf(in, span);
    const bool odd = ((int)floorf(in / span)) % 2 != 0;
    if (dsign) *dsign = (d < 0.0f) != odd ? -1.0f : 1.0f;
    return odd ? (span - extra + mn) : (extra + mn);
}
template <bool AC>
__device__ __forceinline__ float reflect_index(float x, int size, float* dsign = nullptr) {
    return AC ? reflect_coord(x, 0, 2 * (size - 1), dsign) : reflect_coord(x, -1, 2 * size - 1, dsign);
}
template <int PAD, bool AC>
__device__ __forceinline__ float source_index(float g, int size) {
    float x = unnormalize<AC>(g, size);
    if (PAD == OFB_PAD_BORDER) {
        x = clip_coord(x, size);
    } else if (PAD == OFB_PAD_REFLECTION) {
        x = clip_coord(reflect_index<AC>(x, size), size);
    }
    return x;
}

// ---- the warp's sampling contract (K1 forward and backward, bilinear_sampler)
//
// Every grid_sample-style kernel takes its source coordinate from warp_source, its taps from bilinear_taps and, when
// it gathers from global memory, its sample from gather4.  Non-finite and far coordinates:
//   * zeros padding: a non-finite source coordinate samples 0, as does a finite one a pixel or more outside the frame;
//     that is what the oracle gives.  ATen's bilinear grid_sample returns NaN for a NaN or +-inf coordinate (its
//     weights are NaN and it multiplies them by the zero padding); it returns 0 for a finite far one.  bilinear_taps
//     leaves such a coordinate no tap in bounds, so gather4 returns 0; a kernel that multiplies zero-filled taps by the
//     weights instead (the NHWC float4 path, the TMA window) must keep it off that path.
//   * border padding: clip_coord maps NaN and -inf to 0 and +inf to size - 1.
//   * reflection: reflect_coord turns every non-finite coordinate into NaN and the clip maps it to 0.  ATen's CPU
//     kernel agrees on both.
// The mask (warp_source's valid) is false for every non-finite coordinate.

// flow multipliers and linspace steps.  x, y: 1 for a normalised flow (the reference's contract); 2/(W-1), 2/(H-1)
// fuse optical_flow.normalize (operator.py:117-130) into the warp -- one separately rounded multiply, as there.
// step_x, step_y: linspace(-1, 1, W / H) steps, divided once on the host (linspace_step, the same IEEE fp32 division).
struct FlowMul {
    float x, y;
    float step_x, step_y;
};

struct SrcPos {
    float ix, iy;   // source position in pixels, after padding
    bool valid;     // the grid coordinate lies strictly inside (-1, 1) on both axes
};

// Grid coordinate of output index i of n along one axis, with flow component f: linspace(-1, 1, n)[i] + f * mul
// (operator.py:49-56)
__device__ __forceinline__ float warp_grid_coord(float f, int i, int n, float step, float mul) {
    return __fadd_rn(linspace_m1_p1(i, n, step), __fmul_rn(f, mul));
}

// Output pixel (i, j) with flow (fx, fy): its grid coordinate, then grid_sample's un-normalise and padding
template <int PAD, bool AC>
__device__ __forceinline__ SrcPos warp_source(float fx, float fy, int i, int j, int H, int W, const FlowMul& fm) {
    const float gx = warp_grid_coord(fx, j, W, fm.step_x, fm.x);
    const float gy = warp_grid_coord(fy, i, H, fm.step_y, fm.y);
    SrcPos s;
    s.ix = source_index<PAD, AC>(gx, W);
    s.iy = source_index<PAD, AC>(gy, H);
    s.valid = (gx > -1.0f) && (gy > -1.0f) && (gx < 1.0f) && (gy < 1.0f);
    return s;
}

// A floor or rounded index as an int, clamped to [-2, size + 1] first: the one guard of the int conversion.  Indices
// outside the frame stay outside it (with their + 1 neighbour), and NaN becomes -2 (fmaxf(NaN, -2) = -2).
__device__ __forceinline__ int tap_index(float f, int size) { return (int)fminf(fmaxf(f, -2.0f), (float)size + 1.0f); }

struct BilinearTaps {
    int x0, y0;                  // upper-left tap (the + 1 taps are right of and below it)
    float wx0, wx1, wy0, wy1;    // per-axis weights of columns x0, x0 + 1 and rows y0, y0 + 1
    float w00, w01, w10, w11;    // tap weights, w<row><column>
    unsigned inb;                // in-bounds mask: bit 0 (x0, y0), 1 (x0 + 1, y0), 2 (x0, y0 + 1), 3 (x0 + 1, y0 + 1)
};

// BilinearTaps::inb of upper-left tap (x0, y0); PAD as bilinear_taps
template <int PAD>
__device__ __forceinline__ unsigned tap_mask(int x0, int y0, int H, int W) {
    bool inx0 = true, iny0 = true;
    if (PAD == OFB_PAD_ZEROS) { inx0 = x0 >= 0 && x0 < W; iny0 = y0 >= 0 && y0 < H; }
    const bool inx1 = (PAD != OFB_PAD_ZEROS || x0 + 1 >= 0) && x0 + 1 < W;
    const bool iny1 = (PAD != OFB_PAD_ZEROS || y0 + 1 >= 0) && y0 + 1 < H;
    return ((iny0 && inx0) ? 1u : 0u) | ((iny0 && inx1) ? 2u : 0u) | ((iny1 && inx0) ? 4u : 0u) |
           ((iny1 && inx1) ? 8u : 0u);
}
// Taps of source position (ix, iy) in an H x W frame (GridSampler.h:330-380).  PAD != zeros promises that ix, iy were
// clipped into [0, size - 1] by source_index: the upper-left tap is then inside, only the + 1 taps can fall off the
// far edge (with weight 0), and no guard is needed.  The zeros form takes any coordinate: a non-finite one has NaN
// weights and no tap in bounds.
template <int PAD>
__device__ __forceinline__ BilinearTaps bilinear_taps(float ix, float iy, int H, int W) {
    const float x0f = floorf(ix), y0f = floorf(iy);
    BilinearTaps t;
    t.wx1 = ix - x0f; t.wx0 = (x0f + 1.0f) - ix;
    t.wy1 = iy - y0f; t.wy0 = (y0f + 1.0f) - iy;
    t.w00 = t.wx0 * t.wy0; t.w01 = t.wx1 * t.wy0; t.w10 = t.wx0 * t.wy1; t.w11 = t.wx1 * t.wy1;
    t.x0 = PAD != OFB_PAD_ZEROS ? (int)x0f : tap_index(x0f, W);
    t.y0 = PAD != OFB_PAD_ZEROS ? (int)y0f : tap_index(y0f, H);
    t.inb = tap_mask<PAD>(t.x0, t.y0, H, W);
    return t;
}

// input element -> fp32: frames, flows, feature maps and mask logits arrive in fp32, or in half precision from an
// autocast caller
__device__ __forceinline__ float ld_f32(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_f32(const __nv_bfloat16* p) {
    return __uint_as_float((unsigned)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}
__device__ __forceinline__ float ld_f32(const __half* p) {
    return __half2float(__ushort_as_half(__ldg(reinterpret_cast<const unsigned short*>(p))));
}

// The bilinear sample at p (the upper-left tap) from global memory, dx / dy elements to the next column / row: the
// in-bounds taps of mask m (bits as BilinearTaps::inb; higher bits are ignored), each widened exactly to fp32 and
// accumulated in tap order with one rounding each.  Taps outside m are not read and add nothing, whatever their weight.
template <typename T>
__device__ __forceinline__ float gather4(const T* p, size_t dx, size_t dy, unsigned m, float w00, float w01, float w10,
                                         float w11) {
    float acc = 0.0f;
    if (m & 1u) acc = __fmaf_rn(ld_f32(p), w00, acc);
    if (m & 2u) acc = __fmaf_rn(ld_f32(p + dx), w01, acc);
    if (m & 4u) acc = __fmaf_rn(ld_f32(p + dy), w10, acc);
    if (m & 8u) acc = __fmaf_rn(ld_f32(p + dy + dx), w11, acc);
    return acc;
}
template <typename T>
__device__ __forceinline__ float gather4(const T* p, size_t dx, size_t dy, const BilinearTaps& t) {
    return gather4(p, dx, dy, t.inb, t.w00, t.w01, t.w10, t.w11);
}

// One tap of the correlation lookup's window (CorrBlock.__call__ + bilinear_sampler, methods/raft/model/corr.py:56-77,
// utils.py:64-80).  Bit-exactness contract (SURVEY.md 8c): the fp32 coordinate sequence is replayed operation by
// operation with round-to-nearest intrinsics so nvcc cannot contract it, and the floor indices and validity masks match
// the reference bit for bit.  `center` is the level-scaled coordinate c = coord / 2^l (corr.py:68, exact):
//     x  = c + (t - r)                       (corr.py:70; window TRANSPOSED: the x taps move the output channel's i)
//     g  = 2*x/(size-1) - 1                  (utils.py:70-71)
//     ix = ((g + 1) * 0.5) * (size-1)        (ATen GridSampler.h:30, align_corners=True; (g+1)/2 == (g+1)*0.5 exactly)
//     fl = floor(ix); valid = -1 < g < 1     (utils.py:77)
// Every lookup kernel (forward, backward, coordinate backward, on-demand) takes its taps from here; each decides what an
// out-of-guard tap contributes.
// The coordinate backward (lookup_coords_bwd.cu) differentiates the samples of these taps as ATen's GridSampler backward
// does (zeros padding): a tap outside the image reads the value 0; a level with a tap outside the guard -- a non-finite
// or far coordinate, or a level of width or height 1 (size - 1 = 0) -- contributes exactly 0 (ATen: NaN for a NaN
// coordinate); elements between w_l and the row pitch never reach the result.
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

// One axis of a (query, level) window for the kernels that stream it row by row (the register-tile forward lookup and
// the coordinate backward).  Within the guarded coordinate range every tap's floor index is t + anchor + {0, 1} (the
// fp32 round trip can move a tap sitting on an integer to the pixel below), so tap t reads window positions t + d[t]
// and t + d[t] + 1 of a D + 2 element window starting at the anchor.
template <int R>
struct TapSet {
    static constexpr int D = 2 * R + 1;
    float w0[D], w1[D];
    int anchor;          // min over taps of (floor index - tap number); tap t reads anchor + t + d[t]
    unsigned dmask;      // bit t = d[t]
    unsigned vmask;      // bit t = utils.py:77 predicate
    bool dead;           // some tap outside the guarded range: every in-range tap is outside the image
};

template <int R>
__device__ __forceinline__ TapSet<R> make_taps(float center, int size, int32_t* idx_dst) {
    constexpr int D = 2 * R + 1;
    TapSet<R> ts;
    int i0[D];
    ts.dead = false;
    ts.vmask = 0;
    int anchor = INT_MAX;
#pragma unroll
    for (int t = 0; t < D; ++t) {
        const LookupTap tp = lookup_tap(center, t, R, size);
        ts.w1[t] = tp.w1;
        ts.w0[t] = tp.w0;
        ts.dead |= !tp.in_guard;
        i0[t] = tp.in_guard ? (int)tp.fl : 0;
        if (idx_dst) idx_dst[t] = (int32_t)tp.fl;
        ts.vmask |= tp.valid ? (1u << t) : 0u;
        anchor = min(anchor, i0[t] - t);
    }
    ts.anchor = anchor;
    ts.dmask = 0;
#pragma unroll
    for (int t = 0; t < D; ++t) {
        const int d = i0[t] - t - anchor;           // 0 or 1 unless dead
        ts.dmask |= (d != 0) ? (1u << t) : 0u;
        ts.dead |= (d > 1);
    }
    return ts;
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

// half-word `hi` (0: low, 1: high) of a 4-byte word of two bf16 / fp16 elements -> fp32
template <typename T> __device__ __forceinline__ float widen16(unsigned wd, int hi);
template <> __device__ __forceinline__ float widen16<__nv_bfloat16>(unsigned wd, int hi) {
    return __uint_as_float(hi ? (wd & 0xffff0000u) : (wd << 16));
}
template <> __device__ __forceinline__ float widen16<__half>(unsigned wd, int hi) {
    return __half2float(__ushort_as_half((unsigned short)(hi ? (wd >> 16) : (wd & 0xffffu))));
}
// fp32 -> an output element, rounded to nearest even: the bits ATen's out_fp32.to(dtype) gives (fp16: beyond +-65504
// is inf).  Its inverse for a 16-bit gradient read back is ld_f32, an exact widening.
template <typename T> __device__ __forceinline__ T narrow(float v);
template <> __device__ __forceinline__ float narrow<float>(float v) { return v; }
template <> __device__ __forceinline__ __half narrow<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 narrow<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// One window row of a 16-bit pyramid from its aligned chunk loads: w[0..7] are the 8-element (16-byte) chunks at
// xa and xa + 8, w[8..9] the first 4 elements at xa + 16, as packed pairs.  px receives elements s .. s + WIN - 1
// (s = xs - xa in 0..7, passed as q1 = bit 1, q2 = bit 2 and hs = 16 * bit 0) widened to fp32: word shifts by 1 and
// 2, then a half-word funnel shift.
template <typename T, int WIN>
__device__ __forceinline__ void realign_row(const uint32_t (&w)[10], unsigned q1, unsigned q2, unsigned hs,
                                            float (&px)[WIN]) {
    constexpr int NW = (WIN + 1) / 2;                           // packed words per realigned row (6 for WIN = 11)
    uint32_t t1[9], t2[NW + 1], v[NW];
#pragma unroll
    for (int k = 0; k < 9; ++k) t1[k] = q1 ? w[k + 1] : w[k];
#pragma unroll
    for (int k = 0; k <= NW; ++k) t2[k] = q2 ? t1[k + 2] : t1[k];
#pragma unroll
    for (int k = 0; k < NW; ++k) v[k] = __funnelshift_r(t2[k], t2[k + 1], hs);
#pragma unroll
    for (int e = 0; e < WIN; ++e) px[e] = widen16<T>(v[e >> 1], e & 1);
}

// The aligned 8-element (16-byte) chunks holding window columns xs .. xs + cols - 1 of a 16-bit level whose row pitch
// is a multiple of 8 (the register-tile forward lookup and the coordinate backward read window rows this way): chunks
// at xa, xa + 8 and xa + 16, of the last only the first 4 elements (s + cols - 1 <= 17).  ck0 .. ck2: the chunk lies
// inside the row (ck2 only when it holds a window column); q1, q2, hs: realign_row's shift of s.
struct RowChunks {
    int xa, s;
    unsigned q1, q2, hs;
    bool ck0, ck1, ck2;
};
__device__ __forceinline__ RowChunks row_chunks(int xs, int cols, int pitch) {
    RowChunks c;
    c.xa = xs & ~7;
    c.s = xs - c.xa;                                            // s in 0..7
    c.q1 = (unsigned)(c.s >> 1) & 1u;
    c.q2 = (unsigned)(c.s >> 2) & 1u;
    c.hs = (unsigned)(c.s & 1) * 16u;
    c.ck0 = c.xa >= 0 && c.xa + 8 <= pitch;
    c.ck1 = c.xa + 8 >= 0 && c.xa + 16 <= pitch;
    c.ck2 = (c.s + cols > 16) && c.xa + 16 >= 0 && c.xa + 24 <= pitch;
    return c;
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

// ---- the correlation pyramid's layout contract (include/ofb200.h): the one check, addressing rule and reader choice
// An ofb_pyramid as the kernels receive it (strides in elements, unused levels zeroed); kernel parameter blocks derive
// from it and add their scalars.
struct PyramidView {
    void* base[OFB_MAX_LEVELS];
    long long q_stride[OFB_MAX_LEVELS];
    int pitch[OFB_MAX_LEVELS];
    int lh[OFB_MAX_LEVELS];
    int lw[OFB_MAX_LEVELS];
    int levels, dtype;
    int blocked;            // 8x4-blocked layouts (OFB_LAYOUT_BLOCK8X4, OFB_LAYOUT_QMINOR8X4)
    long long blk_stride;   // elements between consecutive 8x4 blocks: 32, or 32 * Q (query-minor)
};

// The 8-element piece at (y, x), x % 8 == 0, of a level of view V with row pitch `pitch`: one row of an 8x4 block
// (V.blocked) or 8 consecutive elements of a row; OFB_PIECE_OFFSET is its offset in the (query, level) slice, OFB_PIECE
// its address, the next piece along x OFB_PIECE_STEP(V) elements further.  Macros, and OFB_PIECE adds the _TERMS to the
// pointer one by one: as an inline function or slice + OFB_PIECE_OFFSET, the register-tile forward's schedule changes.
#define OFB_BLOCK_TERMS(V, y, x, pitch) ((long long)((y) >> 2) * ((pitch) >> 3) + ((x) >> 3)) * (V).blk_stride + ((y) & 3) * 8
#define OFB_ROW_TERMS(y, x, pitch) (long long)(y) * (pitch) + (x)
#define OFB_PIECE_OFFSET(V, y, x, pitch) ((V).blocked ? (OFB_BLOCK_TERMS(V, y, x, pitch)) : (OFB_ROW_TERMS(y, x, pitch)))
#define OFB_PIECE(slice, V, y, x, pitch) \
    ((V).blocked ? (slice) + OFB_BLOCK_TERMS(V, y, x, pitch) : (slice) + OFB_ROW_TERMS(y, x, pitch))
#define OFB_PIECE_STEP(V) ((V).blocked ? (V).blk_stride : 8)

// Fills v from pyr (Q = B * h * w queries) and checks the rules every user relies on, else OFB_EINVAL: 1 ..
// OFB_MAX_LEVELS levels, a known dtype and layout, per level a base, a positive size, pitch >= width, and q_stride = 32
// in the query-minor layout.  Each entry point then checks only its own requirements.
inline int check_pyramid(const ofb_pyramid* pyr, long long Q, PyramidView& v) {
    if (pyr->levels < 1 || pyr->levels > OFB_MAX_LEVELS) return OFB_EINVAL;
    if (!ofb_float_dtype(pyr->dtype)) return OFB_EINVAL;
    if (pyr->layout < OFB_LAYOUT_ROWS || pyr->layout > OFB_LAYOUT_QMINOR8X4) return OFB_EINVAL;
    const bool qminor = pyr->layout == OFB_LAYOUT_QMINOR8X4;
    v.levels = pyr->levels; v.dtype = pyr->dtype;
    v.blocked = pyr->layout != OFB_LAYOUT_ROWS;
    v.blk_stride = qminor ? 32 * Q : 32;
    for (int l = 0; l < OFB_MAX_LEVELS; ++l) {
        const bool on = l < pyr->levels;
        v.base[l] = on ? pyr->base[l] : nullptr;
        v.q_stride[l] = on ? pyr->q_stride[l] : 0;
        v.pitch[l] = on ? pyr->row_pitch[l] : 0;
        v.lh[l] = on ? pyr->lvl_h[l] : 0;
        v.lw[l] = on ? pyr->lvl_w[l] : 0;
        if (on && (!v.base[l] || v.lh[l] <= 0 || v.lw[l] <= 0 || v.pitch[l] < v.lw[l] || (qminor && v.q_stride[l] != 32)))
            return OFB_EINVAL;
    }
    return OFB_OK;
}

// The radii the register-tile forward lookup is built for
constexpr bool tile_radius(int radius) { return radius == 3 || radius == 4; }

// How ofb_corr_lookup and ofb_corr_lookup_coords_backward read v at `radius` (both decide here, so they accept the same
// pyramids).  *chunked: 16-bit rows or 8x4 blocks in 16-byte aligned 8-element chunks, read whole by the register-tile
// forward at tile_radius and by the coordinate backward; other rows are read element-wise.  OFB_EUNSUPPORTED: a level
// above 65536, or blocks the register-tile forward does not read; OFB_EALIGN: 16-bit levels not in 4-byte words.
inline int lookup_reader(const PyramidView& v, int radius, bool& chunked) {
    const bool half16 = chunked = v.dtype != OFB_DTYPE_F32;
    for (int l = 0; l < v.levels; ++l) {
        const uintptr_t base = reinterpret_cast<uintptr_t>(v.base[l]);
        if (v.lh[l] > 65536 || v.lw[l] > 65536) return OFB_EUNSUPPORTED;
        if (half16 && ((v.pitch[l] & 1) || (v.q_stride[l] & 1) || (base & 3))) return OFB_EALIGN;
        chunked = chunked && v.pitch[l] % 8 == 0 && v.q_stride[l] % 8 == 0 && (base & 15) == 0;
    }
    if (v.blocked && !(chunked && tile_radius(radius))) return OFB_EUNSUPPORTED;
    return OFB_OK;
}

}  // namespace ofb
