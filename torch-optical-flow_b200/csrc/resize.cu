// resize.cu -- K4a: bilinear flow resize with magnitude rescale, and scale/normalize.
//
// Replaces F.interpolate(mode="bilinear") + scale() in optical_flow.resize (reference
// optical_flow/operator/operator.py:85-114, align_corners=False) and
// 8 * F.interpolate(align_corners=True) in upflow8 (methods/raft/model/utils.py:89-91).
// Source index / lambda as ATen UpSample.h:259-313,442-476.  Write-bound: one thread produces
// four consecutive output pixels (one 16-byte store when the row allows it).
#include "common.cuh"

namespace {

__device__ __forceinline__ void src_index(float ratio, int dst, int in_size, int out_size, bool ac, int& i0, int& i1,
                                          float& l0, float& l1) {
    if (out_size == in_size) { i0 = dst; i1 = dst; l0 = 1.0f; l1 = 0.0f; return; }
    float r;
    if (ac) {
        r = __fmul_rn(ratio, (float)dst);
    } else {
        r = __fmaf_rn(ratio, (float)dst + 0.5f, -0.5f);
        r = r < 0.0f ? 0.0f : r;
    }
    int idx = (int)floorf(r);
    idx = min(idx, in_size - 1);
    float lam = fminf(fmaxf(r - (float)idx, 0.0f), 1.0f);
    i0 = idx;
    i1 = idx + (idx < in_size - 1 ? 1 : 0);
    l1 = lam;
    l0 = 1.0f - lam;
}

__global__ void __launch_bounds__(256) resize_kernel(const float* __restrict__ in, float* __restrict__ out, int NC,
                                                     int H, int W, int Ho, int Wo, int ac, float rh, float rw,
                                                     float mul_x, float mul_y, int vec_ok) {
    const int Wq = (Wo + 3) / 4;
    const size_t total = (size_t)NC * Ho * Wq;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int xq = (int)(t % Wq);
        const int oy = (int)((t / Wq) % Ho);
        const int nc = (int)(t / ((size_t)Wq * Ho));
        const float* src = in + (size_t)nc * H * W;
        const float mul = (nc & 1) ? mul_y : mul_x;   // channel index c = nc % C, C even -> parity of nc
        int y0, y1; float ly0, ly1;
        src_index(rh, oy, H, Ho, ac != 0, y0, y1, ly0, ly1);
        float r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int ox = xq * 4 + k;
            r[k] = 0.0f;
            if (ox < Wo) {
                int x0, x1; float lx0, lx1;
                src_index(rw, ox, W, Wo, ac != 0, x0, x1, lx0, lx1);
                const float a = __ldg(src + (size_t)y0 * W + x0), b = __ldg(src + (size_t)y0 * W + x1);
                const float c = __ldg(src + (size_t)y1 * W + x0), d = __ldg(src + (size_t)y1 * W + x1);
                const float top = __fmaf_rn(lx0, a, __fmul_rn(lx1, b));
                const float bot = __fmaf_rn(lx0, c, __fmul_rn(lx1, d));
                r[k] = __fmul_rn(__fmaf_rn(ly0, top, __fmul_rn(ly1, bot)), mul);
            }
        }
        float* dst = out + ((size_t)nc * Ho + oy) * Wo + (size_t)xq * 4;
        if (vec_ok && xq * 4 + 3 < Wo) {
            *reinterpret_cast<float4*>(dst) = make_float4(r[0], r[1], r[2], r[3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (xq * 4 + k < Wo) dst[k] = r[k];
        }
    }
}

// Candidate outputs whose taps may touch source index `src` along one axis: every dst with src_index(dst) in
// {src - 1, src}, i.e. a source coordinate r in [src - 1, src + 1), from the inverse of the forward's mapping, widened
// by 2 for its rounding and clamped to [0, out_size).  Only a superset: the caller re-checks each candidate's taps.
__device__ __forceinline__ void dst_range(float ratio, int src, int in_size, int out_size, bool ac, int& lo, int& hi) {
    if (out_size == in_size) { lo = hi = src; return; }
    if (ratio == 0.0f) { lo = 0; hi = out_size - 1; return; }   // align_corners with one output: every dst reads 0
    float a, b;
    if (ac) {
        a = (float)(src - 1) / ratio;
        b = (float)(src + 1) / ratio;
    } else {
        a = ((float)(src - 1) + 0.5f) / ratio - 0.5f;
        b = ((float)(src + 1) + 0.5f) / ratio - 0.5f;
    }
    a = src <= 1 ? 0.0f : fmaxf(floorf(a) - 2.0f, 0.0f);   // r < 0 is clamped to 0: taps 0 and 1 (weight 0)
    b = fminf(ceilf(b) + 2.0f, (float)(out_size - 1));
    lo = (int)a;
    hi = (int)b;
}

// Adjoint of resize_kernel (what autograd computes through F.interpolate + scale, operator.py:112-113, and through
// 8 * F.interpolate in upflow8), as a gather: one thread per source pixel sums, in ascending output order (row, then
// column, then the taps 00, 01, 10, 11), the forward weight times the magnitude-scaled gradient of every output tap
// that lands on it -- the terms ATen's backward scatters, zero-weight taps included.  The taps are recomputed with the
// forward's own src_index, so no inverted float formula decides which outputs count.  Deterministic: the same bits
// on every run; d_in is accumulated into with one add per element.
__global__ void __launch_bounds__(256) resize_bwd_kernel(const float* __restrict__ d_out, float* __restrict__ d_in,
                                                         int NC, int H, int W, int Ho, int Wo, int ac, float rh, float rw,
                                                         float mul_x, float mul_y) {
    const size_t total = (size_t)NC * H * W;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int ix = (int)(t % W);
        const int iy = (int)((t / W) % H);
        const int nc = (int)(t / ((size_t)W * H));
        const float mul = (nc & 1) ? mul_y : mul_x;
        const float* src = d_out + (size_t)nc * Ho * Wo;
        int oy0, oy1, ox0, ox1;
        dst_range(rh, iy, H, Ho, ac != 0, oy0, oy1);
        dst_range(rw, ix, W, Wo, ac != 0, ox0, ox1);
        float acc = 0.0f;
        for (int oy = oy0; oy <= oy1; ++oy) {
            int y0, y1; float ly0, ly1;
            src_index(rh, oy, H, Ho, ac != 0, y0, y1, ly0, ly1);
            const bool hy0 = y0 == iy, hy1 = y1 == iy;
            if (!hy0 && !hy1) continue;
            for (int ox = ox0; ox <= ox1; ++ox) {
                int x0, x1; float lx0, lx1;
                src_index(rw, ox, W, Wo, ac != 0, x0, x1, lx0, lx1);
                const bool hx0 = x0 == ix, hx1 = x1 == ix;
                if (!hx0 && !hx1) continue;
                const float g = __fmul_rn(__ldg(src + (size_t)oy * Wo + ox), mul);
                if (hy0 && hx0) acc += ly0 * lx0 * g;
                if (hy0 && hx1) acc += ly0 * lx1 * g;
                if (hy1 && hx0) acc += ly1 * lx0 * g;
                if (hy1 && hx1) acc += ly1 * lx1 * g;
            }
        }
        d_in[t] += acc;
    }
}

__global__ void __launch_bounds__(256) scale_flow_kernel(const float* __restrict__ in, float* __restrict__ out, int B,
                                                         int64_t HW, float fx, float fy) {
    const int64_t total = (int64_t)B * 2 * HW;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)((t / HW) & 1);
        out[t] = __fmul_rn(__ldg(in + t), c ? fy : fx);
    }
}

// scale in the flow's own dtype (the reference's scale is dtype-preserving, operator.py:59-82: the factor is filled
// into a tensor of the flow's dtype, then one multiply).  Half types: factor rounded to the type, the exact fp32
// product of two 8- / 11-bit significands rounded once -- what a native half multiply returns.
template <typename T> struct ScaleT;
template <> struct ScaleT<double> {
    static __device__ __forceinline__ double mul(double x, double f) { return __dmul_rn(x, f); }
    static __host__ double factor(double f) { return f; }
};
template <> struct ScaleT<__half> {
    static __device__ __forceinline__ __half mul(__half x, double f) { return __float2half_rn(__fmul_rn(__half2float(x), (float)f)); }
    static __host__ double factor(double f) { return (double)__half2float(__float2half_rn((float)f)); }
};
template <> struct ScaleT<__nv_bfloat16> {
    static __device__ __forceinline__ __nv_bfloat16 mul(__nv_bfloat16 x, double f) {
        return __float2bfloat16_rn(__fmul_rn(__bfloat162float(x), (float)f));
    }
    static __host__ double factor(double f) { return (double)__bfloat162float(__float2bfloat16_rn((float)f)); }
};

template <typename T>
__global__ void __launch_bounds__(256) scale_flow_any_kernel(const T* __restrict__ in, T* __restrict__ out, int B,
                                                             int64_t HW, double fx, double fy) {
    const int64_t total = (int64_t)B * 2 * HW;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)((t / HW) & 1);
        out[t] = ScaleT<T>::mul(in[t], c ? fy : fx);
    }
}

template <typename T>
int launch_scale_any(const void* flow, void* out, int B, int64_t HW, double fx, double fy, int blocks, cudaStream_t st) {
    scale_flow_any_kernel<T><<<blocks, 256, 0, st>>>(reinterpret_cast<const T*>(flow), reinterpret_cast<T*>(out), B, HW,
                                                     ScaleT<T>::factor(fx), ScaleT<T>::factor(fy));
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

}  // namespace

OFB_API int ofb_resize_bilinear_f32(const float* in, float* out, int N, int C, int H, int W, int Ho, int Wo,
                                    int align_corners, float mul_x, float mul_y, void* stream) {
    if (N == 0 || C == 0 || Ho == 0 || Wo == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!in || !out || N < 0 || C < 0 || H <= 0 || W <= 0 || Ho < 0 || Wo < 0) return OFB_EINVAL;
    if ((C & 1) && (mul_x != mul_y)) return OFB_EINVAL;   // per-axis factors need (x,y) channel pairs
    const size_t total = (size_t)N * C * Ho * ((Wo + 3) / 4);
    if (total == 0) return OFB_OK;
    float rh, rw;
    if (align_corners) {
        rh = Ho > 1 ? (float)(H - 1) / (float)(Ho - 1) : 0.0f;
        rw = Wo > 1 ? (float)(W - 1) / (float)(Wo - 1) : 0.0f;
    } else {
        rh = (float)H / (float)Ho;
        rw = (float)W / (float)Wo;
    }
    int blocks = (int)((total + 255) / 256);
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    const int vec_ok = (Wo % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    resize_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(in, out, N * C, H, W, Ho, Wo, align_corners, rh, rw, mul_x,
                                                             mul_y, vec_ok);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_resize_bilinear_backward_f32(const float* d_out, float* d_in, int N, int C, int H, int W, int Ho, int Wo,
                                             int align_corners, float mul_x, float mul_y, void* stream) {
    if (N == 0 || C == 0 || Ho == 0 || Wo == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!d_out || !d_in || N < 0 || C < 0 || H <= 0 || W <= 0 || Ho < 0 || Wo < 0) return OFB_EINVAL;
    if ((C & 1) && (mul_x != mul_y)) return OFB_EINVAL;
    if ((size_t)N * C * Ho * Wo == 0) return OFB_OK;
    const size_t total = (size_t)N * C * H * W;   // one thread per source pixel
    float rh, rw;
    if (align_corners) {
        rh = Ho > 1 ? (float)(H - 1) / (float)(Ho - 1) : 0.0f;
        rw = Wo > 1 ? (float)(W - 1) / (float)(Wo - 1) : 0.0f;
    } else {
        rh = (float)H / (float)Ho;
        rw = (float)W / (float)Wo;
    }
    size_t blocks = (total + 255) / 256;
    const size_t cap = (size_t)ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    resize_bwd_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(d_out, d_in, N * C, H, W, Ho, Wo, align_corners, rh,
                                                                      rw, mul_x, mul_y);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_scale_flow_f32(const float* flow, float* out, int B, int64_t HW, float fx, float fy, void* stream) {
    if (B == 0 || HW == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!flow || !out || B < 0 || HW < 0) return OFB_EINVAL;
    const int64_t total = (int64_t)B * 2 * HW;
    if (total == 0) return OFB_OK;
    int64_t blocks = (total + 255) / 256;
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    scale_flow_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(flow, out, B, HW, fx, fy);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_scale_flow(const void* flow, void* out, int dtype, int B, int64_t HW, double fx, double fy, void* stream) {
    if (dtype == OFB_DTYPE_F32)
        return ofb_scale_flow_f32(reinterpret_cast<const float*>(flow), reinterpret_cast<float*>(out), B, HW, (float)fx, (float)fy, stream);
    if (B == 0 || HW == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!flow || !out || B < 0 || HW < 0) return OFB_EINVAL;
    int64_t blocks = ((int64_t)B * 2 * HW + 255) / 256;
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == OFB_DTYPE_F64) return launch_scale_any<double>(flow, out, B, HW, fx, fy, (int)blocks, st);
    if (dtype == OFB_DTYPE_F16) return launch_scale_any<__half>(flow, out, B, HW, fx, fy, (int)blocks, st);
    if (dtype == OFB_DTYPE_BF16) return launch_scale_any<__nv_bfloat16>(flow, out, B, HW, fx, fy, (int)blocks, st);
    return OFB_EINVAL;
}
