// corr_simt.cu -- operand preparation for K2 and a CUDA-core correlation-pyramid builder.
//
//  * ofb_corr_prep_bf16 / _from / _to: fmap (B,C,h,w) NCHW -> (B,(h/pool)*(w/pool),C) bf16 or fp16, K-major, times
//    `scale`, optionally averaged over complete pool x pool blocks.  Replaces the .view /
//    .transpose(1,2) in CorrBlock.corr (reference methods/raft/model/corr.py:82-85), folds the
//    1/sqrt(C) of corr.py:87 into fmap1, and -- pool = 4 on fmap2 -- feeds the run that produces
//    pyramid levels 2 and 3 (avg_pool2d is linear: corr.py:52-54).  The only extra passes the
//    tensor-core path needs (0.2 GB at the Sintel configuration against 2.1 GB of pyramid).
//  * ofb_pyramid_layout: strides of the pyramid buffers (see include/ofb200.h).
//  * ofb_corr_pyramid_simt_f32: fp32 CUDA-core GEMM + successive 2x2 pooling -- the reference's
//    own op order (corr.py:44-54,79-87), fp32, bf16 or fp16 stored.  Not the fast path: tests use it as an on-device
//    cross-check of the tcgen05 builder at sizes the CPU oracle cannot reach.
#include <type_traits>

#include "common.cuh"

namespace {

// ---------------------------------------------------------------- cast + transpose
constexpr int TP = 32;    // pixels per tile
constexpr int TCMAX = 256;  // channels per tile (the whole K extent of the tensor-core path)

// One CTA turns a 32-pixel x C-channel tile: reads are 128-byte lines (32 pixels of one channel), 8 in
// flight per thread; writes are whole 2*C-byte pixel rows of the K-major operand (TOut: bf16 or fp16).
template <int POOL, typename TIn, typename TOut>
__global__ void __launch_bounds__(256) prep_kernel(const TIn* __restrict__ in, TOut* __restrict__ out, int C,
                                                   int h, int w, float scale) {
    // output pixel p = (yo, xo) of the (h/POOL) x (w/POOL) image = mean of a complete POOL x POOL block
    extern __shared__ float tile[];                       // [Ct][TP + 1]
    const int ho = h / POOL, wo = w / POOL, HWo = ho * wo, HW = h * w;
    const int b = blockIdx.z, p0 = blockIdx.x * TP, c0 = blockIdx.y * TCMAX;
    const int Ct = min(TCMAX, C - c0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = p0 + lane;
    const int yo = p / wo, xo = p - yo * wo;
    const TIn* src0 = in + ((size_t)b * C + c0) * HW + (size_t)(yo * POOL) * w + xo * POOL;
    const bool pok = p < HWo;
    for (int cb = warp; cb < Ct; cb += 64) {              // 8 warps x 8 independent channel rows per pass
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int c = cb + 8 * u;
            v[u] = 0.0f;
            if (pok && c < Ct) {
                const TIn* src = src0 + (size_t)c * HW;
                if (POOL == 1) {
                    v[u] = ofb::ld_f32(src);
                } else {
                    float a = 0.0f;
#pragma unroll
                    for (int dy = 0; dy < POOL; ++dy)
#pragma unroll
                        for (int dx = 0; dx < POOL; ++dx) a += ofb::ld_f32(src + dy * w + dx);
                    v[u] = a * (1.0f / (float)(POOL * POOL));
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int c = cb + 8 * u;
            if (c < Ct) tile[c * (TP + 1) + lane] = v[u] * scale;
        }
    }
    __syncthreads();
    // write: one pixel row (Ct channels) per warp pass, two 16-bit elements per lane, 128 bytes per instruction
    for (int q = warp; q < TP; q += 8) {
        const int pp = p0 + q;
        if (pp >= HWo) break;
        TOut* dst = out + ((size_t)b * HWo + pp) * C + c0;
        for (int cc = 2 * lane; cc < Ct; cc += 64) {
            if constexpr (std::is_same<TOut, __half>::value) {
                __half2 v2 = __floats2half2_rn(tile[cc * (TP + 1) + q], tile[(cc + 1) * (TP + 1) + q]);
                *reinterpret_cast<__half2*>(dst + cc) = v2;
            } else {
                __nv_bfloat162 v2 = __floats2bfloat162_rn(tile[cc * (TP + 1) + q], tile[(cc + 1) * (TP + 1) + q]);
                *reinterpret_cast<__nv_bfloat162*>(dst + cc) = v2;
            }
        }
    }
}

// ---------------------------------------------------------------- fp32 GEMM (level 0)
template <typename T> __device__ __forceinline__ T cvt_out(float v);
template <> __device__ __forceinline__ float cvt_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half cvt_out<__half>(float v) { return __float2half_rn(v); }

constexpr int GT = 32;

template <typename T>
__global__ void __launch_bounds__(GT * GT / 4) corr_l0_kernel(const float* __restrict__ f1, const float* __restrict__ f2,
                                                              T* __restrict__ l0, long long q_stride, int pitch, int C,
                                                              int h, int w, float scale) {
    // C[p][n] = sum_c f1[c][p] * f2[c][n]; 32x32 output tile, 8x32 threads, 4 rows per thread
    __shared__ float sa[GT][GT + 1];
    __shared__ float sb[GT][GT + 1];
    const int N = h * w;
    const int b = blockIdx.z, p0 = blockIdx.y * GT, n0 = blockIdx.x * GT;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // ty in 0..7
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k0 = 0; k0 < C; k0 += GT) {
        for (int r = ty; r < GT; r += 8) {
            const int c = k0 + r;
            sa[r][tx] = (c < C && p0 + tx < N) ? __ldg(f1 + ((size_t)b * C + c) * N + p0 + tx) : 0.0f;
            sb[r][tx] = (c < C && n0 + tx < N) ? __ldg(f2 + ((size_t)b * C + c) * N + n0 + tx) : 0.0f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < GT; ++k) {
            const float bv = sb[k][tx];
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[r] = fmaf(sa[k][ty + 8 * r], bv, acc[r]);
        }
        __syncthreads();
    }
    const int n = n0 + tx;
    if (n < N) {
        const int y = n / w, x = n - y * w;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int p = p0 + ty + 8 * r;
            if (p < N) l0[((size_t)b * N + p) * q_stride + (size_t)y * pitch + x] = cvt_out<T>(acc[r] * scale);
        }
    }
}

template <typename T> __device__ __forceinline__ float cvt_in(T v);
template <> __device__ __forceinline__ float cvt_in<float>(float v) { return v; }
template <> __device__ __forceinline__ float cvt_in<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float cvt_in<__half>(__half v) { return __half2float(v); }

template <typename T>
__global__ void __launch_bounds__(256) pool2_kernel(const T* __restrict__ src, T* __restrict__ dst, long long Qn,
                                                    long long sq, int spitch, long long dq, int dpitch, int dh, int dw) {
    const long long per = (long long)dh * dw, total = Qn * per;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long q = t / per;
        const int r = (int)(t - q * per), y = r / dw, x = r - y * dw;
        const T* s = src + q * sq + (size_t)(2 * y) * spitch + 2 * x;
        float v = cvt_in<T>(s[0]);
        v += cvt_in<T>(s[1]);
        v += cvt_in<T>(s[spitch]);
        v += cvt_in<T>(s[spitch + 1]);
        dst[q * dq + (size_t)y * dpitch + x] = cvt_out<T>(v / 4.0f);
    }
}

template <typename T>
int build_simt(const float* f1, const float* f2, const ofb::PyramidView& v, int B, int C, int h, int w, float scale,
               cudaStream_t st) {
    const int N = h * w;
    dim3 grid((N + GT - 1) / GT, (N + GT - 1) / GT, B);
    corr_l0_kernel<T><<<grid, GT * GT / 4, 0, st>>>(f1, f2, reinterpret_cast<T*>(v.base[0]), v.q_stride[0], v.pitch[0], C, h,
                                                    w, scale);
    OFB_LAUNCH_CHECK();
    for (int l = 1; l < v.levels; ++l) {
        const long long total = (long long)B * N * v.lh[l] * v.lw[l];
        if (total == 0) continue;
        long long blocks = (total + 255) / 256;
        const int cap = ofb_num_sms() * 32;
        if (blocks > cap) blocks = cap;
        pool2_kernel<T><<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const T*>(v.base[l - 1]), reinterpret_cast<T*>(v.base[l]),
                                                     (long long)B * N, v.q_stride[l - 1], v.pitch[l - 1], v.q_stride[l],
                                                     v.pitch[l], v.lh[l], v.lw[l]);
        OFB_LAUNCH_CHECK();
    }
    return OFB_OK;
}

}  // namespace

template <typename TIn, typename TOut>
static int launch_prep(const void* fmap, TOut* out, int B, int C, int h, int w, int pool, float scale, int HWo,
                       cudaStream_t st) {
    dim3 grid((HWo + TP - 1) / TP, (C + TCMAX - 1) / TCMAX, B);
    const size_t smem = (size_t)(C < TCMAX ? C : TCMAX) * (TP + 1) * sizeof(float);      // <= 33 KiB
    const TIn* in = reinterpret_cast<const TIn*>(fmap);
    if (pool == 1) prep_kernel<1, TIn, TOut><<<grid, 256, smem, st>>>(in, out, C, h, w, scale);
    else if (pool == 2) prep_kernel<2, TIn, TOut><<<grid, 256, smem, st>>>(in, out, C, h, w, scale);
    else if (pool == 4) prep_kernel<4, TIn, TOut><<<grid, 256, smem, st>>>(in, out, C, h, w, scale);
    else prep_kernel<8, TIn, TOut><<<grid, 256, smem, st>>>(in, out, C, h, w, scale);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

template <typename TOut>
static int launch_prep_from(const void* fmap, int in_dtype, TOut* out, int B, int C, int h, int w, int pool, float scale,
                            int HWo, cudaStream_t st) {
    if (in_dtype == OFB_DTYPE_F32) return launch_prep<float>(fmap, out, B, C, h, w, pool, scale, HWo, st);
    if (in_dtype == OFB_DTYPE_BF16) return launch_prep<__nv_bfloat16>(fmap, out, B, C, h, w, pool, scale, HWo, st);
    return launch_prep<__half>(fmap, out, B, C, h, w, pool, scale, HWo, st);
}

OFB_API int ofb_corr_prep_to(const void* fmap_nchw, int in_dtype, void* out_km, int out_dtype, int B, int C, int h, int w,
                             int pool, float scale, void* stream) {
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!fmap_nchw || !out_km || B < 0 || C <= 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (pool != 1 && pool != 2 && pool != 4 && pool != 8) return OFB_EINVAL;
    if (in_dtype != OFB_DTYPE_F32 && in_dtype != OFB_DTYPE_BF16 && in_dtype != OFB_DTYPE_F16) return OFB_EINVAL;
    if (out_dtype != OFB_DTYPE_BF16 && out_dtype != OFB_DTYPE_F16) return OFB_EINVAL;
    if (C & 1) return OFB_EUNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(out_km) & 3) return OFB_EALIGN;
    if (reinterpret_cast<uintptr_t>(fmap_nchw) & (in_dtype == OFB_DTYPE_F32 ? 3 : 1)) return OFB_EALIGN;
    const int HWo = (h / pool) * (w / pool);
    if (HWo == 0) return OFB_OK;
    if (B > 65535) return OFB_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (out_dtype == OFB_DTYPE_F16)
        return launch_prep_from(fmap_nchw, in_dtype, reinterpret_cast<__half*>(out_km), B, C, h, w, pool, scale, HWo, st);
    return launch_prep_from(fmap_nchw, in_dtype, reinterpret_cast<__nv_bfloat16*>(out_km), B, C, h, w, pool, scale, HWo, st);
}

OFB_API int ofb_corr_prep_from(const void* fmap_nchw, int in_dtype, void* out_km_bf16, int B, int C, int h, int w, int pool,
                               float scale, void* stream) {
    return ofb_corr_prep_to(fmap_nchw, in_dtype, out_km_bf16, OFB_DTYPE_BF16, B, C, h, w, pool, scale, stream);
}

OFB_API int ofb_corr_prep_bf16(const float* fmap_nchw, void* out_km_bf16, int B, int C, int h, int w, int pool,
                               float scale, void* stream) {
    return ofb_corr_prep_from(fmap_nchw, OFB_DTYPE_F32, out_km_bf16, B, C, h, w, pool, scale, stream);
}

OFB_API int ofb_pyramid_layout(int h, int w, int levels, int mode, ofb_pyramid* pyr, int64_t elems[OFB_MAX_LEVELS]) {
    if (!pyr || h <= 0 || w <= 0 || levels < 1 || levels > OFB_MAX_LEVELS || mode < 0 || mode > 3) return OFB_EINVAL;
    pyr->levels = levels;
    pyr->layout = mode == 2 ? OFB_LAYOUT_BLOCK8X4 : mode == 3 ? OFB_LAYOUT_QMINOR8X4 : OFB_LAYOUT_ROWS;
    pyr->reserved = 0;
    for (int l = 0; l < OFB_MAX_LEVELS; ++l) {
        pyr->base[l] = nullptr;
        pyr->q_stride[l] = 0; pyr->row_pitch[l] = 0; pyr->lvl_h[l] = 0; pyr->lvl_w[l] = 0;
        if (elems) elems[l] = 0;
    }
    for (int l = 0; l < levels; ++l) {
        const int hl = h >> l, wl = w >> l;
        if (hl <= 0 || wl <= 0) return OFB_EINVAL;   // F.avg_pool2d raises "Output size is too small" (corr.py:53)
        // padded rows start on 32-byte sectors (bf16); 8x4 blocks are 64-byte aligned by construction
        const int pitch = mode == 1 ? ((wl + 15) & ~15) : mode >= 2 ? ((wl + 7) & ~7) : wl;
        const int rows = mode >= 2 ? ((hl + 3) & ~3) : hl;
        pyr->lvl_h[l] = hl; pyr->lvl_w[l] = wl; pyr->row_pitch[l] = pitch;
        pyr->q_stride[l] = mode == 3 ? 32 : (int64_t)pitch * rows;
        if (elems) elems[l] = (int64_t)pitch * rows;  // per query; caller multiplies by B*h*w
    }
    return OFB_OK;
}

OFB_API int ofb_corr_pyramid_simt_f32(const float* fmap1, const float* fmap2, const ofb_pyramid* pyr, int B, int C,
                                      int h, int w, float scale, void* stream) {
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!fmap1 || !fmap2 || !pyr || B < 0 || C <= 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    ofb::PyramidView v;
    if (const int rc = ofb::check_pyramid(pyr, (long long)B * h * w, v)) return rc;
    if (v.blocked) return OFB_EUNSUPPORTED;                           // the CUDA-core builder writes rows
    for (int l = 0; l < v.levels; ++l)      // level l of the (h, w) feature maps: (h >> l) x (w >> l)
        if (v.lh[l] != (h >> l) || v.lw[l] != (w >> l)) return OFB_EINVAL;
    if (B > 65535 || (h * w + GT - 1) / GT > 65535) return OFB_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (v.dtype == OFB_DTYPE_F32) return build_simt<float>(fmap1, fmap2, v, B, C, h, w, scale, st);
    if (v.dtype == OFB_DTYPE_BF16) return build_simt<__nv_bfloat16>(fmap1, fmap2, v, B, C, h, w, scale, st);
    return build_simt<__half>(fmap1, fmap2, v, B, C, h, w, scale, st);
}
