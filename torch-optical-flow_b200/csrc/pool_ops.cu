// pool_ops.cu -- the two small passes around the backward GEMMs of CorrBlock (training path, SURVEY.md 8f row 3).
//
// The pyramid is linear in the feature maps: level l = fmap1^T . avgpool_l(fmap2) / sqrt(C) (reference corr.py:45-54,
// avg_pool2d being linear).  Its backward therefore needs
//   (1) the B operand of  d fmap1 += dP_l . avgpool_l(fmap2)^T : the pooled map as (B, C, K) bf16 with K = h_l*w_l padded
//       to the GEMM's pitch -- ofb_pool_cast_bf16 (replaces an avg_pool2d chain, a cast and a zero-fill + slice copy);
//   (2) the adjoint of the pooling for  d fmap2 = sum_l avgpool_l^T( d avgpool_l(fmap2) ) : every pixel of a complete
//       2^l x 2^l block receives 1/4^l of the block's gradient, pixels the floor cropped receive nothing
//       (what autograd computes through the avg_pool2d chain) -- ofb_pool_adjoint_f32, which also turns the GEMMs'
//       (B, N_l, C) outputs into the (B, C, h, w) layout of the feature map in the same pass.
#include "common.cuh"

namespace {

// out[b, c, k] = bf16(mean of the pool x pool block k of fmap[b, c]) for k < (h/pool)*(w/pool), 0 for the padding
template <typename TIn>
__global__ void __launch_bounds__(256) pool_cast_kernel(const TIn* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                        long long planes, int h, int w, int pool, int nk, int pk) {
    const int wo = w / pool;
    const float inv = 1.0f / (float)(pool * pool);
    const long long total = planes * pk;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long plane = t / pk;
        const int k = (int)(t - plane * pk);
        float v = 0.0f;
        if (k < nk) {
            const int yo = k / wo, xo = k - yo * wo;
            const TIn* src = in + plane * (long long)h * w + (long long)(yo * pool) * w + xo * pool;
            float a = 0.0f;
            for (int dy = 0; dy < pool; ++dy)
                for (int dx = 0; dx < pool; ++dx) a += ofb::ld_f32(src + dy * w + dx);
            v = a * inv;
        }
        out[t] = __float2bfloat16_rn(v);
    }
}

struct AdjParams {
    const float* lvl[OFB_MAX_LEVELS];   // (B, n_l, C) fp32
    int lh[OFB_MAX_LEVELS], lw[OFB_MAX_LEVELS];
    int levels, C, h, w;
};

// out[b, c, y, x] = sum_l [y>>l < h_l and x>>l < w_l] lvl_l[b, (y>>l)*w_l + (x>>l), c] / 4^l
// 32 pixels x 32 channels per CTA: reads are coalesced over channels, writes over pixels (shared-memory transpose).
__global__ void __launch_bounds__(256) pool_adjoint_kernel(const AdjParams P, float* __restrict__ out) {
    __shared__ float tile[32][33];
    const int hw = P.h * P.w;
    const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 x 8 threads
    for (int r = ty; r < 32; r += 8) {
        const int p = p0 + r, c = c0 + tx;
        float acc = 0.0f;
        if (p < hw && c < P.C) {
            const int y = p / P.w, x = p - y * P.w;
            float wgt = 1.0f;
            for (int l = 0; l < P.levels; ++l, wgt *= 0.25f) {
                const int yl = y >> l, xl = x >> l;
                if (yl < P.lh[l] && xl < P.lw[l])
                    acc += wgt * __ldg(P.lvl[l] + ((long long)b * P.lh[l] * P.lw[l] + (long long)yl * P.lw[l] + xl) * P.C + c);
            }
        }
        tile[r][tx] = acc;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, p = p0 + tx;
        if (c < P.C && p < hw) out[((long long)b * P.C + c) * hw + p] = tile[tx][r];
    }
}

template <typename TIn>
int launch_pool_cast(const void* fmap, void* out, long long planes, int h, int w, int pool, int nk, int pk, cudaStream_t st) {
    long long blocks = (planes * pk + 255) / 256;
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    pool_cast_kernel<TIn><<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const TIn*>(fmap), reinterpret_cast<__nv_bfloat16*>(out),
                                                       planes, h, w, pool, nk, pk);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

}  // namespace

OFB_API int ofb_pool_cast_bf16(const void* fmap_nchw, int in_dtype, void* out_bck_bf16, int B, int C, int h, int w, int pool,
                               int pitch_k, void* stream) {
    if (B == 0 || C == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!fmap_nchw || !out_bck_bf16 || B < 0 || C < 0 || h <= 0 || w <= 0 || pool < 1) return OFB_EINVAL;
    const int nk = (h / pool) * (w / pool);
    if (pitch_k < nk || pitch_k <= 0) return OFB_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const long long planes = (long long)B * C;
    if (in_dtype == OFB_DTYPE_F32) return launch_pool_cast<float>(fmap_nchw, out_bck_bf16, planes, h, w, pool, nk, pitch_k, st);
    if (in_dtype == OFB_DTYPE_BF16) return launch_pool_cast<__nv_bfloat16>(fmap_nchw, out_bck_bf16, planes, h, w, pool, nk, pitch_k, st);
    if (in_dtype == OFB_DTYPE_F16) return launch_pool_cast<__half>(fmap_nchw, out_bck_bf16, planes, h, w, pool, nk, pitch_k, st);
    return OFB_EINVAL;
}

OFB_API int ofb_pool_adjoint_f32(const float* const* d_levels_bnc, float* d_fmap_nchw, int B, int C, int h, int w, int levels,
                                 void* stream) {
    if (B == 0 || C == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!d_levels_bnc || !d_fmap_nchw || B < 0 || C < 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (levels < 1 || levels > OFB_MAX_LEVELS) return OFB_EINVAL;
    if (B > 65535 || (C + 31) / 32 > 65535) return OFB_EUNSUPPORTED;
    AdjParams P = {};
    for (int l = 0; l < levels; ++l) {
        if (!d_levels_bnc[l] || (h >> l) <= 0 || (w >> l) <= 0) return OFB_EINVAL;
        P.lvl[l] = d_levels_bnc[l];
        P.lh[l] = h >> l; P.lw[l] = w >> l;
    }
    P.levels = levels; P.C = C; P.h = h; P.w = w;
    const dim3 grid((h * w + 31) / 32, (C + 31) / 32, B);
    pool_adjoint_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(P, d_fmap_nchw);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
