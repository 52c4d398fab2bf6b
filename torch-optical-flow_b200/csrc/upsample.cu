// upsample.cu -- K4b: RAFT convex 8x flow upsampling in one pass.
//
// Replaces RAFT.upsample_flow (reference methods/raft/model/raft.py:73-85):
//   out[n,c,8y+i,8x+j] = sum_k softmax_k(mask[n, k*64 + i*8 + j, y, x]) * 8*flow_pad[n,c,y+ky-1,x+kx-1]
// with k = ky*3+kx over the zero-padded 3x3 neighbourhood.  The reference materialises the
// softmax (B,1,9,8,8,h,w), the unfolded flow (9x) and their product (9x the output); here
// nothing but the 576-channel mask is read and the upsampled flow written.
//
// Mapping: thread = (coarse pixel p = y*w+x, sub-row i).  Mask planes are contiguous over p,
// so every mask load of a warp is a full 128-byte line; each thread produces the eight
// consecutive outputs j = 0..7 of fine row 8y+i (two 16-byte stores per flow component).
// HBM roofline: 4*(576 + 2) bytes read + 4*128 bytes written per coarse pixel.
#include "common.cuh"

namespace {

constexpr int PX = 32;   // coarse pixels per CTA
constexpr int NT = PX * 8;

template <typename TM>
__global__ void __launch_bounds__(NT) convex_upsample_kernel(const float* __restrict__ flow,
                                                             const TM* __restrict__ mask,
                                                             float* __restrict__ out, int N, int h, int w) {
    const int hw = h * w;
    const int lane_p = threadIdx.x % PX;
    const int i = threadIdx.x / PX;                     // sub-row 0..7 (warp-uniform)
    const int n = blockIdx.y;
    const int p = blockIdx.x * PX + lane_p;
    if (p >= hw) return;
    const int y = p / w, x = p - y * w;

    // 3x3 neighbourhood of 8*flow, zero padded (F.unfold(8*flow, 3, padding=1))
    float nbx[9], nby[9];
    const float* fx = flow + (size_t)n * 2 * hw;
    const float* fy = fx + hw;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int yy = y + ky - 1, xx = x + kx - 1;
            const bool in = yy >= 0 && yy < h && xx >= 0 && xx < w;
            nbx[ky * 3 + kx] = in ? 8.0f * __ldg(fx + yy * w + xx) : 0.0f;
            nby[ky * 3 + kx] = in ? 8.0f * __ldg(fy + yy * w + xx) : 0.0f;
        }

    // mask logits: fp32, or half precision under the reference's `precision: 16` (autocast convolution; softmax
    // itself autocasts to fp32, raft.py:78)
    const TM* mp = mask + (size_t)n * 576 * hw + (size_t)(i * 8) * hw + p;
    float ox[8], oy[8];
    // JG sub-columns at a time: 9*JG independent 128-byte-coalesced loads are in flight per warp before
    // the first softmax starts (the kernel is a pure stream of the 576-channel mask: latency, not math)
    constexpr int JG = 4;
#pragma unroll
    for (int jg = 0; jg < 8; jg += JG) {
        float m[JG][9];
#pragma unroll
        for (int jj = 0; jj < JG; ++jj)
#pragma unroll
            for (int k = 0; k < 9; ++k) m[jj][k] = ofb::ld_f32(mp + (size_t)(k * 64 + jg + jj) * hw);
#pragma unroll
        for (int jj = 0; jj < JG; ++jj) {
            float mx = m[jj][0];
#pragma unroll
            for (int k = 1; k < 9; ++k) mx = fmaxf(mx, m[jj][k]);
            float s = 0.0f;
#pragma unroll
            for (int k = 0; k < 9; ++k) { m[jj][k] = expf(m[jj][k] - mx); s += m[jj][k]; }
            // softmax-weighted sums, normalised once at the end: sum_k e_k v_k / sum_k e_k (one division per
            // component instead of nine; differs from the reference's per-weight division by <= 2 ulp)
            float ax = 0.0f, ay = 0.0f;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                ax = __fmaf_rn(m[jj][k], nbx[k], ax);
                ay = __fmaf_rn(m[jj][k], nby[k], ay);
            }
            const float inv = __fdiv_rn(1.0f, s);
            ox[jg + jj] = ax * inv; oy[jg + jj] = ay * inv;
        }
    }
    const size_t W8 = (size_t)8 * w, H8 = (size_t)8 * h;
    float* dx = out + ((size_t)n * 2 + 0) * H8 * W8 + (size_t)(8 * y + i) * W8 + 8 * x;
    float* dy = dx + H8 * W8;
    // rows are 8*w floats and x offsets multiples of 8 -> 32-byte aligned
    reinterpret_cast<float4*>(dx)[0] = make_float4(ox[0], ox[1], ox[2], ox[3]);
    reinterpret_cast<float4*>(dx)[1] = make_float4(ox[4], ox[5], ox[6], ox[7]);
    reinterpret_cast<float4*>(dy)[0] = make_float4(oy[0], oy[1], oy[2], oy[3]);
    reinterpret_cast<float4*>(dy)[1] = make_float4(oy[4], oy[5], oy[6], oy[7]);
}

// Backward of the convex upsampling (what autograd computes through softmax, unfold and the weighted sum of
// raft.py:77-85).  With p_k = softmax_k(mask), v_k = 8*flow_pad (3x3 neighbourhood) and g = d_out at the fine pixel:
//   a_k = g_x v_k,x + g_y v_k,y ;  d_mask_k = p_k (a_k - sum_m p_m a_m)
//   S_k(p) = sum_{i,j} p_k(p;i,j) g(p;i,j) ;  d_flow[q] += 8 * sum_k S_k(q - off_k),  off_k = (ky-1, kx-1)
// Deterministic: the same bits on every run.  Every d_flow element gathers its nine sums in fixed k order and is
// written by one thread, so no two threads add to the same address.  A CTA owns a TX x TY tile of coarse pixels and
// recomputes S for a one-pixel halo ring around it (BX x BY pixels in all, one warp per row, lane = column: each mask
// load of a warp is 32 consecutive elements of one plane).  A thread sums its pixel's eight sub-rows and eight
// sub-columns in order (i outer, j inner), keeps S in shared memory, writes d_mask for tile pixels only and, after
// one barrier, adds 8 * sum_k S_k(q - off_k) to d_flow[q].  The halo re-reads ~20 % more mask and d_out than the tile
// alone (30 x 14 tile: 32 * 16 / (30 * 14) = 1.22); without d_flow the halo is skipped.
// The mask and d_mask share the element type TM, as in the forward: a 16-bit logit is widened exactly, d_mask is
// computed in fp32 and rounded once (ofb::narrow), the bits of the fp32 gradient cast to the mask's dtype -- what
// autocast's cast backward hands the mask head.  d_out, flow and d_flow stay fp32 (the upsampled flow is fp32).
constexpr int BX = 32, BY = 16;            // tile with its halo ring
constexpr int TX = BX - 2, TY = BY - 2;    // pixels whose d_mask and d_flow the CTA writes
constexpr int NTB = BX * BY;

template <typename TM>
__global__ void __launch_bounds__(NTB, 1) convex_upsample_bwd_kernel(const float* __restrict__ flow,
                                                                     const TM* __restrict__ mask,
                                                                     const float* __restrict__ d_out,
                                                                     float* __restrict__ d_flow, TM* __restrict__ d_mask,
                                                                     int N, int h, int w, int tiles_x) {
    __shared__ float s_sum[2][9][BY][BX];
    const int hw = h * w;
    const int lx = threadIdx.x % BX, ly = threadIdx.x / BX;
    const int n = blockIdx.y;
    const int x = (int)(blockIdx.x % tiles_x) * TX + lx - 1;
    const int y = (int)(blockIdx.x / tiles_x) * TY + ly - 1;
    const bool in_img = x >= 0 && x < w && y >= 0 && y < h;
    const bool own = in_img && lx >= 1 && lx <= TX && ly >= 1 && ly <= TY;
    float sx[9], sy[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) sx[k] = sy[k] = 0.0f;   // pixels outside the frame contribute nothing
    if (own || (in_img && d_flow)) {
        const int p = y * w + x;
        float nbx[9], nby[9];
        const float* fx = flow + (size_t)n * 2 * hw;
        const float* fy = fx + hw;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int yy = y + ky - 1, xx = x + kx - 1;
                const bool in = yy >= 0 && yy < h && xx >= 0 && xx < w;
                nbx[ky * 3 + kx] = in ? 8.0f * __ldg(fx + yy * w + xx) : 0.0f;
                nby[ky * 3 + kx] = in ? 8.0f * __ldg(fy + yy * w + xx) : 0.0f;
            }
        const size_t W8 = (size_t)8 * w, H8 = (size_t)8 * h;
        TM* dm = own ? d_mask : nullptr;
#pragma unroll 1
        for (int i = 0; i < 8; ++i) {
            const float* gxp = d_out + ((size_t)n * 2 + 0) * H8 * W8 + (size_t)(8 * y + i) * W8 + 8 * x;
            const float* gyp = gxp + H8 * W8;
            float gx[8], gy[8];
            {
                const float4 a = __ldg(reinterpret_cast<const float4*>(gxp)), b = __ldg(reinterpret_cast<const float4*>(gxp) + 1);
                const float4 c = __ldg(reinterpret_cast<const float4*>(gyp)), d = __ldg(reinterpret_cast<const float4*>(gyp) + 1);
                gx[0] = a.x; gx[1] = a.y; gx[2] = a.z; gx[3] = a.w; gx[4] = b.x; gx[5] = b.y; gx[6] = b.z; gx[7] = b.w;
                gy[0] = c.x; gy[1] = c.y; gy[2] = c.z; gy[3] = c.w; gy[4] = d.x; gy[5] = d.y; gy[6] = d.z; gy[7] = d.w;
            }
            const size_t moff = (size_t)n * 576 * hw + (size_t)(i * 8) * hw + p;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float m[9];
#pragma unroll
                for (int k = 0; k < 9; ++k) m[k] = ofb::ld_f32(mask + moff + (size_t)(k * 64 + j) * hw);
                float mx = m[0];
#pragma unroll
                for (int k = 1; k < 9; ++k) mx = fmaxf(mx, m[k]);
                float s = 0.0f;
#pragma unroll
                for (int k = 0; k < 9; ++k) { m[k] = expf(m[k] - mx); s += m[k]; }
                const float inv = __fdiv_rn(1.0f, s);
                float a[9], dot = 0.0f;
#pragma unroll
                for (int k = 0; k < 9; ++k) {
                    m[k] *= inv;
                    a[k] = __fmaf_rn(gx[j], nbx[k], gy[j] * nby[k]);
                    dot = __fmaf_rn(m[k], a[k], dot);
                    sx[k] = __fmaf_rn(m[k], gx[j], sx[k]);
                    sy[k] = __fmaf_rn(m[k], gy[j], sy[k]);
                }
                if (dm) {
#pragma unroll
                    for (int k = 0; k < 9; ++k) dm[moff + (size_t)(k * 64 + j) * hw] = ofb::narrow<TM>(m[k] * (a[k] - dot));
                }
            }
        }
    }
    if (!d_flow) return;   // uniform over the CTA
#pragma unroll
    for (int k = 0; k < 9; ++k) { s_sum[0][k][ly][lx] = sx[k]; s_sum[1][k][ly][lx] = sy[k]; }
    __syncthreads();
    if (!own) return;
    float ax = 0.0f, ay = 0.0f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {   // q is neighbour k of p = q - off_k
            ax += s_sum[0][ky * 3 + kx][ly + 1 - ky][lx + 1 - kx];
            ay += s_sum[1][ky * 3 + kx][ly + 1 - ky][lx + 1 - kx];
        }
    float* dfx = d_flow + (size_t)n * 2 * hw + y * w + x;
    dfx[0] += 8.0f * ax;
    dfx[hw] += 8.0f * ay;
}

}  // namespace

OFB_API int ofb_convex_upsample(const float* flow, const void* mask, int mask_dtype, float* out, int N, int h, int w,
                                void* stream) {
    if (N == 0 || h == 0 || w == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!flow || !mask || !out || N < 0 || h < 0 || w < 0) return OFB_EINVAL;
    if (mask_dtype != OFB_DTYPE_F32 && mask_dtype != OFB_DTYPE_BF16 && mask_dtype != OFB_DTYPE_F16) return OFB_EINVAL;
    if ((size_t)N * h * w == 0) return OFB_OK;
    if (N > 65535) return OFB_EUNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(out) & 15) return OFB_EALIGN;
    if (reinterpret_cast<uintptr_t>(mask) & (mask_dtype == OFB_DTYPE_F32 ? 3 : 1)) return OFB_EALIGN;
    dim3 grid((h * w + PX - 1) / PX, N);
    cudaStream_t st = (cudaStream_t)stream;
    if (mask_dtype == OFB_DTYPE_F32)
        convex_upsample_kernel<float><<<grid, NT, 0, st>>>(flow, reinterpret_cast<const float*>(mask), out, N, h, w);
    else if (mask_dtype == OFB_DTYPE_BF16)
        convex_upsample_kernel<__nv_bfloat16><<<grid, NT, 0, st>>>(flow, reinterpret_cast<const __nv_bfloat16*>(mask), out, N, h, w);
    else
        convex_upsample_kernel<__half><<<grid, NT, 0, st>>>(flow, reinterpret_cast<const __half*>(mask), out, N, h, w);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_convex_upsample_f32(const float* flow, const float* mask, float* out, int N, int h, int w, void* stream) {
    return ofb_convex_upsample(flow, mask, OFB_DTYPE_F32, out, N, h, w, stream);
}

OFB_API int ofb_convex_upsample_backward(const float* flow, const void* mask, int mask_dtype, const float* d_out,
                                         float* d_flow_or_null, void* d_mask_or_null, int N, int h, int w, void* stream) {
    if (!ofb_float_dtype(mask_dtype)) return OFB_EINVAL;
    if (N == 0 || h == 0 || w == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!flow || !mask || !d_out || N < 0 || h < 0 || w < 0) return OFB_EINVAL;
    if ((size_t)N * h * w == 0 || (!d_flow_or_null && !d_mask_or_null)) return OFB_OK;
    if (N > 65535) return OFB_EUNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(d_out) & 15) return OFB_EALIGN;
    const uintptr_t elem = mask_dtype == OFB_DTYPE_F32 ? 3 : 1;
    if ((reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(d_mask_or_null)) & elem) return OFB_EALIGN;
    const int tiles_x = (w + TX - 1) / TX;
    dim3 grid(tiles_x * ((h + TY - 1) / TY), N);
    return ofb_dispatch_dtype(mask_dtype, [&](auto t) {
        using TM = decltype(t);
        convex_upsample_bwd_kernel<TM><<<grid, NTB, 0, (cudaStream_t)stream>>>(
            flow, static_cast<const TM*>(mask), d_out, d_flow_or_null, static_cast<TM*>(d_mask_or_null), N, h, w, tiles_x);
        OFB_LAUNCH_CHECK();
        return OFB_OK;
    });
}

OFB_API int ofb_convex_upsample_backward_f32(const float* flow, const float* mask, const float* d_out,
                                             float* d_flow_or_null, float* d_mask_or_null, int N, int h, int w,
                                             void* stream) {
    return ofb_convex_upsample_backward(flow, mask, OFB_DTYPE_F32, d_out, d_flow_or_null, d_mask_or_null, N, h, w, stream);
}
