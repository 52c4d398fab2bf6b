// warp_bwd.cu -- K1 backward: gradients of the flow-based bilinear warp with respect to the frame and the flow.
//
// The reference's warp (optical_flow/operator/operator.py:8-33) is F.grid_sample on grid = linspace + flow, so its
// backward is ATen's grid_sampler_2d_backward followed by the identity d grid / d flow (operator.py:56) and the
// (B,H,W,2) -> (B,2,H,W) permute (operator.py:28).  One pass, one thread per output pixel, lane <-> column:
//   d_frame[b,c,tap] += w_tap * d_out[b,c,i,j]                       (4 red.global.add.f32, in-bounds taps only)
//   d ix = sum_c d_out * ((v01 - v00) * wy0 + (v11 - v10) * wy1)      (evaluated in ATen's term order)
//   d iy = sum_c d_out * ((v10 - v00) * wx0 + (v11 - v01) * wx1)
//   d_flow[b,0,i,j] = flow_mul_x * (d ix * d ix/d gx),  d_flow[b,1,i,j] = flow_mul_y * (d iy * d iy/d gy)
// with d ix / d gx from the un-normalise / clip / reflect chain (ATen GridSampler.h:38-54,62-83,110-140,180-203):
// W/2 or (W-1)/2, times 0 where border padding clips, times -1 on odd reflections.
// Neither the grid nor its gradient is materialised.  HBM: reads frame + flow + d_out, writes d_flow, RMW d_frame.
#include "common.cuh"

namespace {

using namespace ofb;

// source index and d(index)/d(grid coordinate).  Its clip is not source_index's: ATen's backward keeps NaN here,
// where the forward's clip_coord maps it to 0.
template <int PAD, bool AC>
__device__ __forceinline__ float source_index_grad(float g, int size, float& grad) {
    grad = AC ? (float)(size - 1) / 2.0f : (float)size / 2.0f;
    float x = unnormalize<AC>(g, size);
    if (PAD == OFB_PAD_REFLECTION) {
        float dsign;
        x = reflect_index<AC>(x, size, &dsign);
        grad *= dsign;
    }
    if (PAD != OFB_PAD_ZEROS) {
        // borders count as out of bounds for the gradient (GridSampler.h:68-69); NaN falls to the last branch as there
        if (x <= 0.0f) { grad = 0.0f; x = 0.0f; }
        else if (x >= (float)(size - 1)) { grad = 0.0f; x = (float)(size - 1); }
    }
    return x;
}

template <int PAD, bool AC>
__global__ void __launch_bounds__(128) warp_bwd_kernel(const float* __restrict__ frame, const float* __restrict__ flow,
                                                       const float* __restrict__ d_out, float* __restrict__ d_frame,
                                                       float* __restrict__ d_flow, int C, int H, int W, FlowMul fm) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y, b = blockIdx.z;
    if (j >= W) return;
    const int HW = H * W;                                  // launch guard: H*W < 2^30
    const int off = i * W + j;
    const float* fxp = flow + (size_t)(b * 2) * HW;
    const float gx = warp_grid_coord(__ldg(fxp + off), j, W, fm.step_x, fm.x);
    const float gy = warp_grid_coord(__ldg(fxp + HW + off), i, H, fm.step_y, fm.y);
    float gmx, gmy;
    const float ix = source_index_grad<PAD, AC>(gx, W, gmx);
    const float iy = source_index_grad<PAD, AC>(gy, H, gmy);
    // the zeros form whatever the padding: the clip above can leave NaN, which has no tap in bounds
    const BilinearTaps t = bilinear_taps<OFB_PAD_ZEROS>(ix, iy, H, W);
    const float wx0 = t.wx0, wx1 = t.wx1, wy0 = t.wy0, wy1 = t.wy1;
    const bool i00 = t.inb & 1u, i01 = t.inb & 2u, i10 = t.inb & 4u, i11 = t.inb & 8u;
    const int o = t.y0 * W + t.x0;
    float gix = 0.0f, giy = 0.0f;
    for (int c = 0; c < C; ++c) {
        const size_t plane = (size_t)(b * C + c) * HW;
        const float g = __ldg(d_out + plane + off);
        if (d_frame) {
            float* p = d_frame + plane + o;
            if (i00) atomicAdd(p, t.w00 * g);
            if (i01) atomicAdd(p + 1, t.w01 * g);
            if (i10) atomicAdd(p + W, t.w10 * g);
            if (i11) atomicAdd(p + W + 1, t.w11 * g);
        }
        if (d_flow) {
            const float* p = frame + plane + o;
            if (i00) { const float v = __ldg(p); gix -= v * wy0 * g; giy -= v * wx0 * g; }
            if (i01) { const float v = __ldg(p + 1); gix += v * wy0 * g; giy -= v * wx1 * g; }
            if (i10) { const float v = __ldg(p + W); gix -= v * wy1 * g; giy += v * wx0 * g; }
            if (i11) { const float v = __ldg(p + W + 1); gix += v * wy1 * g; giy += v * wx1 * g; }
        }
    }
    if (d_flow) {
        float* dp = d_flow + (size_t)(b * 2) * HW + off;
        dp[0] = fm.x * (gmx * gix);
        dp[HW] = fm.y * (gmy * giy);
    }
}

template <int PAD, bool AC>
int launch(const float* frame, const float* flow, const float* d_out, float* d_frame, float* d_flow, int B, int C, int H,
           int W, const FlowMul& fm, cudaStream_t stream) {
    const dim3 grid((W + 127) / 128, H, B);
    warp_bwd_kernel<PAD, AC><<<grid, 128, 0, stream>>>(frame, flow, d_out, d_frame, d_flow, C, H, W, fm);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

}  // namespace

OFB_API int ofb_warp_backward_f32(const float* frame, const float* flow, const float* d_out, float* d_frame_or_null,
                                  float* d_flow_or_null, int B, int C, int H, int W, int padding_mode, int align_corners,
                                  float flow_mul_x, float flow_mul_y, void* stream) {
    if (B == 0 || H == 0 || W == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!frame || !flow || !d_out || B < 0 || C < 0 || H < 0 || W < 0) return OFB_EINVAL;
    if (padding_mode < 0 || padding_mode > 2) return OFB_EINVAL;
    if ((size_t)B * H * W == 0 || (!d_frame_or_null && !d_flow_or_null)) return OFB_OK;
    if (B > 65535 || H > 65535 || (long long)H * W >= (1LL << 30) || (long long)B * (C > 2 ? C : 2) * H * W >= (1LL << 40))
        return OFB_EUNSUPPORTED;
    const ofb::FlowMul fm{flow_mul_x, flow_mul_y, ofb::linspace_step(W), ofb::linspace_step(H)};
    return ofb_dispatch_pad_ac(padding_mode, align_corners != 0, [&](auto P, auto A) {
        return launch<P, A>(frame, flow, d_out, d_frame_or_null, d_flow_or_null, B, C, H, W, fm, (cudaStream_t)stream);
    });
}
