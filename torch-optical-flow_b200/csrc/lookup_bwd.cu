// lookup_bwd.cu -- K3 backward: gradient of the correlation lookup with respect to the pyramid.
//
// The reference's CorrBlock.__call__ (methods/raft/model/corr.py:56-77) samples every level with
// bilinear_sampler = F.grid_sample(align_corners=True, zeros padding) (utils.py:64-80); its backward with respect
// to the sampled image scatters weight * grad into the four taps of every sample.  RAFT detaches the coordinates
// (raft.py:127), so only d / d pyramid is produced.
//
// thread = (query, level), lane <-> query (d_out reads are 128-byte rows).  A (query, level) slice is touched by
// exactly one thread per launch, so the accumulation into the fp32 gradient pyramid needs no atomicity; it is
// still issued as red.global.add.f32 (result unused): one fire-and-forget operation per element instead of a load
// + store round trip (measured 0.75 -> 0.40 ms per iteration at C4).  The 12 refinement iterations accumulate
// into the same buffer, launch after launch.
//   * regular windows (taps on consecutive integer positions -- all but coordinates on rounding boundaries): the
//     (2r+1)^2 gradients are pushed through the separable 2-tap filters in registers, one output row at a time:
//       T[j][c]  = g[c][j] * w0x[c] + g[c-1][j] * w1x[c-1]            (x pass; the window is transposed: i moves x)
//       dP[r][c] += T[r][c] * w0y[r] + T[r-1][c] * w1y[r-1]           (y pass)
//     i.e. (2r+2)^2 accumulations in 2r+2 short rows instead of 4 (2r+1)^2 scattered ones;
//   * anything else: the direct 4-tap scatter.
// The tap positions and weights are the forward kernels' (ofb::lookup_tap, common.cuh).
#include "common.cuh"

namespace {

struct BwdParams : ofb::PyramidLevels {
    int levels, B, h, w;
};

struct Tap {
    int i0;
    float w0, w1;
};

// one axis, one window offset; a tap outside the guard gets index TAP_FAR and zero weights
__device__ __forceinline__ Tap make_tap(float cen, int t, int radius, int size) {
    const ofb::LookupTap tp = ofb::lookup_tap(cen, t, radius, size);
    return tp.in_guard ? Tap{(int)tp.fl, tp.w0, tp.w1} : Tap{ofb::TAP_FAR, 0.0f, 0.0f};
}

template <int R>
__global__ void __launch_bounds__(128) lookup_bwd_kernel(const __grid_constant__ BwdParams P, const float* __restrict__ coords,
                                                         const float* __restrict__ d_out) {
    constexpr int D = 2 * R + 1, DD = D * D;
    const long long HW = (long long)P.h * P.w, Q = (long long)P.B * HW;
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int l = blockIdx.y;
    if (q >= Q) return;
    const long long b = q / HW, p = q - b * HW;
    const int Wl = P.lw[l], Hl = P.lh[l], pitch = P.pitch[l];
    float* slice = static_cast<float*>(P.base[l]) + q * P.q_stride[l];
    const float inv = 1.0f / (float)(1 << l);
    const float cx = __fmul_rn(__ldg(coords + (b * 2 + 0) * HW + p), inv);
    const float cy = __fmul_rn(__ldg(coords + (b * 2 + 1) * HW + p), inv);
    const float* g0 = d_out + (b * (long long)(P.levels * DD) + (long long)l * DD) * HW + p;   // channel c at g0[c * HW]

    float wx0[D], wx1[D], wy0[D], wy1[D];
    int ax = 0, ay = 0;
    bool regular = true;
#pragma unroll
    for (int t = 0; t < D; ++t) {
        const Tap tx = make_tap(cx, t, R, Wl), ty = make_tap(cy, t, R, Hl);
        wx0[t] = tx.w0; wx1[t] = tx.w1; wy0[t] = ty.w0; wy1[t] = ty.w1;
        if (t == 0) { ax = tx.i0; ay = ty.i0; }
        regular = regular && tx.i0 != ofb::TAP_FAR && ty.i0 != ofb::TAP_FAR && tx.i0 == ax + t && ty.i0 == ay + t;
    }

    if (regular) {
        float tprev[D + 1];
#pragma unroll
        for (int c = 0; c <= D; ++c) tprev[c] = 0.0f;
#pragma unroll
        for (int j = 0; j <= D; ++j) {
            float tcur[D + 1];
#pragma unroll
            for (int c = 0; c <= D; ++c) tcur[c] = 0.0f;
            if (j < D) {
                float g[D];
#pragma unroll
                for (int i = 0; i < D; ++i) g[i] = __ldg(g0 + (long long)(i * D + j) * HW);
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    tcur[c] = __fmaf_rn(g[c], wx0[c], tcur[c]);
                    tcur[c + 1] = __fmaf_rn(g[c], wx1[c], tcur[c + 1]);
                }
            }
            const int y = ay + j;
            if (y >= 0 && y < Hl) {
                float* row = slice + (long long)y * pitch + ax;
#pragma unroll
                for (int c = 0; c <= D; ++c) {
                    float v = 0.0f;
                    if (j < D) v = tcur[c] * wy0[j < D ? j : 0];
                    if (j > 0) v = __fmaf_rn(tprev[c], wy1[j > 0 ? j - 1 : 0], v);
                    const int x = ax + c;
                    if (x >= 0 && x < Wl) atomicAdd(row + c, v);
                }
            }
#pragma unroll
            for (int c = 0; c <= D; ++c) tprev[c] = tcur[c];
        }
        return;
    }
    // irregular window: direct scatter, taps recomputed per sample (no dynamically indexed register arrays)
#pragma unroll 1
    for (int j = 0; j < D; ++j) {
        const Tap ty = make_tap(cy, j, R, Hl);
        if (ty.i0 == ofb::TAP_FAR) continue;
#pragma unroll 1
        for (int i = 0; i < D; ++i) {
            const Tap tx = make_tap(cx, i, R, Wl);
            if (tx.i0 == ofb::TAP_FAR) continue;
            const float g = __ldg(g0 + (long long)(i * D + j) * HW);
            const bool inx0 = tx.i0 >= 0 && tx.i0 < Wl, inx1 = tx.i0 + 1 >= 0 && tx.i0 + 1 < Wl;
            const bool iny0 = ty.i0 >= 0 && ty.i0 < Hl, iny1 = ty.i0 + 1 >= 0 && ty.i0 + 1 < Hl;
            float* r0 = slice + (long long)ty.i0 * pitch + tx.i0;
            float* r1 = r0 + pitch;
            if (iny0 && inx0) atomicAdd(r0, g * tx.w0 * ty.w0);
            if (iny0 && inx1) atomicAdd(r0 + 1, g * tx.w1 * ty.w0);
            if (iny1 && inx0) atomicAdd(r1, g * tx.w0 * ty.w1);
            if (iny1 && inx1) atomicAdd(r1 + 1, g * tx.w1 * ty.w1);
        }
    }
}

}  // namespace

OFB_API int ofb_corr_lookup_backward_f32(const ofb_pyramid* d_pyr, const float* coords, const float* d_out, int B, int h,
                                         int w, int radius, void* stream) {
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!d_pyr || !coords || !d_out || B < 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (d_pyr->dtype != OFB_DTYPE_F32 || d_pyr->layout != OFB_LAYOUT_ROWS) return OFB_EUNSUPPORTED;
    if (radius < 0 || radius > 4) return OFB_EUNSUPPORTED;
    BwdParams P;
    if (const int rc = ofb::unpack_levels(*d_pyr, P)) return rc;
    P.levels = d_pyr->levels; P.B = B; P.h = h; P.w = w;
    const long long Q = (long long)B * h * w;
    const long long blocks = (Q + 127) / 128;
    if (blocks > 0x7fffffffLL) return OFB_EUNSUPPORTED;
    const dim3 grid((unsigned)blocks, (unsigned)d_pyr->levels);
    cudaStream_t st = (cudaStream_t)stream;
    switch (radius) {
        case 0: lookup_bwd_kernel<0><<<grid, 128, 0, st>>>(P, coords, d_out); break;
        case 1: lookup_bwd_kernel<1><<<grid, 128, 0, st>>>(P, coords, d_out); break;
        case 2: lookup_bwd_kernel<2><<<grid, 128, 0, st>>>(P, coords, d_out); break;
        case 3: lookup_bwd_kernel<3><<<grid, 128, 0, st>>>(P, coords, d_out); break;
        default: lookup_bwd_kernel<4><<<grid, 128, 0, st>>>(P, coords, d_out); break;
    }
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
