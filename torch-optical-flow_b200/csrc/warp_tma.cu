// warp_tma.cu -- K1, TMA-staged variant: the sampled neighbourhood of a 64x16 output tile is brought into shared
// memory by the copy engine, the bilinear gather then runs on shared memory.
//
// Same arithmetic as warp.cu's row kernel (reference optical_flow/operator/operator.py:8-56 -> F.grid_sample);
// what changes is where the four taps come from:
//   * a producer lane reads the flow at the tile centre, turns it into the tile's integer displacement (dx, dy)
//     and issues one 3-D TMA box per channel: [WIN_W x WIN_H x 1] of the frame viewed as (W, H, B*C), anchored
//     at tile origin + (dx, dy) - MARGIN.  Out-of-image parts of the box are zero-filled by the TMA unit, which
//     is exactly what zeros padding samples there and is multiplied by a zero weight under border / reflection.
//   * the CTAs are persistent with two window slots: the producer fills one while the 8 consumer warps (who
//     loaded their four flow vectors a tile ahead) run the coordinate pipeline and gather from the other.
//   * a pixel whose taps leave the window (|flow - centre flow| > MARGIN) falls back to the global gather of
//     the row kernel, so the result never depends on the staging.
// HBM sees every frame line about once (neighbouring windows overlap in L2); L1 sees 4 shared-memory
// wavefronts per channel per warp instead of up to 4 x 32 sector requests.
#include "sm100.cuh"

namespace {

using namespace ofb;

constexpr int TW = 64, TH = 16, NT = 256, RPT = 4;     // 64 columns x 4 row groups, 4 rows per thread
constexpr int MARGIN = 8;
constexpr int WIN_W = 84;                                // TW + 2*MARGIN + 1, rounded up to 16 bytes
constexpr int WIN_H = TH + 2 * MARGIN + 1;               // 33
constexpr int PLANE_BYTES = ((WIN_W * WIN_H * 4 + 127) / 128) * 128;
constexpr int PLANE = PLANE_BYTES / 4;
constexpr int CGRP = 4;                                  // channels staged per pipeline slot
constexpr int STAGES = 2;

struct TileCoord {
    int b, tile_x, tile_y;
};
__device__ __forceinline__ TileCoord decode_tile(int t, int ntx, int nty) {
    TileCoord tc;
    tc.b = t / (ntx * nty);
    const int r = t - tc.b * (ntx * nty);
    const int ty = r / ntx;
    tc.tile_y = ty * TH;
    tc.tile_x = (r - ty * ntx) * TW;
    return tc;
}

// Persistent CTAs: 8 consumer warps (64 columns x 4 row groups, 4 rows per thread) + 1 producer warp that runs
// one pipeline slot ahead: it reads the next tile's centre flow, derives the window origin and issues the TMA
// boxes while the consumers gather from the other slot.  full[s] / empty[s] mbarriers hand the slots over.
template <int PAD, bool AC>
__global__ void __launch_bounds__(NT + 32, 3) warp_tma_kernel(const __grid_constant__ CUtensorMap map,
                                                              const float* __restrict__ frame,
                                                              const float* __restrict__ flow, float* __restrict__ out,
                                                              uint8_t* __restrict__ valid, int C, int H, int W, int ntx,
                                                              int nty, int ntiles, FlowMul fm) {
    extern __shared__ __align__(128) float win[];    // [STAGES][cgmax][PLANE]
    __shared__ __align__(8) unsigned long long s_full[STAGES], s_empty[STAGES];
    __shared__ int s_org[STAGES][2];
    const int HW = H * W;                                  // launch guard: H*W < 2^30
    const int cgmax = min(CGRP, C);
    const int ngrp = (C + CGRP - 1) / CGRP;
    const uint32_t stage_bytes = (uint32_t)cgmax * PLANE_BYTES;
    const uint32_t win_s = smem_u32(win);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&s_full[s]), 1); mbar_init(smem_u32(&s_empty[s]), NT / 32); }
        fence_barrier_init();
    }
    __syncthreads();

    if (threadIdx.x >= NT) {
        // ------------------------------------------------------------------ producer (one lane)
        if (threadIdx.x != NT) return;
        int slot = 0;
        uint32_t ph = 0;
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
            const TileCoord tc = decode_tile(t, ntx, nty);
            // the tile's displacement: where the centre pixel samples from, relative to itself
            const int ic = min(tc.tile_y + TH / 2, H - 1), jc = min(tc.tile_x + TW / 2, W - 1);
            const float* fxp = flow + (size_t)(tc.b * 2) * HW;
            const SrcPos sc =
                warp_source<PAD, AC>(__ldg(fxp + ic * W + jc), __ldg(fxp + HW + ic * W + jc), ic, jc, H, W, fm);
            // NaN -> 0 displacement; far-out coordinates are clamped (their pixels take the fallback anyway)
            const int dx = (int)floorf(fminf(fmaxf(sc.ix - (float)jc, -1.0e6f), 1.0e6f));
            const int dy = (int)floorf(fminf(fmaxf(sc.iy - (float)ic, -1.0e6f), 1.0e6f));
            // measured on sm_100a: an un-swizzled fp32 box whose first in-bounds element is not 16-byte aligned
            // in global memory faults (illegal instruction), so the window starts on a multiple of 4 columns --
            // WIN_W carries the 3 spare columns
            const int ox = (tc.tile_x + dx - MARGIN) & ~3, oy = tc.tile_y + dy - MARGIN;
            for (int g = 0; g < ngrp; ++g) {
                const int cg = min(CGRP, C - g * CGRP);
                mbar_wait(smem_u32(&s_empty[slot]), ph ^ 1);
                s_org[slot][0] = ox;
                s_org[slot][1] = oy;
                const uint32_t full = smem_u32(&s_full[slot]);
                mbar_expect_tx(full, (uint32_t)(cg * WIN_W * WIN_H * 4));
                for (int c = 0; c < cg; ++c)
                    tma_load_3d(win_s + slot * stage_bytes + c * PLANE_BYTES, &map, full, ox, oy, tc.b * C + g * CGRP + c);
                if (++slot == STAGES) { slot = 0; ph ^= 1; }
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const int tx = threadIdx.x & (TW - 1), tg = threadIdx.x / TW;
    int slot = 0;
    uint32_t ph = 0;
    float nfx[RPT], nfy[RPT];                              // this tile's flow, loaded one tile ahead
    auto load_flow = [&](int t) {
        if (t >= ntiles) return;
        const TileCoord tc = decode_tile(t, ntx, nty);
        const float* fxp = flow + (size_t)(tc.b * 2) * HW;
        const int j = tc.tile_x + tx, i0 = tc.tile_y + tg * RPT;
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            nfx[k] = nfy[k] = 0.0f;
            if (i0 + k < H && j < W) {
                nfx[k] = __ldg(fxp + (i0 + k) * W + j);
                nfy[k] = __ldg(fxp + HW + (i0 + k) * W + j);
            }
        }
    };
    load_flow(blockIdx.x);
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const TileCoord tc = decode_tile(t, ntx, nty);
        const int b = tc.b, j = tc.tile_x + tx, i0 = tc.tile_y + tg * RPT;
        // coordinate pipeline of this thread's 4 pixels (does not depend on the window)
        float w00[RPT], w01[RPT], w10[RPT], w11[RPT];
        int x0[RPT], y0[RPT];
        unsigned fin = 0;                                  // bit k: pixel k's source position is finite
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            const int i = i0 + k;
            w00[k] = w01[k] = w10[k] = w11[k] = 0.0f; x0[k] = y0[k] = 0;
            if (i >= H || j >= W) continue;
            const SrcPos s = warp_source<PAD, AC>(nfx[k], nfy[k], i, j, H, W, fm);
            if (valid) valid[(size_t)b * HW + i * W + j] = s.valid ? 1 : 0;
            const BilinearTaps tp = bilinear_taps<PAD>(s.ix, s.iy, H, W);
            w00[k] = tp.w00; w01[k] = tp.w01; w10[k] = tp.w10; w11[k] = tp.w11;
            x0[k] = tp.x0; y0[k] = tp.y0;
            // a non-finite position has NaN weights, which the window's zero-filled taps must not meet
            if (fabsf(s.ix) < 1.0e9f && fabsf(s.iy) < 1.0e9f) fin |= 1u << k;
        }
        load_flow(t + gridDim.x);                          // in flight during the gather below

        for (int g = 0; g < ngrp; ++g) {
            const int c0 = g * CGRP, cg = min(CGRP, C - c0);
            mbar_wait(smem_u32(&s_full[slot]), ph);
            const int wx0g = s_org[slot][0], wy0g = s_org[slot][1];
            const float* wbase = win + (size_t)slot * (stage_bytes / 4);
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                const int i = i0 + k;
                if (i >= H || j >= W) continue;
                const int lx = x0[k] - wx0g, ly = y0[k] - wy0g;
                const bool fast = ((fin >> k) & 1u) && lx >= 0 && lx + 1 < WIN_W && ly >= 0 && ly + 1 < WIN_H;
                float* op = out + (size_t)(b * C + c0) * HW + i * W + j;
                if (fast) {
                    const float* s = wbase + ly * WIN_W + lx;
                    for (int c = 0; c < cg; ++c, s += PLANE) {
                        float acc = __fmaf_rn(s[0], w00[k], 0.0f);
                        acc = __fmaf_rn(s[1], w01[k], acc);
                        acc = __fmaf_rn(s[WIN_W], w10[k], acc);
                        acc = __fmaf_rn(s[WIN_W + 1], w11[k], acc);
                        op[(size_t)c * HW] = acc;
                    }
                } else {
                    const int o = y0[k] * W + x0[k];
                    for (int c = 0; c < cg; ++c)
                        op[(size_t)c * HW] = gather4(frame + (size_t)(b * C + c0 + c) * HW + o, 1, W,
                                                     tap_mask<PAD>(x0[k], y0[k], H, W), w00[k], w01[k], w10[k], w11[k]);
                }
            }
            __syncwarp();
            if ((threadIdx.x & 31) == 0) mbar_arrive(smem_u32(&s_empty[slot]));   // this warp is done with the slot
            if (++slot == STAGES) { slot = 0; ph ^= 1; }
        }
    }
}

template <int PAD, bool AC>
int launch(const CUtensorMap& map, const float* frame, const float* flow, float* out, uint8_t* valid, int B, int C,
           int H, int W, const FlowMul& fm, cudaStream_t st) {
    OFB_CUDA(ofb_smem_once<warp_tma_kernel<PAD, AC>>(STAGES * CGRP * PLANE_BYTES));
    const int cg = C < CGRP ? C : CGRP;
    const size_t smem = (size_t)STAGES * cg * PLANE_BYTES;
    const int ntx = (W + TW - 1) / TW, nty = (H + TH - 1) / TH;
    const long long ntiles = (long long)ntx * nty * B;
    if (ntiles >= (1LL << 31)) return OFB_EUNSUPPORTED;
    const int per_sm = (int)((227 * 1024) / (smem + 1024)) < 3 ? (int)((227 * 1024) / (smem + 1024)) : 3;
    const long long cap = (long long)ofb_num_sms() * per_sm;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    warp_tma_kernel<PAD, AC><<<grid, NT + 32, smem, st>>>(map, frame, flow, out, valid, C, H, W, ntx, nty, (int)ntiles, fm);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

}  // namespace

// frame must be 16-byte aligned with W % 4 == 0 (TMA global strides are multiples of 16 bytes); the caller
// (warp.cu) checks that and the 32-bit offset limits.
int ofb_warp_tma_launch(const float* frame, const float* flow, float* out, uint8_t* valid, int B, int C, int H, int W,
                        int pad, int ac, const ofb::FlowMul& fm, cudaStream_t st) {
    CUtensorMap map;
    const cuuint64_t gdim[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B * C};
    const cuuint64_t gstr[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
    const cuuint32_t box[3] = {WIN_W, WIN_H, 1};
    if (!encode_tiled(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, frame, gdim, gstr, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B))
        return OFB_EDRIVER;
    return ofb_dispatch_pad_ac(pad, ac, [&](auto P, auto A) {
        return launch<P, A>(map, frame, flow, out, valid, B, C, H, W, fm, st);
    });
}
