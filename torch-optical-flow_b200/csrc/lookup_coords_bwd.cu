// lookup_coords_bwd.cu -- K3 backward: gradient of the correlation lookup with respect to its coordinates.
//
// The reference's CorrBlock.__call__ (methods/raft/model/corr.py:56-77) samples every level with bilinear_sampler =
// F.grid_sample(align_corners=True, zeros padding) (utils.py:64-80), which is differentiable in the coordinates too.
// For level l, window cell (i, j) (i moves x: corr.py:64-70) with taps (x0, wx0, wx1) and (y0, wy0, wy1) from
// ofb::lookup_tap and v(y, x) the stored level value (0 outside the image), ATen's GridSampler backward gives
//     gx_ij = wy0 (v(y0, x0+1) - v(y0, x0)) + wy1 (v(y0+1, x0+1) - v(y0+1, x0))
//     gy_ij = wx0 (v(y0+1, x0) - v(y0, x0)) + wx1 (v(y0+1, x0+1) - v(y0, x0+1))
//     d coords = sum_l 2^-l sum_ij d_out[l, i, j] (gx_ij, gy_ij)
// (the chain factors (W_l-1)/2 of GridSampler.h:30 and 2/(W_l-1) of utils.py:70 multiply to 1 and are applied as 1).
// Out-of-range coordinates follow the forward lookup's policy (common.cuh, next to lookup_tap).
//
// thread = (query, level), lane <-> query, warp <-> level, as in the register-tile forward: d_out rows are 128-byte
// reads, and neighbouring queries of the query-minor layout are read by neighbouring lanes.  Each thread streams the
// D + 2 rows of its window (ofb::TapSet: a tap that slid by one pixel reads one column / row further, so regular and
// irregular windows take the same path) and folds it with d_out:
//     x:  sum_r sum_j wy_rj sum_i d_out[i, j] (v(r, b_i) - v(r, a_i))
//     y:  sum_r sum_j sy_rj sum_i d_out[i, j] (wx0_i v(r, a_i) + wx1_i v(r, b_i))
// with a_i, b_i the two columns of x tap i, and (wy_rj, sy_rj) = (wy0_j, -1) when r is the upper row of sample j,
// (wy1_j, +1) when it is its lower row (a row serves at most three samples: j = r, r - 1, r - 2).  The levels are
// summed in shared memory in level order and d coords is written once, without atomics: the same bits on every run.
// d_out is read in fp32, fp16 or bf16 (the dtype of the forward's output) and widened exactly on load.
// HBM roofline per query: L*(2r+2)^2*esize window + L*(2r+1)^2*(d_out esize) + 8 coordinates read, 8 written.
#include "common.cuh"

namespace {

using ofb::MAX_D;

struct CoordsBwdParams : ofb::PyramidView {
    int h, w, B;   // in this order: (h, w) is one 8-byte constant load
};

// Window row y, columns xs .. xs + WIN - 1 of a (query, level) slice -> px, 0 outside the image.  CHUNKED: 16-bit
// levels whose rows (or 8x4 blocks) are 16-byte aligned 8-element chunks, read as the register-tile forward reads them;
// otherwise one element at a time (fp32, and 16-bit rows of any even pitch).
template <typename T, bool CHUNKED, int WIN>
__device__ __forceinline__ void load_row(float (&px)[WIN], const T* slice, const CoordsBwdParams& P, int pitch, int Wl,
                                         int xs, int y, bool rok) {
    if constexpr (CHUNKED) {
        const ofb::RowChunks ck = ofb::row_chunks(xs, WIN, pitch);
        uint32_t w[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) w[k] = 0u;
        if (rok) {
            const long long cstep = OFB_PIECE_STEP(P);
            const T* row = OFB_PIECE(slice, P, y, ck.xa, pitch);
            if (ck.ck0) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(row));
                w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
            }
            if (ck.ck1) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(row + cstep));
                w[4] = v.x; w[5] = v.y; w[6] = v.z; w[7] = v.w;
            }
            if (ck.ck2) {
                const uint2 v = __ldg(reinterpret_cast<const uint2*>(row + 2 * cstep));
                w[8] = v.x; w[9] = v.y;
            }
        }
        ofb::realign_row<T>(w, ck.q1, ck.q2, ck.hs, px);
#pragma unroll
        for (int e = 0; e < WIN; ++e)       // padding columns (and chunks never loaded) are outside the image
            if (xs + e < 0 || xs + e >= Wl) px[e] = 0.0f;
    } else {
        const T* row = slice + (long long)y * pitch + xs;       // element e at row[e]
#pragma unroll
        for (int e = 0; e < WIN; ++e)
            px[e] = (rok && (unsigned)(xs + e) < (unsigned)Wl) ? ofb::ld_f32(row + e) : 0.0f;
    }
}

template <int R, typename T, bool CHUNKED, typename G>
__global__ void __launch_bounds__(128, 4) lookup_coords_bwd_kernel(const __grid_constant__ CoordsBwdParams P,
                                                                const float* __restrict__ coords,
                                                                const G* __restrict__ d_out,
                                                                float* __restrict__ d_coords) {
    constexpr int D = 2 * R + 1, DD = D * D, WIN = D + 2;
    constexpr int GROUPS_UNROLLED = CHUNKED ? (WIN + 2) / 3 : 1;
    __shared__ float part[2][OFB_MAX_LEVELS][32];
    const int l = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long HW = (long long)P.h * P.w, Q = (long long)P.B * HW;
    const long long q = (long long)blockIdx.x * 32 + lane;
    const long long b = q / HW, p = q - b * HW;
    float gx = 0.0f, gy = 0.0f;
    if (q < Q) {
        const int Wl = P.lw[l], Hl = P.lh[l], pitch = P.pitch[l];
        const float inv = 1.0f / (float)(1 << l);                   // exact power of two
        const float cx = __fmul_rn(__ldg(coords + (b * 2 + 0) * HW + p), inv);
        const float cy = __fmul_rn(__ldg(coords + (b * 2 + 1) * HW + p), inv);
        const ofb::TapSet<R> tx = ofb::make_taps<R>(cx, Wl, nullptr);
        const ofb::TapSet<R> ty = ofb::make_taps<R>(cy, Hl, nullptr);
        // a tap outside the guard: every tap of its axis is outside the image, so the level contributes 0 (its
        // weights may be NaN and are never used)
        if (!tx.dead && !ty.dead) {
            const int xs = tx.anchor, ys = ty.anchor;
            const T* slice = reinterpret_cast<const T*>(P.base[l]) + q * P.q_stride[l];
            // d_out of window cell (i, j) at g0[(i*D + j) * HW]
            const G* g0 = d_out + (b * (long long)(P.levels * DD) + (long long)l * DD) * HW + p;
            // window rows some sample reads (tap j: rows j + d[j] and j + d[j] + 1); the others are never loaded, so
            // an inf stored there is not multiplied by an exact-zero coefficient
            unsigned used_rows = 0;
#pragma unroll
            for (int j = 0; j < D; ++j) used_rows |= 3u << (j + ((ty.dmask >> j) & 1u));
            float g[3][D];                                          // d_out rows j = r, r-1, r-2 at g[j % 3]
            float acc_x = 0.0f, acc_y = 0.0f;
            // rows in groups of three, so that g[j % 3] is a register index either way.  The chunked path unrolls
            // every row (its loads overlap the arithmetic of earlier rows; 128 registers, 4 CTAs per SM, as the
            // forward); the element-wise path runs one group at a time, or its (D + 2)^2 loads, unrolled, would take
            // more registers than a thread has -- its y weights are then indexed at run time, from local memory.
#pragma unroll (GROUPS_UNROLLED)
            for (int r0 = 0; r0 < WIN; r0 += 3) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const int r = r0 + c;
                    if (r >= WIN) break;
                    const int y = ys + r;
                    float px[WIN];
                    load_row<T, CHUNKED>(px, slice, P, pitch, Wl, xs, y, ((used_rows >> r) & 1u) && y >= 0 && y < Hl);
                    // x differences and horizontal samples of the row, tap by tap (tap i reads columns i + d[i], + 1).
                // wx0 is formed as 1 - wx1, one register per tap fewer: for a floor >= 0, wx1 = ic - floor is exact, so
                // 1 - wx1 and lookup_tap's (floor + 1) - ic round the same real number; for a floor < 0, column floor is
                // outside the image and wx0 multiplies 0.
                    float dxr[D], hxr[D];
#pragma unroll
                    for (int i = 0; i < D; ++i) {
                        const bool d = (tx.dmask >> i) & 1u;
                        const float va = d ? px[i + 1] : px[i], vb = d ? px[i + 2] : px[i + 1];
                        dxr[i] = __fsub_rn(vb, va);
                        hxr[i] = __fmaf_rn(tx.w1[i], vb, __fmul_rn(__fsub_rn(1.0f, tx.w1[i]), va));
                    }
                    if (r < D) {
#pragma unroll
                        for (int i = 0; i < D; ++i) g[c][i] = ofb::ld_f32(g0 + (long long)(i * D + r) * HW);
                    }
                    // row r is the upper row of sample j = r - k when k = d[j], its lower row when k = d[j] + 1
                    float row_x = 0.0f, row_y = 0.0f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const int j = r - k;
                        if (j < 0 || j >= D) continue;
                        const int d = (ty.dmask >> j) & 1u;
                        if (k != d && k != d + 1) continue;
                        float sx = 0.0f, sy = 0.0f;
#pragma unroll
                        for (int i = 0; i < D; ++i) {
                            sx = __fmaf_rn(g[(c - k + 3) % 3][i], dxr[i], sx);
                            sy = __fmaf_rn(g[(c - k + 3) % 3][i], hxr[i], sy);
                        }
                        const bool upper = k == d;
                        row_x = __fmaf_rn(upper ? ty.w0[j] : ty.w1[j], sx, row_x);
                        row_y = upper ? __fsub_rn(row_y, sy) : __fadd_rn(row_y, sy);
                    }
                    acc_x = __fadd_rn(acc_x, row_x);
                    acc_y = __fadd_rn(acc_y, row_y);
                }
            }
            gx = __fmul_rn(acc_x, inv);
            gy = __fmul_rn(acc_y, inv);
        }
    }
    part[0][l][lane] = gx;
    part[1][l][lane] = gy;
    __syncthreads();
    if (l == 0 && q < Q) {                                          // levels summed in level order
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            float s = part[a][0][lane];
            for (int k = 1; k < P.levels; ++k) s = __fadd_rn(s, part[a][k][lane]);
            d_coords[(b * 2 + a) * HW + p] = s;
        }
    }
}

template <int R, typename T, bool CHUNKED, typename G>
int launch(const CoordsBwdParams& P, const float* coords, const G* d_out, float* d_coords, int blocks,
           cudaStream_t st) {
    lookup_coords_bwd_kernel<R, T, CHUNKED, G><<<blocks, 32 * P.levels, 0, st>>>(P, coords, d_out, d_coords);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

template <typename T, bool CHUNKED, typename G>
int launch_radius(const CoordsBwdParams& P, const float* coords, const G* d_out, float* d_coords, int radius,
                  int blocks, cudaStream_t st) {
    switch (radius) {
        case 0: return launch<0, T, CHUNKED>(P, coords, d_out, d_coords, blocks, st);
        case 1: return launch<1, T, CHUNKED>(P, coords, d_out, d_coords, blocks, st);
        case 2: return launch<2, T, CHUNKED>(P, coords, d_out, d_coords, blocks, st);
        case 3: return launch<3, T, CHUNKED>(P, coords, d_out, d_coords, blocks, st);
        default: return launch<4, T, CHUNKED>(P, coords, d_out, d_coords, blocks, st);
    }
}

template <typename G>
int launch_pyramid(const CoordsBwdParams& P, bool chunked, const float* coords, const G* d_out, float* d_coords,
                   int radius, int blocks, cudaStream_t st) {
    if (P.dtype == OFB_DTYPE_F32)
        return launch_radius<float, false>(P, coords, d_out, d_coords, radius, blocks, st);
    if (P.dtype == OFB_DTYPE_F16)
        return chunked ? launch_radius<__half, true>(P, coords, d_out, d_coords, radius, blocks, st)
                       : launch_radius<__half, false>(P, coords, d_out, d_coords, radius, blocks, st);
    return chunked ? launch_radius<__nv_bfloat16, true>(P, coords, d_out, d_coords, radius, blocks, st)
                   : launch_radius<__nv_bfloat16, false>(P, coords, d_out, d_coords, radius, blocks, st);
}

}  // namespace

OFB_API int ofb_corr_lookup_coords_backward_from(const ofb_pyramid* pyr, const float* coords, const void* d_out,
                                                 int d_out_dtype, float* d_coords, int B, int h, int w, int radius,
                                                 void* stream) {
    if (!ofb_float_dtype(d_out_dtype)) return OFB_EINVAL;
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!pyr || !coords || !d_out || !d_coords || B < 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (radius < 0 || 2 * radius + 1 > MAX_D) return OFB_EUNSUPPORTED;
    const long long Q = (long long)B * h * w;
    CoordsBwdParams P;
    if (const int rc = ofb::check_pyramid(pyr, Q, P)) return rc;
    bool chunked;
    if (const int rc = ofb::lookup_reader(P, radius, chunked)) return rc;
    P.B = B; P.h = h; P.w = w;
    const long long blocks = (Q + 31) / 32;
    if (blocks > 0x7fffffffLL) return OFB_EUNSUPPORTED;
    return ofb_dispatch_dtype(d_out_dtype, [&](auto g) {
        using G = decltype(g);
        return launch_pyramid(P, chunked, coords, static_cast<const G*>(d_out), d_coords, radius, (int)blocks,
                              (cudaStream_t)stream);
    });
}

OFB_API int ofb_corr_lookup_coords_backward(const ofb_pyramid* pyr, const float* coords, const float* d_out,
                                            float* d_coords, int B, int h, int w, int radius, void* stream) {
    return ofb_corr_lookup_coords_backward_from(pyr, coords, d_out, OFB_DTYPE_F32, d_coords, B, h, w, radius, stream);
}
