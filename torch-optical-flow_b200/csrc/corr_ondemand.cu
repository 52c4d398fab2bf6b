// corr_ondemand.cu -- on-demand correlation lookup: CorrBlock.__call__ without a materialised volume (SURVEY.md 8f row 4).
//
// The reference builds the whole (B*h*w) x (h*w) volume and its pooled copies first (methods/raft/model/corr.py:45-54:
// 4.26 GB fp32 / 2.83 GB bf16 per 1088x1920 pair with the pyramid) and then samples (2r+1)^2 windows from it
// (corr.py:56-77).  Average pooling is linear -- avgpool_l(f1^T f2) = f1^T avgpool_l(f2) -- so a lookup only needs
//     corr_l[q, (y, x)] = < f1[:, q] / sqrt(C) , avgpool_l(f2)[:, y, x] >
// at the ~(2r+2)^2 positions its window touches.  This kernel evaluates exactly those dot products from the K-major
// bf16 operands the tcgen05 builder uses (ofb_corr_prep_from: fmap1 * 1/sqrt(C), and fmap2 pooled by 1, 2, 4, 8) and
// samples them as the generic lookup does (ofb::warp_window, common.cuh).  Memory per pair: 4 small operand maps (22 MB
// at 1080p) instead of the 2.83 GB pyramid; cost: ~100x the arithmetic of a lookup per iteration, on the CUDA cores.
// It is a capacity feature (batch sizes / resolutions whose pyramid does not fit), not a faster path: see DESIGN.md.
//
// Work decomposition: a work item is an 8 x 4 tile of queries at ONE pyramid level; its 4 warps own the 4 tile rows and walk
// them left to right side by side, so the windows of the queries in flight overlap (10 of 11 columns with the previous
// query of the same warp, 10 of 11 rows with the neighbouring warp) and most fmap2 rows (512 B each at C = 256) come from
// L1 instead of L2: a window is ~60 KB of operand rows, and with one level per warp and 7 CTAs per SM the first version
// ran at the L2 -> SM limit (65 GB per iteration at the bench shape: 8.6 ms).  CTAs are persistent, OFB_ONDEMAND_OCC
// (default 4 = the register limit) per SM.  Measured (profiles/r02_ondemand.jsonl): with white-noise coordinates
// (sigma = 4 px, the bench's) consecutive windows overlap by only ~1/3 and the kernel stays at the L2 -> SM limit
// (9.4 ms per iteration for 8 pairs at 136x240); smooth coordinates reuse their rows from L1.  Per query a warp
//   1. computes the 2*(2r+1) tap coordinates with the reference's fp32 round trip (ofb::lookup_tap, SURVEY.md 8c),
//   2. evaluates the <= 12 x 12 patch of dot products: lane <-> 8 consecutive channels, 32 positions per pass,
//      one 16-byte load + 8 FMAs per position and lane, then ONE transposing butterfly (31 shuffles) turns the 32 lanes'
//      partial sums of 32 positions into one finished value per lane,
//   3. samples the (2r+1)^2 outputs from the patch, 3 per lane,
// and stages 8 queries' outputs so that the global writes are runs of 8 elements (32 bytes in fp32; the output may also
// be fp16 or bf16, each fp32 sample rounded once, as ofb_corr_lookup_to does).
#include <cstdlib>

#include "common.cuh"

namespace {

constexpr int TQ = 8;         // queries per tile row (one warp walks them)
constexpr int TQY = 4;        // tile rows = warps per CTA
using ofb::PD;
using ofb::MAX_D;
constexpr int MAX_DD = MAX_D * MAX_D;

struct OdParams {
    const __nv_bfloat16* f1;                       // (B, h*w, C), already scaled by 1/sqrt(C)
    const __nv_bfloat16* f2[OFB_MAX_LEVELS];       // (B, h_l*w_l, C), fmap2 averaged over complete 2^l x 2^l blocks
    int lh[OFB_MAX_LEVELS], lw[OFB_MAX_LEVELS];
    int levels, radius, B, C, h, w, tiles_x, tiles_y;
    long long n_items;
};

template <int CPL> struct Slice;                  // CPL consecutive channels of one K-major row -> fp32
template <> struct Slice<8> {
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[8]) {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
        const unsigned w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
    }
};
template <> struct Slice<4> {
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[4]) {
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
        v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xffff0000u);
        v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xffff0000u);
    }
};
template <> struct Slice<2> {
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[2]) {
        const unsigned u = __ldg(reinterpret_cast<const unsigned*>(p));
        v[0] = __uint_as_float(u << 16); v[1] = __uint_as_float(u & 0xffff0000u);
    }
};

// 32 lanes x 32 partial sums -> lane i holds the total of value i
__device__ __forceinline__ float transpose_reduce(float (&v)[32], int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool up = lane & s;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = up ? v[i] : v[i + s];
            const float keep = up ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0];
}

template <int CPL, typename O>
__global__ void __launch_bounds__(128) ondemand_lookup_kernel(const OdParams P, const float* __restrict__ coords,
                                                              O* __restrict__ out) {
    __shared__ float patch_s[TQY][PD * PD];
    __shared__ float otile_s[TQY][MAX_DD][TQ + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* patch = patch_s[warp];
    float (*otile)[TQ + 1] = otile_s[warp];
    const int D = 2 * P.radius + 1, DD = D * D, CH = P.levels * DD;
    const int tiles = P.tiles_x * P.tiles_y;
    const long long HW = (long long)P.h * P.w;
    for (long long item = blockIdx.x; item < P.n_items; item += gridDim.x) {
    // item -> (batch, level, tile): tiles of one level are neighbours in time, the operand map of a level stays hot in L2
    const int trem = (int)(item % tiles);
    const int l = (int)((item / tiles) % P.levels), b = (int)(item / ((long long)tiles * P.levels));
    const int ty = trem / P.tiles_x, tx = trem - ty * P.tiles_x;
    const int Wl = P.lw[l], Hl = P.lh[l];
    const __nv_bfloat16* f2 = P.f2[l] + (long long)b * Hl * Wl * P.C + lane * CPL;
    const float inv = 1.0f / (float)(1 << l);                  // exact power of two
    const int x_tile = tx * TQ, nqx = min(TQ, P.w - x_tile);

    {
        const int y = ty * TQY + warp;
        if (y >= P.h) continue;
        for (int qx = 0; qx < nqx; ++qx) {
            const long long p = (long long)y * P.w + x_tile + qx;
            float a[CPL];
            Slice<CPL>::load(P.f1 + ((long long)b * HW + p) * P.C + lane * CPL, a);
            const float cx0 = __ldg(coords + ((long long)b * 2 + 0) * HW + p);
            const float cy0 = __ldg(coords + ((long long)b * 2 + 1) * HW + p);
            // ---- 1. tap coordinates.  A window with a tap outside the guard lies outside the image (ofb::LookupTap): its
            // dot products are skipped and its samples are 0
            ofb::WarpWindow win = ofb::warp_window<false>(cx0, cy0, inv, P.radius, Wl, Hl, lane);
            const bool guarded = __any_sync(0xffffffffu, win.i0 == ofb::TAP_FAR && (lane & 15) < D);
            win.patch_ok = win.patch_ok && !guarded;
            const int px0 = win.px0, py0 = win.py0, cols = win.cols;
            // ---- 2. the patch of dot products, 32 positions per pass
            if (win.patch_ok) {
                const int npos = win.rows * cols;
                int r = 0, c = 0;                                     // uniform raster walk over the patch
                for (int g0 = 0; g0 < npos; g0 += 32) {
                    float part[32];
                    // 8 positions per batch: all 8 loads are issued before the first FMA (a load under a branch would be
                    // serialised with its use: ~450 cycles per position).  Positions outside the image / past the patch
                    // read the clamped address and are multiplied out.
#pragma unroll
                    for (int i8 = 0; i8 < 32; i8 += 8) {
                        float v[8][CPL];
                        float keep[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int yy = py0 + r, xx = px0 + c;
                            const bool in = g0 + i8 + u < npos && yy >= 0 && yy < Hl && xx >= 0 && xx < Wl;   // zeros padding
                            keep[u] = in ? 1.0f : 0.0f;
                            const int yc = min(max(yy, 0), Hl - 1), xc = min(max(xx, 0), Wl - 1);
                            Slice<CPL>::load(f2 + ((long long)yc * Wl + xc) * P.C, v[u]);
                            if (++c == cols) { c = 0; ++r; }
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            float sacc = 0.0f;
#pragma unroll
                            for (int k = 0; k < CPL; ++k) sacc = __fmaf_rn(a[k], v[u][k], sacc);
                            part[i8 + u] = sacc * keep[u];
                        }
                    }
                    const float total = transpose_reduce(part, lane);
                    const int e = g0 + lane;
                    if (e < npos) {
                        const int er = e / cols;
                        patch[er * PD + (e - er * cols)] = total;
                    }
                }
            }
            __syncwarp();
            // ---- 3. (2r+1)^2 samples, 3 per lane
            ofb::warp_window_samples(
                win, patch, P.radius, lane,
                [](int, int, float, float, float, float) { return 0.0f; },
                [&](int k, int, int, float v) { otile[k][qx] = v; });
            __syncwarp();
        }
        // ---- one tile row of queries is done: 32-byte runs per channel
        O* dst = out + ((long long)b * CH + (long long)l * DD) * HW + (long long)y * P.w + x_tile;
        for (int idx = lane; idx < DD * TQ; idx += 32) {
            const int k = idx >> 3, qx = idx & 7;
            if (qx < nqx) dst[(long long)k * HW + qx] = ofb::narrow<O>(otile[k][qx]);
        }
        __syncwarp();
    }
    }
}

}  // namespace

OFB_API int ofb_corr_lookup_ondemand_to(const void* f1_km, const void* const* f2_km_levels, const float* coords,
                                        void* out, int out_dtype, int B, int C, int h, int w, int levels, int radius,
                                        void* stream) {
    if (!ofb_float_dtype(out_dtype)) return OFB_EINVAL;
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!f1_km || !f2_km_levels || !coords || !out || B < 0 || C <= 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (levels < 1 || levels > OFB_MAX_LEVELS) return OFB_EINVAL;
    if (radius < 0 || 2 * radius + 1 > MAX_D) return OFB_EUNSUPPORTED;
    if (C != 64 && C != 128 && C != 256) return OFB_EUNSUPPORTED;
    OdParams P = {};
    P.f1 = reinterpret_cast<const __nv_bfloat16*>(f1_km);
    if (reinterpret_cast<uintptr_t>(f1_km) & 15) return OFB_EALIGN;
    for (int l = 0; l < levels; ++l) {
        P.lh[l] = h >> l; P.lw[l] = w >> l;
        if (!f2_km_levels[l] || P.lh[l] <= 0 || P.lw[l] <= 0) return OFB_EINVAL;
        if (reinterpret_cast<uintptr_t>(f2_km_levels[l]) & 15) return OFB_EALIGN;
        if (P.lh[l] > 65536 || P.lw[l] > 65536) return OFB_EUNSUPPORTED;
        P.f2[l] = reinterpret_cast<const __nv_bfloat16*>(f2_km_levels[l]);
    }
    P.levels = levels; P.radius = radius; P.B = B; P.C = C; P.h = h; P.w = w;
    P.tiles_x = (w + TQ - 1) / TQ; P.tiles_y = (h + TQY - 1) / TQY;
    P.n_items = (long long)B * levels * P.tiles_x * P.tiles_y;
    static const int occ = [] {
        const char* e = getenv("OFB_ONDEMAND_OCC");                 // resident CTAs per SM (tuning override)
        const int n = e ? atoi(e) : 4;
        return (n < 1 || n > 16) ? 4 : n;
    }();
    long long blocks = (long long)ofb_num_sms() * occ;
    if (blocks > P.n_items) blocks = P.n_items;
    cudaStream_t st = (cudaStream_t)stream;
    const int threads = 32 * TQY;
    return ofb_dispatch_dtype(out_dtype, [&](auto o) {
        using O = decltype(o);
        O* dst = static_cast<O*>(out);
        if (C == 256) ondemand_lookup_kernel<8, O><<<(int)blocks, threads, 0, st>>>(P, coords, dst);
        else if (C == 128) ondemand_lookup_kernel<4, O><<<(int)blocks, threads, 0, st>>>(P, coords, dst);
        else ondemand_lookup_kernel<2, O><<<(int)blocks, threads, 0, st>>>(P, coords, dst);
        OFB_LAUNCH_CHECK();
        return OFB_OK;
    });
}

OFB_API int ofb_corr_lookup_ondemand(const void* f1_km, const void* const* f2_km_levels, const float* coords, float* out,
                                     int B, int C, int h, int w, int levels, int radius, void* stream) {
    return ofb_corr_lookup_ondemand_to(f1_km, f2_km_levels, coords, out, OFB_DTYPE_F32, B, C, h, w, levels, radius,
                                       stream);
}
