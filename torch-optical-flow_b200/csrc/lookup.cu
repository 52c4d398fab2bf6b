// lookup.cu -- K3: correlation-pyramid lookup, all levels in one pass.
//
// Replaces CorrBlock.__call__ + bilinear_sampler (reference methods/raft/model/corr.py:56-77,
// methods/raft/model/utils.py:64-80).  The reference runs ~70 small ATen launches per
// refinement iteration (delta grid + H2D copy, 3 materialised (N,9,9,2) coordinate tensors,
// grid_sample, 5 concatenations); here one kernel reads the coordinates and the pyramid and
// writes the (B, L*(2r+1)^2, h, w) fp32 output.
//
// The tap coordinates follow the bit-exact sequence of ofb::lookup_tap (common.cuh, SURVEY.md 8c).
//
// Work decomposition: a CTA owns 32 consecutive queries; each of its 8 warps walks 4 of them.
// Per (query, level) the warp
//   1. computes the 2*(2r+1) tap coordinates, one per lane (ofb::warp_window),
//   2. loads the <=12x12 patch of the query's level slice that covers all taps into a private
//      shared-memory patch (4-byte words; out-of-image elements become zeros = zeros padding),
//   3. produces the (2r+1)^2 samples, 3 per lane (ofb::warp_window_samples).
// Results are staged in a [channel][query] shared tile so the global writes are 128-byte rows.
// HBM roofline per query and iteration (SURVEY.md 8d): L*(2r+2)^2*esize + 8 read, 4*L*(2r+1)^2 written.
#include <climits>

#include "common.cuh"

namespace {

using ofb::PD;
using ofb::MAX_D;
constexpr int QT = 32;        // queries per CTA
constexpr int NW = 8;         // warps per CTA
constexpr int OT_PITCH = QT + 1;

struct LookupParams : ofb::PyramidLevels {
    int levels, radius, B, h, w;
    int blocked;   // 8x4-blocked layouts (register-tile kernel only, 16-bit pyramids)
    long long blk_stride;   // elements between consecutive blocks: 32, or 32 * Q (query-minor)
};

// patch load: bf16 / fp16 -> two elements per 4-byte word (px0 and pitch are even, the slice base is 4-byte aligned)
template <typename T>
__device__ __forceinline__ void load_patch(float* patch, const T* slice, int pitch, int Hl, int Wl, int px0, int py0,
                                           int rows, int lane) {
#pragma unroll
    for (int e = lane; e < PD * (PD / 2); e += 32) {
        const int r = e / (PD / 2), cw = e - r * (PD / 2);
        const int y = py0 + r, x = px0 + 2 * cw;
        float v0 = 0.0f, v1 = 0.0f;
        if (r < rows && y >= 0 && y < Hl && x >= 0 && x < Wl) {
            const unsigned wd = __ldg(reinterpret_cast<const unsigned*>(slice + (size_t)y * pitch + x));
            v0 = ofb::widen16<T>(wd, 0);
            if (x + 1 < Wl) v1 = ofb::widen16<T>(wd, 1);
        }
        patch[r * PD + 2 * cw] = v0;
        patch[r * PD + 2 * cw + 1] = v1;
    }
}

// fp32 -> one element per word
template <>
__device__ __forceinline__ void load_patch<float>(float* patch, const float* slice, int pitch, int Hl, int Wl, int px0,
                                                  int py0, int rows, int lane) {
#pragma unroll
    for (int e = lane; e < PD * PD; e += 32) {
        const int r = e / PD, c = e - r * PD;
        const int y = py0 + r, x = px0 + c;
        float v = 0.0f;
        if (r < rows && y >= 0 && y < Hl && x >= 0 && x < Wl) v = __ldg(slice + (size_t)y * pitch + x);
        patch[e] = v;
    }
}

template <typename T>
__global__ void __launch_bounds__(NW * 32) lookup_kernel(const LookupParams P, const float* __restrict__ coords,
                                                         float* __restrict__ out, int32_t* __restrict__ idx_out,
                                                         uint8_t* __restrict__ valid_out) {
    extern __shared__ float smem[];
    const int D = 2 * P.radius + 1, DD = D * D, CH = P.levels * DD;
    float* otile = smem;                              // [CH][OT_PITCH]
    float* patches = smem + (size_t)CH * OT_PITCH;    // [NW][PD*PD]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* patch = patches + warp * PD * PD;
    const long long HW = (long long)P.h * P.w, Q = (long long)P.B * HW;
    const long long q0 = (long long)blockIdx.x * QT;

    for (int qi = warp; qi < QT; qi += NW) {
        const long long q = q0 + qi;
        if (q >= Q) break;
        const long long b = q / HW, p = q - b * HW;
        const float cx0 = __ldg(coords + (b * 2 + 0) * HW + p);
        const float cy0 = __ldg(coords + (b * 2 + 1) * HW + p);
        for (int l = 0; l < P.levels; ++l) {
            const int Wl = P.lw[l], Hl = P.lh[l], pitch = P.pitch[l];
            const T* slice = reinterpret_cast<const T*>(P.base[l]) + q * P.q_stride[l];
            const float inv = 1.0f / (float)(1 << l);          // exact power of two
            // ---- 1. tap coordinates; 16-bit patches start on an even column (word loads)
            const ofb::WarpWindow win = ofb::warp_window<sizeof(T) == 2>(cx0, cy0, inv, P.radius, Wl, Hl, lane);
            const int t = lane & 15, isy = lane >> 4;
            if (idx_out && t < D)
                idx_out[((q * P.levels + l) * 2 + isy) * D + t] = (int32_t)win.fl;
            const unsigned vmask = __ballot_sync(0xffffffffu, win.valid);   // bit lane: that tap's utils.py:77 predicate
            // ---- 2. stage the patch
            if (win.patch_ok) load_patch<T>(patch, slice, pitch, Hl, Wl, win.px0, win.py0, win.rows, lane);
            __syncwarp();
            // ---- 3. (2r+1)^2 samples; a window the patch does not cover reads its taps straight from global memory
            ofb::warp_window_samples(
                win, patch, P.radius, lane,
                [&](int x0, int y0, float wx0, float wx1, float wy0, float wy1) {
                    const bool inx0 = x0 >= 0 && x0 < Wl, inx1 = x0 + 1 >= 0 && x0 + 1 < Wl;
                    const bool iny0 = y0 >= 0 && y0 < Hl, iny1 = y0 + 1 >= 0 && y0 + 1 < Hl;
                    const float v00 = (iny0 && inx0) ? ofb::ld_f32(slice + (size_t)y0 * pitch + x0) : 0.0f;
                    const float v01 = (iny0 && inx1) ? ofb::ld_f32(slice + (size_t)y0 * pitch + x0 + 1) : 0.0f;
                    const float v10 = (iny1 && inx0) ? ofb::ld_f32(slice + (size_t)(y0 + 1) * pitch + x0) : 0.0f;
                    const float v11 = (iny1 && inx1) ? ofb::ld_f32(slice + (size_t)(y0 + 1) * pitch + x0 + 1) : 0.0f;
                    return ofb::bilinear(v00, v01, v10, v11, wx0, wx1, wy0, wy1);
                },
                [&](int k, int i, int j, float v) {
                    otile[(l * DD + k) * OT_PITCH + qi] = v;
                    if (valid_out)
                        valid_out[(q * P.levels + l) * DD + k] = (uint8_t)((vmask >> i) & (vmask >> (16 + j)) & 1u);
                });
            __syncwarp();
        }
    }
    __syncthreads();
    // ---- coalesced write-out: one channel row (32 queries) per warp instruction
    const long long q = q0 + lane;
    if (q < Q) {
        const long long b = q / HW, p = q - b * HW;
        float* dst = out + b * CH * HW + p;
        for (int ch = warp; ch < CH; ch += NW) dst[(long long)ch * HW] = otile[ch * OT_PITCH + lane];
    }
}

// ------------------------------------------------------------------------------------------------
// Register-tile lookup for 16-bit (bf16 / fp16) pyramids (the product path).
//
// thread = (query, level): lane <-> query (coordinates in, channel rows out are 128-byte coalesced),
// warp <-> pyramid level.  Each thread
//   1. evaluates its 2*(2R+1) tap coordinates with ofb::lookup_tap;
//   2. anchors an 11 x 11 element window at (xs, ys) = min over taps of (floor index - tap number).
//      Within the guarded coordinate range every tap's floor index is tap + anchor + {0, 1} (the fp32
//      round trip can move a tap sitting on an integer to the pixel below), so tap i reads window
//      columns i .. i+2 through a 3-tap filter (w0, w1, 0) or (0, w0, w1) -- the same products as
//      the reference's 2-tap form plus exact zeros;
//   3. streams the window row by row: 16-byte aligned chunk loads (2.25 per row on average),
//      realigned in registers with two select stages (word shift) and a funnel shift (half-word),
//      widened to fp32 (bf16: a shift or mask of the word; fp16: a conversion of each half),
//      horizontal filter -> 9 values, vertical filter accumulated into three live output rows;
//   4. writes each finished output row straight to its 9 channels.
// No shared memory, no shuffles, ~56 warp instructions per (query, level) against ~230 before.
// Contract with the builder: elements between w_l and the row pitch hold FINITE values (the tcgen05
// builder writes zeros there); they are multiplied by zero weights.
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
        const ofb::LookupTap tp = ofb::lookup_tap(center, t, R, size);
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

// T: the pyramid's 16-bit type.  Only the widening of the realigned words depends on it: the coordinates, floor
// indices, validity masks and filter weights are the same code for both types.
template <int R, int GR, typename T>
__global__ void __launch_bounds__(128) lookup_tile_kernel(const LookupParams P, const float* __restrict__ coords,
                                                           float* __restrict__ out, int32_t* __restrict__ idx_out,
                                                           uint8_t* __restrict__ valid_out) {
    constexpr int D = 2 * R + 1, DD = D * D, WIN = D + 2;       // window rows / columns
    constexpr int NW = (WIN + 1) / 2;                           // packed words per realigned row (6 for R = 4)
    const int l = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long HW = (long long)P.h * P.w, Q = (long long)P.B * HW;
    const long long q = (long long)blockIdx.x * 32 + lane;
    if (q >= Q) return;
    const long long b = q / HW, p = q - b * HW;
    const int Wl = P.lw[l], Hl = P.lh[l], pitch = P.pitch[l];
    const float inv = 1.0f / (float)(1 << l);                   // exact power of two
    const float cx = __fmul_rn(__ldg(coords + (b * 2 + 0) * HW + p), inv);
    const float cy = __fmul_rn(__ldg(coords + (b * 2 + 1) * HW + p), inv);

    int32_t* idx_q = idx_out ? idx_out + ((q * P.levels + l) * 2) * D : nullptr;
    const TapSet<R> tx = make_taps<R>(cx, Wl, idx_q);
    const TapSet<R> ty = make_taps<R>(cy, Hl, idx_q ? idx_q + D : nullptr);
    const bool dead = tx.dead || ty.dead;
    if (valid_out) {
        uint8_t* vq = valid_out + (q * P.levels + l) * DD;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = 0; j < D; ++j) vq[i * D + j] = (uint8_t)(((tx.vmask >> i) & 1u) & ((ty.vmask >> j) & 1u));
    }

    // horizontal 3-tap filters; a column outside [0, w_l) gets weight zero (zeros padding)
    const int xs = dead ? 0 : tx.anchor, ys = dead ? 0 : ty.anchor;
    float fw[D][3];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        const bool d = (tx.dmask >> i) & 1u;
        float a0 = d ? 0.0f : tx.w0[i], a1 = d ? tx.w0[i] : tx.w1[i], a2 = d ? tx.w1[i] : 0.0f;
        const int c0 = xs + i;
        if (dead || c0 < 0 || c0 >= Wl) a0 = 0.0f;
        if (dead || c0 + 1 < 0 || c0 + 1 >= Wl) a1 = 0.0f;
        if (dead || c0 + 2 < 0 || c0 + 2 >= Wl) a2 = 0.0f;
        fw[i][0] = a0; fw[i][1] = a1; fw[i][2] = a2;
    }

    // chunk geometry: 8-element (16-byte) aligned chunks covering columns xs .. xs + WIN - 1
    const int xa = xs & ~7, s = xs - xa;                        // s in 0..7
    const unsigned q1 = (unsigned)(s >> 1) & 1u, q2 = (unsigned)(s >> 2) & 1u, hs = (unsigned)(s & 1) * 16u;
    const bool ck0 = xa >= 0 && xa + 8 <= pitch;
    const bool ck1 = xa + 8 >= 0 && xa + 16 <= pitch;
    // the last window column / row only carries weight when some tap slid by one (dmask != 0)
    const int wcols = tx.dmask ? WIN : WIN - 1, wrows = ty.dmask ? WIN : WIN - 1;
    const bool ck2 = (s + wcols > 16) && xa + 16 >= 0 && xa + 24 <= pitch;
    const T* slice = reinterpret_cast<const T*>(P.base[l]) + q * P.q_stride[l];
    float* outp = out + (b * (long long)(P.levels * DD) + (long long)l * DD) * HW + p;

    float acc[3][D];                                            // output rows j = r, r-1, r-2 in flight
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int i = 0; i < D; ++i) acc[k][i] = 0.0f;

    // Window rows -> this thread's private shared-memory slots with cp.async (zero-filled when the chunk is outside
    // the slice): every load of the window is in flight at once and none of them holds a register.  Chunks 0 and 1
    // are 16-byte slots at ((r*2 + c) * blockDim + t) * 16; of chunk 2 only the first 4 elements can fall inside
    // the window (s + WIN - 1 <= 17), so it gets an 8-byte slot at CK2_BASE + (r * blockDim + t) * 8.  A warp's
    // accesses are contiguous and conflict-free; 40 bytes per row and thread keep 4 CTAs (16 warps) on an SM.
    extern __shared__ __align__(16) uint8_t win_smem[];
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(win_smem);
    const uint32_t my_slot = smem0 + threadIdx.x * 16u;
    const uint32_t slot_stride = blockDim.x * 16u;
    const uint32_t my_slot2 = smem0 + (uint32_t)(WIN * 2) * slot_stride + threadIdx.x * 8u;
    const uint32_t slot2_stride = blockDim.x * 8u;
    {
        const long long cstep = P.blocked ? P.blk_stride : 8;
#pragma unroll
        for (int r = 0; r < WIN; ++r) {
            const int y = ys + r;
            const bool rok = !dead && r < wrows && y >= 0 && y < Hl;
            // an aligned 8-element chunk is one row of an 8x4 block (blocked) or 8 consecutive row elements
            const T* row = P.blocked
                ? slice + ((long long)(y >> 2) * (pitch >> 3) + (xa >> 3)) * P.blk_stride + (y & 3) * 8
                : slice + (long long)y * pitch + xa;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const bool ok = rok && (c == 0 ? ck0 : ck1);
                const void* src = ok ? (const void*)(row + c * cstep) : (const void*)slice;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(my_slot + (uint32_t)(r * 2 + c) * slot_stride),
                             "l"(src), "r"(ok ? 16 : 0) : "memory");
            }
            {
                const bool ok = rok && ck2;
                const void* src = ok ? (const void*)(row + 2 * cstep) : (const void*)slice;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(my_slot2 + (uint32_t)r * slot2_stride),
                             "l"(src), "r"(ok ? 8 : 0) : "memory");
            }
            // one commit group per GR rows: the filter below starts on the first rows while the rest are in flight
            if (r % GR == GR - 1 || r == WIN - 1) asm volatile("cp.async.commit_group;" ::: "memory");
        }
    }
#pragma unroll
    for (int r = 0; r < WIN; ++r) {
        if (r % GR == 0) {                                      // groups complete in order: wait for this row's group
            constexpr int NG = (WIN + GR - 1) / GR;
            const int pending = NG - 1 - r / GR;                // groups allowed to be still in flight
            if (pending >= 3) asm volatile("cp.async.wait_group 3;" ::: "memory");
            else if (pending == 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
            else if (pending == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        uint32_t w[10];
#pragma unroll
        for (int c = 0; c < 2; ++c)
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(w[4 * c]), "=r"(w[4 * c + 1]), "=r"(w[4 * c + 2]), "=r"(w[4 * c + 3])
                         : "r"(my_slot + (uint32_t)(r * 2 + c) * slot_stride));
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(w[8]), "=r"(w[9]) : "r"(my_slot2 + (uint32_t)r * slot2_stride));
        // ---- realign: drop s leading elements (word shifts by 1 and 2, then a half-word funnel shift)
        uint32_t t1[9], t2[NW + 1], v[NW];
#pragma unroll
        for (int k = 0; k < 9; ++k) t1[k] = q1 ? w[k + 1] : w[k];
#pragma unroll
        for (int k = 0; k <= NW; ++k) t2[k] = q2 ? t1[k + 2] : t1[k];
#pragma unroll
        for (int k = 0; k < NW; ++k) v[k] = __funnelshift_r(t2[k], t2[k + 1], hs);
        float px[WIN];
#pragma unroll
        for (int e = 0; e < WIN; ++e) px[e] = ofb::widen16<T>(v[e >> 1], e & 1);
        // ---- horizontal filter
        float hrow[D];
#pragma unroll
        for (int i = 0; i < D; ++i)
            hrow[i] = __fmaf_rn(fw[i][2], px[i + 2], __fmaf_rn(fw[i][1], px[i + 1], __fmul_rn(fw[i][0], px[i])));
        // ---- vertical filter: window row r feeds output rows j = r (tap 0), r-1 (tap 1), r-2 (tap 2)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int j = r - k;
            if (j < 0 || j >= D) continue;
            const bool d = (ty.dmask >> j) & 1u;
            float vw = k == 0 ? (d ? 0.0f : ty.w0[j]) : k == 1 ? (d ? ty.w0[j] : ty.w1[j]) : (d ? ty.w1[j] : 0.0f);
            if (dead) vw = 0.0f;            // non-finite / far-away coordinates: the weights may be NaN, the result is 0
#pragma unroll
            for (int i = 0; i < D; ++i) acc[(j % 3)][i] = __fmaf_rn(vw, hrow[i], acc[(j % 3)][i]);
        }
        // ---- output row j = r - 2 is complete: channel = l*DD + i*D + j  (i moves x: corr.py:64-70)
        if (r >= 2) {
            const int j = r - 2;
#pragma unroll
            for (int i = 0; i < D; ++i) {
                outp[(long long)(i * D + j) * HW] = acc[j % 3][i];
                acc[j % 3][i] = 0.0f;
            }
        }
    }
}

__global__ void __launch_bounds__(256) bilinear_sampler_kernel(const float* __restrict__ img,
                                                               const float* __restrict__ coords,
                                                               float* __restrict__ out, float* __restrict__ mask, int N,
                                                               int C, int H, int W, int Ho, int Wo) {
    const size_t HWo = (size_t)Ho * Wo, total = (size_t)N * HWo;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t n = t / HWo, p = t - n * HWo;
        const float2 c = __ldg(reinterpret_cast<const float2*>(coords) + t);
        const float gx = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, c.x), (float)(W - 1)), 1.0f);
        const float gy = __fsub_rn(__fdiv_rn(__fmul_rn(2.0f, c.y), (float)(H - 1)), 1.0f);
        const float ix = ofb::unnormalize<true>(gx, W), iy = ofb::unnormalize<true>(gy, H);
        if (mask) mask[t] = ((gx > -1.0f) && (gy > -1.0f) && (gx < 1.0f) && (gy < 1.0f)) ? 1.0f : 0.0f;
        const float x0f = floorf(ix), y0f = floorf(iy);
        const bool fin = x0f >= -8.0f && x0f <= 1.0e6f && y0f >= -8.0f && y0f <= 1.0e6f;
        const int x0 = fin ? (int)x0f : -100, y0 = fin ? (int)y0f : -100;
        const float wx1 = ix - x0f, wx0 = (x0f + 1.0f) - ix, wy1 = iy - y0f, wy0 = (y0f + 1.0f) - iy;
        const bool inx0 = x0 >= 0 && x0 < W, inx1 = x0 + 1 >= 0 && x0 + 1 < W;
        const bool iny0 = y0 >= 0 && y0 < H, iny1 = y0 + 1 >= 0 && y0 + 1 < H;
        for (int ch = 0; ch < C; ++ch) {
            const float* plane = img + ((size_t)n * C + ch) * H * W;
            float acc = 0.0f;
            if (iny0 && inx0) acc = __fmaf_rn(__ldg(plane + (size_t)y0 * W + x0), wx0 * wy0, acc);
            if (iny0 && inx1) acc = __fmaf_rn(__ldg(plane + (size_t)y0 * W + x0 + 1), wx1 * wy0, acc);
            if (iny1 && inx0) acc = __fmaf_rn(__ldg(plane + (size_t)(y0 + 1) * W + x0), wx0 * wy1, acc);
            if (iny1 && inx1) acc = __fmaf_rn(__ldg(plane + (size_t)(y0 + 1) * W + x0 + 1), wx1 * wy1, acc);
            out[((size_t)n * C + ch) * HWo + p] = acc;
        }
    }
}

// window rows per cp.async commit group: 3 for radius 4 (measured ~2 % faster than one group for the whole window)
template <typename T>
int launch_tile(const LookupParams& P, const float* coords, float* out, int32_t* idx, uint8_t* valid, int radius,
                int blocks, int threads, size_t wsm, cudaStream_t st) {
    OFB_CUDA(ofb_smem_once<lookup_tile_kernel<4, 3, T>>(11 * 128 * 40));
    OFB_CUDA(ofb_smem_once<lookup_tile_kernel<3, 16, T>>(9 * 128 * 40));
    if (radius == 4) lookup_tile_kernel<4, 3, T><<<blocks, threads, wsm, st>>>(P, coords, out, idx, valid);
    else lookup_tile_kernel<3, 16, T><<<blocks, threads, wsm, st>>>(P, coords, out, idx, valid);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

}  // namespace

OFB_API int ofb_corr_lookup(const ofb_pyramid* pyr, const float* coords, float* out, int32_t* idx_or_null,
                            uint8_t* valid_or_null, int B, int h, int w, int radius, void* stream) {
    if (B == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!pyr || !coords || !out || B < 0 || h <= 0 || w <= 0) return OFB_EINVAL;
    if (radius < 0 || 2 * radius + 1 > MAX_D) return OFB_EUNSUPPORTED;
    if (pyr->dtype != OFB_DTYPE_F32 && pyr->dtype != OFB_DTYPE_BF16 && pyr->dtype != OFB_DTYPE_F16) return OFB_EINVAL;
    if (pyr->layout < OFB_LAYOUT_ROWS || pyr->layout > OFB_LAYOUT_QMINOR8X4) return OFB_EINVAL;
    const bool half16 = pyr->dtype != OFB_DTYPE_F32;      // 16-bit storage: bf16 or fp16
    LookupParams P;
    if (const int rc = ofb::unpack_levels(*pyr, P)) return rc;
    P.levels = pyr->levels; P.radius = radius; P.B = B; P.h = h; P.w = w;
    P.blocked = pyr->layout != OFB_LAYOUT_ROWS;
    P.blk_stride = pyr->layout == OFB_LAYOUT_QMINOR8X4 ? 32LL * B * h * w : 32LL;
    for (int l = 0; l < P.levels; ++l) {
        if (P.lh[l] > 65536 || P.lw[l] > 65536) return OFB_EUNSUPPORTED;
        if (half16 && ((P.pitch[l] & 1) || (P.q_stride[l] & 1) || (reinterpret_cast<uintptr_t>(P.base[l]) & 3)))
            return OFB_EALIGN;
    }
    const int D = 2 * radius + 1, CH = pyr->levels * D * D;
    const size_t smem = ((size_t)CH * OT_PITCH + (size_t)NW * PD * PD) * sizeof(float);
    const long long Q = (long long)B * h * w;
    const long long blocks = (Q + QT - 1) / QT;
    if (blocks > 0x7fffffffLL) return OFB_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    // product path: 16-bit pyramid with padded rows (pitch multiple of 8, 16-byte aligned slices)
    bool tile_ok = half16 && (radius == 4 || radius == 3);
    for (int l = 0; l < pyr->levels && tile_ok; ++l)
        tile_ok = (P.pitch[l] % 8 == 0) && (P.q_stride[l] % 8 == 0) && ((reinterpret_cast<uintptr_t>(P.base[l]) & 15) == 0);
    if (tile_ok) {
        const int threads = 32 * pyr->levels;
        const size_t wsm = (size_t)(2 * radius + 3) * threads * 40;               // window slots: rows x (16 + 16 + 8) B
        if (pyr->dtype == OFB_DTYPE_F16) return launch_tile<__half>(P, coords, out, idx_or_null, valid_or_null, radius,
                                                                    (int)blocks, threads, wsm, st);
        return launch_tile<__nv_bfloat16>(P, coords, out, idx_or_null, valid_or_null, radius, (int)blocks, threads, wsm, st);
    }
    if (P.blocked) return OFB_EUNSUPPORTED;   // the generic kernels read rows
    if (pyr->dtype == OFB_DTYPE_BF16) {
        OFB_CUDA(cudaFuncSetAttribute(lookup_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lookup_kernel<__nv_bfloat16><<<(int)blocks, NW * 32, smem, st>>>(P, coords, out, idx_or_null, valid_or_null);
    } else if (pyr->dtype == OFB_DTYPE_F16) {
        OFB_CUDA(cudaFuncSetAttribute(lookup_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lookup_kernel<__half><<<(int)blocks, NW * 32, smem, st>>>(P, coords, out, idx_or_null, valid_or_null);
    } else {
        OFB_CUDA(cudaFuncSetAttribute(lookup_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lookup_kernel<float><<<(int)blocks, NW * 32, smem, st>>>(P, coords, out, idx_or_null, valid_or_null);
    }
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_bilinear_sampler_f32(const float* img, const float* coords, float* out, float* mask_or_null, int N, int C,
                                     int H, int W, int Ho, int Wo, void* stream) {
    if (N == 0 || C == 0 || Ho == 0 || Wo == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!img || !coords || !out || N < 0 || C < 0 || H <= 0 || W <= 0 || Ho < 0 || Wo < 0) return OFB_EINVAL;
    const size_t total = (size_t)N * Ho * Wo;
    if (total == 0) return OFB_OK;
    int blocks = (int)((total + 255) / 256);
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    bilinear_sampler_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(img, coords, out, mask_or_null, N, C, H, W, Ho, Wo);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
