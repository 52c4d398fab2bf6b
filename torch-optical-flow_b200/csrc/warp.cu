// warp.cu -- K1: flow-based backward warp (bilinear / nearest) + in-kernel validity mask.
//
// Replaces optical_flow.warp + warp_grid (reference optical_flow/operator/operator.py:8-56):
//   gx = linspace(-1,1,W)[j] + flow[b,0,i,j] ; gy = linspace(-1,1,H)[i] + flow[b,1,i,j]
//   out[b,c,i,j] = grid_sample(frame[b,c], (gx,gy), mode, padding_mode, align_corners)
// Neither the base grid nor grid+flow is ever materialised.
//
// Bilinear NCHW kernels (variant argument of ofb_warp / ofb_warp_f32; all produce the same bits):
//   * rows (default): lane <-> column, a thread owns 2 consecutive rows of its column, coordinates / weights /
//     tap offsets computed once per pixel and reused per channel; interior pixels take a predicate-free channel
//     loop with every gather in flight before the first FMA.  32 registers -> 64 resident warps per SM: the
//     kernel is bound by latency and instruction issue, not by HBM (DESIGN.md section 4).
//   * direct: one thread per output pixel, grid-stride; also serves nearest mode and NHWC frames.
//   * staged: one CTA per 64x16 output tile, bounding box of the taps copied to shared memory with cp.async.
//   * TMA window (warp_tma.cu): persistent CTAs, the tile's neighbourhood arrives as 3-D TMA boxes.
// HBM roofline (SURVEY.md 8d): 4*(C + 2 + C) bytes per pixel (+1 for the u8 mask); 2 per frame or flow element instead
// of 4 for a 16-bit one (the direct and row kernels read frames and flows in fp32, fp16 or bf16; the output is fp32).
#include <cstdlib>

#include "common.cuh"

namespace {

using namespace ofb;

// ------------------------------------------------------------------------------ direct kernel
// TI, TV: element types of the frame and the flow (float, __half, __nv_bfloat16), each widened exactly on load; the
// arithmetic is the fp32 kernel's.  A 16-bit NHWC frame takes the scalar gather4 path: a float4-style 8-byte load of 4
// halves would add a second vector path (and its alignment rule) to a kernel that is not the default, for a warp that
// is bound by issue and latency rather than bytes (DESIGN.md section 4).
template <int MODE, int PAD, bool AC, bool NHWC, typename TI = float, typename TV = float>
__global__ void __launch_bounds__(256) warp_direct_kernel(const TI* __restrict__ frame, const TV* __restrict__ flow,
                                                          float* __restrict__ out, uint8_t* __restrict__ valid, int B,
                                                          int C, int H, int W, FlowMul fm) {
    const size_t HW = (size_t)H * W;
    const size_t total = (size_t)B * HW;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(q / HW);
        const size_t p = q - (size_t)b * HW;
        const int i = (int)(p / W), j = (int)(p - (size_t)i * W);
        const TV* fxp = flow + (size_t)b * 2 * HW + p;
        const SrcPos s = warp_source<PAD, AC>(ld_f32(fxp), ld_f32(fxp + HW), i, j, H, W, fm);
        if (valid) valid[q] = s.valid ? 1 : 0;
        if (MODE == OFB_MODE_NEAREST) {
            const int x = tap_index(rintf(s.ix), W), y = tap_index(rintf(s.iy), H);
            const bool in = x >= 0 && x < W && y >= 0 && y < H;
            if constexpr (std::is_same<TI, float>::value) {
                for (int c = 0; c < C; ++c) {
                    float v = 0.0f;
                    if (in) v = NHWC ? ld_f32(frame + ((size_t)b * HW + (size_t)y * W + x) * C + c)
                                     : ld_f32(frame + ((size_t)b * C + c) * HW + (size_t)y * W + x);
                    out[((size_t)b * C + c) * HW + p] = v;
                }
            } else {
                // the same loop, kept rolled: unrolled, ptxas spills a register in the fp16-frame border instances
#pragma unroll 1
                for (int c = 0; c < C; ++c) {
                    float v = 0.0f;
                    if (in) v = NHWC ? ld_f32(frame + ((size_t)b * HW + (size_t)y * W + x) * C + c)
                                     : ld_f32(frame + ((size_t)b * C + c) * HW + (size_t)y * W + x);
                    out[((size_t)b * C + c) * HW + p] = v;
                }
            }
            continue;
        }
        const BilinearTaps t = bilinear_taps<PAD>(s.ix, s.iy, H, W);
        if (NHWC && !t.inb) {
            // no tap in the frame: 0, which the float4 path would not give for the NaN weights of a non-finite position
            for (int c = 0; c < C; ++c) out[((size_t)b * C + c) * HW + p] = 0.0f;
            continue;
        }
        if (NHWC) {
            const TI* p00 = frame + ((size_t)b * HW + (size_t)t.y0 * W + t.x0) * C;
            const size_t row = (size_t)W * C;
            if (std::is_same<TI, float>::value && (C & 3) == 0) {
                const TI *p01 = p00 + C, *p10 = p00 + row, *p11 = p10 + C;
                for (int c = 0; c < C; c += 4) {
                    float4 a = make_float4(0, 0, 0, 0), bb = a, cc = a, dd = a;
                    if (t.inb & 1u) a = __ldg(reinterpret_cast<const float4*>(p00 + c));
                    if (t.inb & 2u) bb = __ldg(reinterpret_cast<const float4*>(p01 + c));
                    if (t.inb & 4u) cc = __ldg(reinterpret_cast<const float4*>(p10 + c));
                    if (t.inb & 8u) dd = __ldg(reinterpret_cast<const float4*>(p11 + c));
                    float r0 = __fmaf_rn(dd.x, t.w11, __fmaf_rn(cc.x, t.w10, __fmaf_rn(bb.x, t.w01, a.x * t.w00)));
                    float r1 = __fmaf_rn(dd.y, t.w11, __fmaf_rn(cc.y, t.w10, __fmaf_rn(bb.y, t.w01, a.y * t.w00)));
                    float r2 = __fmaf_rn(dd.z, t.w11, __fmaf_rn(cc.z, t.w10, __fmaf_rn(bb.z, t.w01, a.z * t.w00)));
                    float r3 = __fmaf_rn(dd.w, t.w11, __fmaf_rn(cc.w, t.w10, __fmaf_rn(bb.w, t.w01, a.w * t.w00)));
                    out[((size_t)b * C + c + 0) * HW + p] = r0;
                    out[((size_t)b * C + c + 1) * HW + p] = r1;
                    out[((size_t)b * C + c + 2) * HW + p] = r2;
                    out[((size_t)b * C + c + 3) * HW + p] = r3;
                }
            } else {
                for (int c = 0; c < C; ++c) out[((size_t)b * C + c) * HW + p] = gather4(p00 + c, C, row, t);
            }
        } else {
            const size_t o00 = (size_t)t.y0 * W + t.x0;
            for (int c = 0; c < C; ++c)
                out[((size_t)b * C + c) * HW + p] = gather4(frame + ((size_t)b * C + c) * HW + o00, 1, W, t);
        }
    }
}

// ------------------------------------------------------------------------------ staged kernel
constexpr int TW = 64, TH = 16, NT = 256, PPT = (TW * TH) / NT;  // 4 pixels per thread
constexpr int MARGIN = 16;                                        // staged window = tile +- MARGIN
constexpr int WIN_W = TW + 2 * MARGIN + 8;                        // +8: 16-byte alignment slack on both sides
constexpr int WIN_H = TH + 2 * MARGIN + 2;
constexpr int CG_MAX = 4;                                         // channels staged per pass

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// Takes its taps in the guarded (zeros) form under every padding, valid for clipped coordinates too.  With that and
// the 2 CTAs per SM its shared memory allows at CG_MAX channels, every instance compiles to 96 registers, no spills.
template <int PAD, bool AC>
__global__ void __launch_bounds__(NT, 2) warp_staged_kernel(const float* __restrict__ frame, const float* __restrict__ flow,
                                                            float* __restrict__ out, uint8_t* __restrict__ valid, int B,
                                                            int C, int H, int W, int vec4, FlowMul fm) {
    extern __shared__ __align__(16) float win[];  // [cg][WIN_H][pitch]
    __shared__ int s_box[4];                      // min x, max x, min y, max y of the taps
    const int b = blockIdx.z;
    const int tile_x = blockIdx.x * TW, tile_y = blockIdx.y * TH;
    const int tx = threadIdx.x % TW, ty = threadIdx.x / TW;  // ty in [0, NT/TW)
    const size_t HW = (size_t)H * W;

    if (threadIdx.x == 0) { s_box[0] = INT_MAX; s_box[1] = INT_MIN; s_box[2] = INT_MAX; s_box[3] = INT_MIN; }
    __syncthreads();

    float ix[PPT], iy[PPT];
    int bx0 = INT_MAX, bx1 = INT_MIN, by0 = INT_MAX, by1 = INT_MIN;
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
        const int i = tile_y + ty + k * (NT / TW), j = tile_x + tx;
        ix[k] = 0.0f; iy[k] = 0.0f;
        if (i < H && j < W) {
            const float* fxp = flow + (size_t)b * 2 * HW + (size_t)i * W + j;
            const SrcPos s = warp_source<PAD, AC>(__ldg(fxp), __ldg(fxp + HW), i, j, H, W, fm);
            ix[k] = s.ix; iy[k] = s.iy;
            if (valid) valid[(size_t)b * HW + (size_t)i * W + j] = s.valid ? 1 : 0;
            const BilinearTaps t = bilinear_taps<OFB_PAD_ZEROS>(s.ix, s.iy, H, W);
            bx0 = min(bx0, t.x0); bx1 = max(bx1, t.x0 + 1);
            by0 = min(by0, t.y0); by1 = max(by1, t.y0 + 1);
        }
    }
    bx0 = warp_min(bx0); bx1 = warp_max(bx1); by0 = warp_min(by0); by1 = warp_max(by1);
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&s_box[0], bx0); atomicMax(&s_box[1], bx1);
        atomicMin(&s_box[2], by0); atomicMax(&s_box[3], by1);
    }
    __syncthreads();
    // staged window: tap bounding box, clamped to tile +- MARGIN and to the frame
    int wx_lo = max(max(s_box[0], tile_x - MARGIN), 0);
    int wx_hi = min(min(s_box[1], tile_x + TW - 1 + MARGIN), W - 1);
    int wy_lo = max(max(s_box[2], tile_y - MARGIN), 0);
    int wy_hi = min(min(s_box[3], tile_y + TH - 1 + MARGIN), H - 1);
    if (vec4) { wx_lo &= ~3; wx_hi |= 3; if (wx_hi > W - 1) wx_hi = W - 1; }
    const int ww = wx_hi - wx_lo + 1, wh = wy_hi - wy_lo + 1;  // may be <= 0: nothing staged
    const int pitch = vec4 ? ww : (ww | 1);
    const int plane_sz = pitch * max(wh, 0);

    for (int c0 = 0; c0 < C; c0 += CG_MAX) {
        const int cg = min(CG_MAX, C - c0);
        if (ww > 0 && wh > 0) {
            if (vec4) {
                const int w4 = ww >> 2, per_c = w4 * wh;
                for (int e = threadIdx.x; e < per_c * cg; e += NT) {
                    int c = e / per_c, r = e - c * per_c;
                    int yy = r / w4, x4 = r - yy * w4;
                    const float* src = frame + ((size_t)b * C + c0 + c) * HW + (size_t)(wy_lo + yy) * W + wx_lo + x4 * 4;
                    cp_async16(win + c * plane_sz + yy * pitch + x4 * 4, src);
                }
                cp_async_wait_all();
            } else {
                const int per_c = ww * wh;
                for (int e = threadIdx.x; e < per_c * cg; e += NT) {
                    int c = e / per_c, r = e - c * per_c;
                    int yy = r / ww, xx = r - yy * ww;
                    win[c * plane_sz + yy * pitch + xx] =
                        __ldg(frame + ((size_t)b * C + c0 + c) * HW + (size_t)(wy_lo + yy) * W + wx_lo + xx);
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
            const int i = tile_y + ty + k * (NT / TW), j = tile_x + tx;
            if (i >= H || j >= W) continue;
            const BilinearTaps t = bilinear_taps<OFB_PAD_ZEROS>(ix[k], iy[k], H, W);
            const bool fast = t.x0 >= wx_lo && t.x0 + 1 <= wx_hi && t.y0 >= wy_lo && t.y0 + 1 <= wy_hi;
            const size_t p = (size_t)i * W + j;
            if (fast) {
                const float* s00 = win + (t.y0 - wy_lo) * pitch + (t.x0 - wx_lo);
                for (int c = 0; c < cg; ++c) {
                    const float* s = s00 + c * plane_sz;
                    float acc = s[0] * t.w00;
                    acc = __fmaf_rn(s[1], t.w01, acc);
                    acc = __fmaf_rn(s[pitch], t.w10, acc);
                    acc = __fmaf_rn(s[pitch + 1], t.w11, acc);
                    out[((size_t)b * C + c0 + c) * HW + p] = acc;
                }
            } else {
                const size_t o00 = (size_t)t.y0 * W + t.x0;
                for (int c = 0; c < cg; ++c) {
                    const float* plane = frame + ((size_t)b * C + c0 + c) * HW;
                    out[((size_t)b * C + c0 + c) * HW + p] = gather4(plane + o00, 1, W, t);
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------ row kernel
// The default NCHW bilinear path.  grid = (column groups, row groups, batch): no per-pixel integer division,
// 32-bit in-plane offsets.  Lane <-> column (every load / store of a warp is one or two 128-byte lines), and a
// thread walks RPT consecutive rows of its column: the lower taps of row i are the upper taps of row i+1 for
// smooth flows, so they hit L1.  The coordinate pipeline and the 4 tap offsets are computed once per pixel
// and reused for every channel.
constexpr int RPT_DEFAULT = 2;   // rows per thread: 32 registers, 64 resident warps per SM (see the sweep in DESIGN.md)

// TI, TV: element types of the frame and the flow, as in the direct kernel.
template <int PAD, bool AC, int RPT, typename TI = float, typename TV = float>
__global__ void __launch_bounds__(128) warp_rows_kernel(const TI* __restrict__ frame, const TV* __restrict__ flow,
                                                        float* __restrict__ out, uint8_t* __restrict__ valid, int C,
                                                        int H, int W, FlowMul fm) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.z;
    const int i0 = blockIdx.y * RPT;
    if (j >= W) return;
    const int HW = H * W;                                     // launch guard: H*W < 2^30
    const TV* fxp = flow + (size_t)(b * 2) * HW;
    const TV* fyp = fxp + HW;
    int o00[RPT];
    float w00[RPT], w01[RPT], w10[RPT], w11[RPT];
    unsigned inb = 0;
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
        const int i = i0 + k;
        o00[k] = 0; w00[k] = w01[k] = w10[k] = w11[k] = 0.0f;
        if (i >= H) continue;
        const int off = i * W + j;
        const SrcPos s = warp_source<PAD, AC>(ld_f32(fxp + off), ld_f32(fyp + off), i, j, H, W, fm);
        if (valid) valid[(size_t)b * HW + off] = s.valid ? 1 : 0;
        const BilinearTaps t = bilinear_taps<PAD>(s.ix, s.iy, H, W);
        w00[k] = t.w00; w01[k] = t.w01; w10[k] = t.w10; w11[k] = t.w11;
        inb |= t.inb << (4 * k);
        o00[k] = t.y0 * W + t.x0;
    }
    // interior pixels (all 4 x RPT taps inside the frame -- everything but the last row / column and, under zeros
    // padding, samples that leave the frame): no predicates, no per-tap address arithmetic.  The kernel is bound
    // by instruction issue, not by HBM, so the channel loop is kept to 4 loads + 4 FMAs + 1 store per pixel.
    if (inb == (RPT == 8 ? 0xFFFFFFFFu : (1u << (4 * RPT)) - 1u)) {
        const TI* plane = frame + (size_t)(b * C) * HW;
        float* op = out + (size_t)(b * C) * HW + i0 * W + j;
#pragma unroll 1
        for (int c = 0; c < C; ++c, plane += HW, op += HW) {
            float v[RPT][4];                              // all 4 x RPT gathers in flight before the first FMA
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                const TI* p = plane + o00[k];
                const TI* q = p + W;
                v[k][0] = ld_f32(p); v[k][1] = ld_f32(p + 1); v[k][2] = ld_f32(q); v[k][3] = ld_f32(q + 1);
            }
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                float acc = __fmaf_rn(v[k][0], w00[k], 0.0f);
                acc = __fmaf_rn(v[k][1], w01[k], acc);
                acc = __fmaf_rn(v[k][2], w10[k], acc);
                acc = __fmaf_rn(v[k][3], w11[k], acc);
                op[k * W] = acc;
            }
        }
        return;
    }
    for (int c = 0; c < C; ++c) {
        const TI* plane = frame + (size_t)(b * C + c) * HW;
        float* op = out + (size_t)(b * C + c) * HW + i0 * W + j;
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            if (i0 + k >= H) continue;
            op[k * W] = gather4(plane + o00[k], 1, W, inb >> (4 * k), w00[k], w01[k], w10[k], w11[k]);
        }
    }
}

__global__ void __launch_bounds__(256) warp_grid_kernel(const float* __restrict__ flow, float* __restrict__ grid, int B,
                                                        int H, int W) {
    const size_t total = (size_t)B * H * W;
    const float step_x = linspace_step(W), step_y = linspace_step(H);
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(q % W), i = (int)((q / W) % H);
        float2 f = __ldg(reinterpret_cast<const float2*>(flow) + q);
        float2 g;
        g.x = __fadd_rn(linspace_m1_p1(j, W, step_x), f.x);
        g.y = __fadd_rn(linspace_m1_p1(i, H, step_y), f.y);
        reinterpret_cast<float2*>(grid)[q] = g;
    }
}

template <int MODE, int PAD, bool AC, typename TI, typename TV>
int launch_direct(const TI* frame, const TV* flow, float* out, uint8_t* valid, int B, int C, int H, int W,
                  int channels_last, FlowMul fm, cudaStream_t st) {
    const size_t total = (size_t)B * H * W;
    int blocks = (int)((total + 255) / 256);
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    if (channels_last)
        warp_direct_kernel<MODE, PAD, AC, true, TI, TV><<<blocks, 256, 0, st>>>(frame, flow, out, valid, B, C, H, W, fm);
    else
        warp_direct_kernel<MODE, PAD, AC, false, TI, TV><<<blocks, 256, 0, st>>>(frame, flow, out, valid, B, C, H, W, fm);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

// Rows per thread of the fp32 row kernel: RPT_DEFAULT, or the OFB_WARP_RPT tuning override
int warp_rpt() {
    static const int rpt = [] {
        const char* e = getenv("OFB_WARP_RPT");
        const int r = e ? atoi(e) : RPT_DEFAULT;
        return (r == 1 || r == 2 || r == 4 || r == 8) ? r : RPT_DEFAULT;
    }();
    return rpt;
}

// A 16-bit frame or flow runs the row kernel at RPT_DEFAULT only: the override is an fp32 tuning knob, and the
// 16-bit instances stay one per (frame, flow, padding, align_corners).
template <int PAD, bool AC, typename TI, typename TV>
int launch_rows(const TI* frame, const TV* flow, float* out, uint8_t* valid, int B, int C, int H, int W,
                FlowMul fm, cudaStream_t st) {
    constexpr bool f32 = std::is_same<TI, float>::value && std::is_same<TV, float>::value;
    const int rpt = f32 ? warp_rpt() : RPT_DEFAULT;
    const dim3 block(128);
    const dim3 grid((W + 127) / 128, (H + rpt - 1) / rpt, B);
    if (grid.y > 65535) return OFB_EUNSUPPORTED;
    if constexpr (f32) {
        if (rpt == 1) warp_rows_kernel<PAD, AC, 1><<<grid, block, 0, st>>>(frame, flow, out, valid, C, H, W, fm);
        else if (rpt == 2) warp_rows_kernel<PAD, AC, 2><<<grid, block, 0, st>>>(frame, flow, out, valid, C, H, W, fm);
        else if (rpt == 8) warp_rows_kernel<PAD, AC, 8><<<grid, block, 0, st>>>(frame, flow, out, valid, C, H, W, fm);
        else warp_rows_kernel<PAD, AC, 4><<<grid, block, 0, st>>>(frame, flow, out, valid, C, H, W, fm);
    } else {
        warp_rows_kernel<PAD, AC, RPT_DEFAULT, TI, TV><<<grid, block, 0, st>>>(frame, flow, out, valid, C, H, W, fm);
    }
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

template <int PAD, bool AC>
int launch_staged(const float* frame, const float* flow, float* out, uint8_t* valid, int B, int C, int H, int W,
                  FlowMul fm, cudaStream_t st) {
    const int cg = C < CG_MAX ? C : CG_MAX;
    const size_t smem = (size_t)cg * WIN_H * WIN_W * sizeof(float);
    OFB_CUDA(ofb_smem_once<warp_staged_kernel<PAD, AC>>((int)(CG_MAX * WIN_H * WIN_W * sizeof(float))));
    const int vec4 = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(frame) & 15) == 0);
    dim3 grid((W + TW - 1) / TW, (H + TH - 1) / TH, B);
    warp_staged_kernel<PAD, AC><<<grid, NT, smem, st>>>(frame, flow, out, valid, B, C, H, W, vec4, fm);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

}  // namespace

// warp_tma.cu
int ofb_warp_tma_launch(const float* frame, const float* flow, float* out, uint8_t* valid, int B, int C, int H, int W,
                        int pad, int ac, const ofb::FlowMul& fm, cudaStream_t st);

OFB_API int ofb_warp(const void* frame, int frame_dtype, const void* flow, int flow_dtype, float* out,
                     uint8_t* valid_or_null, int B, int C, int H, int W, int mode, int padding_mode, int align_corners,
                     int channels_last, int variant, float flow_mul_x, float flow_mul_y, void* stream) {
    if (!ofb_float_dtype(frame_dtype) || !ofb_float_dtype(flow_dtype)) return OFB_EINVAL;
    if (B == 0 || C == 0 || H == 0 || W == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!frame || !flow || !out || B < 0 || C < 0 || H < 0 || W < 0) return OFB_EINVAL;
    if (mode != OFB_MODE_BILINEAR && mode != OFB_MODE_NEAREST) return OFB_EINVAL;
    if (padding_mode < 0 || padding_mode > 2 || variant < 0 || variant > 4) return OFB_EINVAL;
    if ((size_t)B * C * H * W == 0) return OFB_OK;
    const bool f32 = frame_dtype == OFB_DTYPE_F32 && flow_dtype == OFB_DTYPE_F32;
    if ((frame_dtype != OFB_DTYPE_F32 && (reinterpret_cast<uintptr_t>(frame) & 1)) ||
        (flow_dtype != OFB_DTYPE_F32 && (reinterpret_cast<uintptr_t>(flow) & 1)))
        return OFB_EALIGN;
    if (B > 65535) return OFB_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const FlowMul fm{flow_mul_x, flow_mul_y, ofb::linspace_step(W), ofb::linspace_step(H)};
    const bool nchw_bilinear = mode == OFB_MODE_BILINEAR && !channels_last;
    const bool can_rows = nchw_bilinear && H <= 65535 * RPT_DEFAULT && (long long)H * W < (1LL << 30) && (long long)B * C * H * W < (1LL << 40);
    // TMA needs 16-byte global strides
    const bool can_tma = can_rows && W % 4 == 0 && (reinterpret_cast<uintptr_t>(frame) & 15) == 0 &&
                         (long long)B * C < (1LL << 31);
    // the staged and TMA kernels read fp32 frames and flows only
    if (((variant == 2 || variant == 4) && !f32) || (variant == 2 && !nchw_bilinear) || (variant == 3 && !can_rows) ||
        (variant == 4 && !can_tma))
        return OFB_EUNSUPPORTED;
    // auto: the row kernel; 1 = direct gather (also nearest / NHWC), 2 = cp.async-staged, 3 = row kernel,
    // 4 = TMA-staged window (warp_tma.cu)
    static const int auto_v = [] {
        const char* e = getenv("OFB_WARP_VARIANT");       // tuning override for variant 0
        return e ? atoi(e) : 0;
    }();
    int v = variant != 0 ? variant : (auto_v == 4 && can_tma && f32 ? 4 : (can_rows ? 3 : 1));
    if (v == 4)
        return ofb_warp_tma_launch(static_cast<const float*>(frame), static_cast<const float*>(flow), out,
                                   valid_or_null, B, C, H, W, padding_mode, align_corners, fm, st);
    if (v == 2)
        return ofb_dispatch_pad_ac(padding_mode, align_corners, [&](auto P, auto A) {
            return launch_staged<P, A>(static_cast<const float*>(frame), static_cast<const float*>(flow), out,
                                       valid_or_null, B, C, H, W, fm, st);
        });
    return ofb_dispatch_dtype(frame_dtype, [&](auto ti) {
        return ofb_dispatch_dtype(flow_dtype, [&](auto tv) {
            using TI = decltype(ti);
            using TV = decltype(tv);
            const TI* fr = static_cast<const TI*>(frame);
            const TV* fl = static_cast<const TV*>(flow);
            return ofb_dispatch_pad_ac(padding_mode, align_corners, [&](auto P, auto A) {
                if (v == 3) return launch_rows<P, A>(fr, fl, out, valid_or_null, B, C, H, W, fm, st);
                const int cl = channels_last;
                if (mode == OFB_MODE_BILINEAR)
                    return launch_direct<OFB_MODE_BILINEAR, P, A>(fr, fl, out, valid_or_null, B, C, H, W, cl, fm, st);
                return launch_direct<OFB_MODE_NEAREST, P, A>(fr, fl, out, valid_or_null, B, C, H, W, cl, fm, st);
            });
        });
    });
}

OFB_API int ofb_warp_f32(const float* frame, const float* flow, float* out, uint8_t* valid_or_null, int B, int C, int H,
                         int W, int mode, int padding_mode, int align_corners, int channels_last, int variant,
                         float flow_mul_x, float flow_mul_y, void* stream) {
    return ofb_warp(frame, OFB_DTYPE_F32, flow, OFB_DTYPE_F32, out, valid_or_null, B, C, H, W, mode, padding_mode,
                    align_corners, channels_last, variant, flow_mul_x, flow_mul_y, stream);
}

OFB_API int ofb_warp_grid_f32(const float* flow_bhw2, float* grid_bhw2, int B, int H, int W, void* stream) {
    if (B == 0 || H == 0 || W == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!flow_bhw2 || !grid_bhw2 || B < 0 || H < 0 || W < 0) return OFB_EINVAL;
    const size_t total = (size_t)B * H * W;
    if (total == 0) return OFB_OK;
    int blocks = (int)((total + 255) / 256);
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    warp_grid_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(flow_bhw2, grid_bhw2, B, H, W);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
