/*
 * ofb200.h -- C ABI of libofb200.so: hand-written sm_100a kernels for the data-parallel hot
 * path of awaelchli/torch-optical-flow (flow warp + validity mask, flow resize / upsampling,
 * RAFT correlation pyramid + lookup, end-point-error reduction).
 *
 * The reference is pure Python and has no FFI layer: its boundary is the Python call
 * surface (optical_flow.operator, methods/raft/model).  Each entry point below replaces the
 * ATen op sequence behind one reference function; the Python shims in
 * torch-optical-flow_b200/{optical_flow,model}/ keep the reference's names, arguments and
 * error behaviour and call these through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless a name ends in
 *     _host; tensors are dense row-major in the layouts stated per function
 *   - the last argument is the CUDA stream (cudaStream_t passed as void*; NULL = default)
 *   - returns 0 on success, a negative OFB_E* code for a rejected argument, or a positive
 *     cudaError_t for a CUDA failure; never throws, never allocates device memory, never
 *     synchronises (ofb_corr_pyramid_bf16*, ofb_corr_pyramid_f16, ofb_gemm_nt_bf16 and the TMA variant of ofb_warp_f32
 *     are the only calls that touch the driver outside a stream: they encode TMA descriptors on the host)
 *   - there is no CPU compute path: without a CUDA device every call fails
 */
#ifndef OFB200_H_
#define OFB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFB_VERSION 120

#define OFB_OK 0
#define OFB_EINVAL (-1)       /* bad size / null pointer / unsupported enum value          */
#define OFB_EUNSUPPORTED (-2) /* valid request this build has no kernel for              */
#define OFB_EALIGN (-3)       /* pointer or pitch not aligned as the kernel requires     */
#define OFB_EDRIVER (-4)      /* driver entry point (cuTensorMapEncodeTiled) unavailable */

#define OFB_MODE_BILINEAR 0
#define OFB_MODE_NEAREST 1
#define OFB_PAD_ZEROS 0
#define OFB_PAD_BORDER 1
#define OFB_PAD_REFLECTION 2

#define OFB_DTYPE_F32 0
#define OFB_DTYPE_BF16 1
#define OFB_DTYPE_F16 2 /* feature maps and operands of ofb_corr_prep_from / _to, correlation pyramids, mask of
                           ofb_convex_upsample and its gradient, ofb_scale_flow, the lookup's output and its gradient */
#define OFB_DTYPE_F64 3 /* ofb_scale_flow only */

#define OFB_MAX_LEVELS 4

int ofb_version(void);
const char* ofb_strerror(int code);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
int64_t ofb_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * K1  backward warp + validity mask.
 * Replaces optical_flow.warp (optical_flow/operator/operator.py:8-33) including warp_grid
 * (operator.py:36-56): grid = (linspace(-1,1,W)[j] + flow_x, linspace(-1,1,H)[i] + flow_y),
 * out = grid_sample(frame, grid, mode, padding_mode, align_corners).
 *   frame (B,C,H,W) fp32 NCHW, or (B,H,W,C) when channels_last != 0
 *   flow  (B,2,H,W) fp32, normalised units (optical_flow.normalize)
 *   out   (B,C,H,W) fp32 NCHW
 *   valid_or_null (B,H,W) u8: 1 iff -1 < grid < 1 on both axes -- the predicate of
 *                 bilinear_sampler's mask (methods/raft/model/utils.py:76-78)
 *   variant: 0 = auto, 1 = direct gather, 2 = shared-memory staged neighbourhood (cp.async), 3 = row kernel,
 *            4 = TMA-staged neighbourhood (bilinear NCHW, W % 4 == 0, 16-byte aligned frame; else OFB_EUNSUPPORTED)
 *   flow_mul_x/y: the flow is multiplied by these (one rounded fp32 multiply) before the grid is
 *                 formed: 1, 1 for the reference's normalised flow; 2/max(W-1,1), 2/max(H-1,1) fuses
 *                 optical_flow.normalize (operator.py:117-130) for pixel-unit flows, bit-identically
 * ------------------------------------------------------------------------------------- */
int ofb_warp_f32(const float* frame, const float* flow, float* out, uint8_t* valid_or_null,
                 int B, int C, int H, int W, int mode, int padding_mode, int align_corners,
                 int channels_last, int variant, float flow_mul_x, float flow_mul_y, void* stream);

/* Backward of ofb_warp_f32 (bilinear, NCHW): what autograd computes for the reference's warp
 * (operator.py:28-33: grid_sample's backward, then d grid / d flow = 1 through warp_grid :56 and the
 * permute :28).  d_out (B,C,H,W).  d_frame_or_null (B,C,H,W) is ACCUMULATED into (zero it first):
 * each in-bounds tap receives weight * d_out.  d_flow_or_null (B,2,H,W) is overwritten, in the
 * units of `flow` (the flow_mul factors are applied).  Either output may be NULL. */
int ofb_warp_backward_f32(const float* frame, const float* flow, const float* d_out,
                          float* d_frame_or_null, float* d_flow_or_null, int B, int C, int H, int W,
                          int padding_mode, int align_corners, float flow_mul_x, float flow_mul_y,
                          void* stream);

/* warp_grid alone (operator.py:36-56): flow (B,H,W,2) -> grid (B,H,W,2). */
int ofb_warp_grid_f32(const float* flow_bhw2, float* grid_bhw2, int B, int H, int W, void* stream);

/* ---------------------------------------------------------------------------------------
 * scale / normalize / denormalize (operator.py:59-82,117-146): out[b,0] = in[b,0]*fx,
 * out[b,1] = in[b,1]*fy over (B,2,H,W) fp32.
 * ------------------------------------------------------------------------------------- */
int ofb_scale_flow_f32(const float* flow, float* out, int B, int64_t HW, float fx, float fy, void* stream);
/* The same multiply in the flow's own dtype (the reference's scale is dtype-preserving: the factor is filled into a tensor
 * of the flow's dtype, operator.py:79-80): dtype OFB_DTYPE_F32 / F64 / F16 / BF16. */
int ofb_scale_flow(const void* flow, void* out, int dtype, int B, int64_t HW, double fx, double fy, void* stream);

/* ---------------------------------------------------------------------------------------
 * K4a  bilinear resize with per-channel magnitude rescale.
 * Replaces F.interpolate(bilinear) + scale in optical_flow.resize (operator.py:85-114,
 * align_corners = 0) and 8 * F.interpolate(align_corners=True) in upflow8
 * (methods/raft/model/utils.py:89-91).  in (N,C,H,W) -> out (N,C,Ho,Wo); channel c is
 * multiplied by mul_x when c is even, mul_y when odd.
 * ------------------------------------------------------------------------------------- */
int ofb_resize_bilinear_f32(const float* in, float* out, int N, int C, int H, int W, int Ho, int Wo,
                            int align_corners, float mul_x, float mul_y, void* stream);
/* Its adjoint (autograd through F.interpolate + scale, operator.py:112-113; through upflow8,
 * utils.py:91): d_out (N,C,Ho,Wo) is scattered into d_in (N,C,H,W), which is ACCUMULATED into
 * (zero it first). */
int ofb_resize_bilinear_backward_f32(const float* d_out, float* d_in, int N, int C, int H, int W,
                                     int Ho, int Wo, int align_corners, float mul_x, float mul_y,
                                     void* stream);

/* ---------------------------------------------------------------------------------------
 * K4b  convex 8x flow upsampling.  Replaces RAFT.upsample_flow
 * (methods/raft/model/raft.py:73-85): flow (N,2,h,w), mask (N,576,h,w) -> out (N,2,8h,8w).
 * ------------------------------------------------------------------------------------- */
int ofb_convex_upsample_f32(const float* flow, const float* mask, float* out, int N, int h, int w, void* stream);
/* The same kernel reading the 576-channel mask in its own precision (mask_dtype OFB_DTYPE_F32 / BF16 / F16): under the
 * reference's `precision: 16` the mask head's output is half precision (the softmax of raft.py:78 autocasts to fp32, as
 * the kernel does after the load).  The flow and the result stay fp32. */
int ofb_convex_upsample(const float* flow, const void* mask, int mask_dtype, float* out, int N, int h, int w, void* stream);
/* Backward of the convex upsampling (autograd through raft.py:77-85): d_out (N,2,8h,8w), 16-byte
 * aligned.  d_mask_or_null (N,576,h,w) is overwritten; d_flow_or_null (N,2,h,w) is ACCUMULATED
 * into (zero it first).  Either may be NULL. */
int ofb_convex_upsample_backward_f32(const float* flow, const float* mask, const float* d_out,
                                     float* d_flow_or_null, float* d_mask_or_null, int N, int h, int w,
                                     void* stream);
/* The same backward with the mask in its own precision, mask_dtype OFB_DTYPE_F32 (= ofb_convex_upsample_backward_f32),
 * BF16 or F16; anything else is OFB_EINVAL.  d_mask_or_null is written in that dtype: each logit is widened exactly, the
 * gradient computed in fp32 with the arithmetic of the fp32 form and rounded once to nearest even -- the bits of the
 * fp32 gradient cast to the mask's dtype, which is what autocast's cast hands the mask head under `precision: 16`
 * (fp16: beyond +-65504 is inf).  flow, d_out and d_flow_or_null stay fp32.  A mask or d_mask not aligned to its
 * element size is OFB_EALIGN. */
int ofb_convex_upsample_backward(const float* flow, const void* mask, int mask_dtype, const float* d_out,
                                 float* d_flow_or_null, void* d_mask_or_null, int N, int h, int w, void* stream);

/* ---------------------------------------------------------------------------------------
 * K4c  end-point-error reduction.  Replaces AverageEndPointError.update
 * (optical_flow/metrics/epe.py:25-35): acc[0] += sum of sqrt(dx^2+dy^2) over pixels with
 * valid >= 0.5 (all pixels when valid_or_null is NULL), acc[1] += their count.
 * pred, target (B,2,H,W) fp32; valid (B,H,W) fp32; acc = double[2] on the device, updated
 * atomically (zero it before the first call; one ncclAllReduce(sum) of it gives the
 * dist_reduce_fx="sum" semantics of epe.py:22-23).
 * ofb_epe_map_f32: end_point_error(reduce=False) (epe.py:41-61) -> out (B,H,W).
 * ------------------------------------------------------------------------------------- */
int ofb_epe_reduce_f32(const float* pred, const float* target, const float* valid_or_null,
                       double* acc, int B, int H, int W, void* stream);
int ofb_epe_map_f32(const float* pred, const float* target, float* out, int B, int H, int W, void* stream);
/* OutlierRatio.update (optical_flow/metrics/f1.py:33-48): acc[0] += number of selected pixels with
 * epe > abs_threshold and epe / |target| > rel_threshold, acc[1] += number of selected pixels. */
int ofb_outlier_reduce_f32(const float* pred, const float* target, const float* valid_or_null,
                           double* acc, int B, int H, int W, float abs_threshold, float rel_threshold,
                           void* stream);
/* sequence_loss (methods/raft/model/raft.py:231-260), forward value, one fused pass:
 *   keep = (valid >= 0.5) & (|flow_gt|_2 < max_flow)
 *   acc[0] += sum_i gamma^(n-1-i) * sum(keep * |preds[i] - flow_gt|)   -> loss = acc[0] / (B*2*H*W)
 *   acc[1] += sum of the end-point error of preds[n-1] over kept pixels
 *   acc[2] += number of kept pixels; acc[3..5] += kept pixels with that error < 1, < 3, < 5 px
 *             -> the reference's "1px" / "3px" / "5px" metrics = acc[3..5] / acc[2]
 * preds: HOST array of n_predictions device pointers, each (B,2,H,W) fp32; n_predictions <=
 * OFB_MAX_PREDICTIONS; acc: 6 device doubles, accumulated (zero them first). */
#define OFB_MAX_PREDICTIONS 24
int ofb_sequence_loss_f32(const float* const* preds, int n_predictions, const float* flow_gt,
                          const float* valid, double* acc, int B, int H, int W, double gamma,
                          float max_flow, void* stream);
/* Its backward: d_preds[i] (HOST array of device pointers, NULL entries skipped) is overwritten with
 * grad_loss[0] * gamma^(n-1-i) / (B*2*H*W) * keep * sign(preds[i] - flow_gt); grad_loss is a DEVICE scalar. */
int ofb_sequence_loss_backward_f32(const float* const* preds, float* const* d_preds, int n_predictions,
                                   const float* flow_gt, const float* valid, const float* grad_loss,
                                   int B, int H, int W, double gamma, float max_flow, void* stream);

/* ---------------------------------------------------------------------------------------
 * Correlation pyramid layout (owned by the caller, described by ofb_pyramid_layout).
 * Level l of query q = (b, y, x) is an h_l x w_l image, h_l = floor(h / 2^l).  Two layouts
 * (strides in ELEMENTS of the pyramid dtype, `np` = row_pitch):
 *   OFB_LAYOUT_ROWS      element (q, yy, xx) at  base[l] + q*q_stride[l] + yy*np + xx
 *   OFB_LAYOUT_BLOCK8X4  8 (x) by 4 (y) element blocks of 32 contiguous elements (64 bytes in bf16 or fp16 =
 *                        one DRAM atom), blocks raster-ordered:
 *                        base[l] + q*q_stride[l] + ((yy>>2)*(np>>3) + (xx>>3))*32 + (yy&3)*8 + (xx&7)
 *                        -- the lookup's 11x11 window touches ~8 atoms instead of ~15.
 *   OFB_LAYOUT_QMINOR8X4 the same 8x4 blocks, but block-major / query-minor: with Q = B*h*w queries,
 *                        base[l] + (((yy>>2)*(np>>3) + (xx>>3))*Q + q)*32 + (yy&3)*8 + (xx&7)
 *                        (q_stride = 32).  Neighbouring queries' copies of one target block are
 *                        adjacent: the builder writes 2 KiB runs per warp, a lookup warp (32
 *                        consecutive queries) reads neighbouring 64-byte slots.  Level bases must be
 *                        32-byte aligned.
 * ofb_pyramid_layout fills the strides: mode 0 = tight rows (row_pitch = w_l), 1 = padded rows
* (row_pitch multiple of 16 elements, so every row starts on a 32-byte sector), 2 = padded 8x4
 * blocks (row_pitch multiple of 8, rows padded to a multiple of 4), 3 = the same blocks query-minor.
 * elems[l] receives the element count of level l PER QUERY (= q_stride[l] except for mode 3).
 * The tensor-core builder needs mode 1, 2 or 3 and writes whole 8-element pieces, i.e. zeros into the
 * padding columns; the 16-bit lookup kernel relies on padding columns holding finite values.
 * The blocked layouts are 16-bit layouts: bf16 or fp16 pyramids, not fp32 ones.
 * Every entry point that takes an ofb_pyramid checks it in one place (ofb::check_pyramid, csrc/common.cuh) and
 * returns OFB_EINVAL when levels is outside 1..OFB_MAX_LEVELS, dtype or layout is not one of the values below, a
 * level has a null base, a non-positive size or row_pitch < lvl_w, or a query-minor level has q_stride != 32; each
 * then adds only its own requirements.  ofb_corr_lookup and ofb_corr_lookup_coords_backward pick their reader in one
 * place too (ofb::lookup_reader), so they accept the same pyramids.
 * ------------------------------------------------------------------------------------- */
#define OFB_LAYOUT_ROWS 0
#define OFB_LAYOUT_BLOCK8X4 1
#define OFB_LAYOUT_QMINOR8X4 2

typedef struct ofb_pyramid {
    void* base[OFB_MAX_LEVELS];
    int64_t q_stride[OFB_MAX_LEVELS];
    int32_t row_pitch[OFB_MAX_LEVELS];
    int32_t lvl_h[OFB_MAX_LEVELS];
    int32_t lvl_w[OFB_MAX_LEVELS];
    int32_t levels;
    int32_t dtype;  /* OFB_DTYPE_F32, OFB_DTYPE_BF16 or OFB_DTYPE_F16 */
    int32_t layout; /* OFB_LAYOUT_ROWS, OFB_LAYOUT_BLOCK8X4 or OFB_LAYOUT_QMINOR8X4 (blocked layouts: 16-bit only) */
    int32_t reserved;
} ofb_pyramid;

int ofb_pyramid_layout(int h, int w, int levels, int mode, ofb_pyramid* pyr_host, int64_t elems_host[OFB_MAX_LEVELS]);

/* ---------------------------------------------------------------------------------------
 * K2  all-pairs correlation pyramid.  Replaces CorrBlock.corr + CorrBlock.__init__
 * (methods/raft/model/corr.py:38-54,79-87): corr[b,p,q] = sum_c f1[b,c,p] f2[b,c,q] / sqrt(C),
 * levels 1.. = 2x2 average pooling over the target (q) image, complete blocks only.
 *
 * Step 1, ofb_corr_prep_bf16: fmap (B,C,h,w) fp32 NCHW -> K-major bf16 operand
 *         (B, (h/pool)*(w/pool), C), multiplied by `scale` and, for pool = 2, 4, 8, averaged over complete
 *         pool x pool blocks (cast + transpose in one pass; replaces the .view/.transpose of corr.py:82-85).
 *         The caller preps fmap1 with scale = 1/sqrt(C) (corr.py:87) and fmap2 twice: pool = 1 and,
 *         for pyramids with more than 2 levels, pool = 4.
 * Step 2, ofb_corr_pyramid_bf16: tcgen05/TMEM GEMM tiles fed by TMA, bf16 x bf16 -> fp32
 *         accumulate; every run writes a level and its 2x2 mean from the same accumulators:
 *         levels 0,1 from f2_km, levels 2,3 from f2q_km (avg_pool2d is linear, corr.py:52-54).
 *         f1_km, f2_km: (B, h*w, C) bf16; f2q_km: (B, (h/4)*(w/4), C) bf16 or NULL when
 *         pyr->levels <= 2 (C multiple of 64, <= 256).  `scale` is applied to the accumulators
 *         (pass 1.0f when it was folded into fmap1).
 *         pyr: layout from ofb_pyramid_layout(padded = 1), dtype BF16.
 *         cta_group: 0 = auto, 1 = one CTA per tile, 2 = CTA pair (cta_group::2), 3 = clusters of two independent
 *         cta_group::1 CTAs with the fmap2 operand ring TMA-multicast into both (query-minor layout only).
 * ofb_corr_pyramid_simt_f32: plain CUDA-core builder (fp32 in, fp32, bf16 or fp16 out) used by tests as an
 *         on-device cross-check and for shapes the tensor-core kernel rejects.  Each pooled level is computed from the
 *         stored level above it, in fp32, and rounded to the pyramid dtype.
 * ------------------------------------------------------------------------------------- */
int ofb_corr_prep_bf16(const float* fmap_nchw, void* out_km_bf16, int B, int C, int h, int w, int pool,
                       float scale, void* stream);
/* The same pass reading the feature map in its own precision: in_dtype OFB_DTYPE_F32, OFB_DTYPE_BF16 or
 * OFB_DTYPE_F16.  The reference's shipped configs run `precision: 16` (methods/raft/config/train/default.yaml:20) and
 * raft.py:110-111 answers with fmap.float() -- a full extra pass and twice the bytes for maps whose values are half
 * precision anyway; here the half-precision map is the kernel's input (element -> fp32 -> * scale -> bf16). */
int ofb_corr_prep_from(const void* fmap_nchw, int in_dtype, void* out_km_bf16, int B, int C, int h, int w, int pool,
                       float scale, void* stream);
/* The same pass with the operand type chosen: out_dtype OFB_DTYPE_BF16 (= ofb_corr_prep_from) or OFB_DTYPE_F16, the
 * operands of ofb_corr_pyramid_f16 (element -> fp32 -> * scale -> round to nearest even).  An fp16 map prepped to fp16
 * with pool = 1 and scale = 1 is an exact transpose. */
int ofb_corr_prep_to(const void* fmap_nchw, int in_dtype, void* out_km, int out_dtype, int B, int C, int h, int w,
                     int pool, float scale, void* stream);
int ofb_corr_pyramid_bf16(const void* f1_km, const void* f2_km, const void* f2q_km, const ofb_pyramid* pyr_host,
                          int B, int C, int h, int w, float scale, int cta_group, void* stream);
/* ofb_corr_pyramid_bf16 in fp16: the precision the reference stores its pyramid in under `precision: 16`
 * (methods/raft/config/train/default.yaml:20): autocast runs the torch.matmul of corr.py:85 on fp16 operands, and
 * avg_pool2d keeps fp16 (corr.py:52-54).  f1_km, f2_km, f2q_km: fp16 K-major operands (ofb_corr_prep_to, out_dtype
 * F16); pyr->dtype must be OFB_DTYPE_F16; everything else as for the bf16 builder.  Prep fmap1 with scale = 1 and pass
 * scale = 1/sqrt(C) here: it is applied to the fp32 accumulators, the reference's order (an fp16 GEMM of the rounded
 * maps, then the scale, corr.py:85-87), and keeps fmap1/sqrt(C) out of fp16 subnormals.  Scaled correlations beyond
 * +-65504 become inf, as in the reference under autocast. */
int ofb_corr_pyramid_f16(const void* f1_km, const void* f2_km, const void* f2q_km, const ofb_pyramid* pyr_host,
                         int B, int C, int h, int w, float scale, int cta_group, void* stream);
/* On-demand correlation lookup (SURVEY.md section 8f row 4): CorrBlock.__call__ (corr.py:56-77) WITHOUT the materialised
 * volume of corr.py:45-54.  avg_pool2d is linear, so level l of the pyramid is f1^T . avgpool_l(f2) / sqrt(C); the kernel
 * evaluates those dot products only at the positions each query's window touches and samples them with the same bit-exact
 * coordinate sequence as ofb_corr_lookup.
 *   f1_km            (B, h*w, C) bf16 K-major, already multiplied by 1/sqrt(C)      (ofb_corr_prep_from, pool 1)
 *   f2_km_levels[l]  (B, (h>>l)*(w>>l), C) bf16 K-major, fmap2 averaged over complete 2^l x 2^l blocks (pool 1, 2, 4, 8)
 *   coords (B,2,h,w) fp32 -> out (B, levels*(2r+1)^2, h, w) fp32 (ofb_corr_lookup_ondemand_to: fp16 / bf16).
 *   C in {64, 128, 256}.
 * Memory: the operand maps (22 MB per 1088x1920 pair) instead of the 2.83 GB pyramid; it is slower than build + lookup
 * (DESIGN.md section 4) -- a capacity feature. */
int ofb_corr_lookup_ondemand(const void* f1_km, const void* const* f2_km_levels_host, const float* coords, float* out,
                             int B, int C, int h, int w, int levels, int radius, void* stream);
/* The same lookup with the output's dtype chosen, as ofb_corr_lookup_to: out_dtype OFB_DTYPE_F32 (= ofb_corr_lookup_ondemand),
 * F16 or BF16; anything else is OFB_EINVAL. */
int ofb_corr_lookup_ondemand_to(const void* f1_km, const void* const* f2_km_levels_host, const float* coords, void* out,
                                int out_dtype, int B, int C, int h, int w, int levels, int radius, void* stream);

/* Diagnostics build of the same kernel: additionally fills prof_dev[2][148][16] (device, uint64; one
 * slot per GEMM run) with per-CTA cycle counters -- [0] TMA warp waiting for a free fmap2 stage,
 * [1] for a free fmap1 block, [2] MMA warp waiting for fmap1, [3] for a drained TMEM accumulator,
 * [4] for fmap2 data, [5] epilogue waiting for a finished accumulator, [7] tiles done, [8] kernel
 * cycles.  Used by tools/k2_profile.py, never by the product path. */
int ofb_corr_pyramid_bf16_profile(const void* f1_km, const void* f2_km, const void* f2q_km,
                                  const ofb_pyramid* pyr_host, int B, int C, int h, int w, float scale,
                                  int cta_group, uint64_t* prof_dev, void* stream);
int ofb_corr_pyramid_simt_f32(const float* fmap1, const float* fmap2, const ofb_pyramid* pyr_host,
                              int B, int C, int h, int w, float scale, void* stream);

/* ---------------------------------------------------------------------------------------
 * K3  pyramid lookup.  Replaces CorrBlock.__call__ + bilinear_sampler
 * (methods/raft/model/corr.py:56-77, methods/raft/model/utils.py:64-80): for every query,
 * level and window cell (i,j): bilinear sample (zeros outside, align_corners=True after the
 * reference's normalise/un-normalise round trip) of the query's level slice at
 * (x/2^l + i - r, y/2^l + j - r); out channel = l*(2r+1)^2 + i*(2r+1) + j.
 *   coords (B,2,h,w) fp32 (ch0 = x, ch1 = y);  out (B, L*(2r+1)^2, h, w) fp32 (ofb_corr_lookup_to: fp16 / bf16)
 *   idx_or_null   (B*h*w, L, 2, 2r+1) int32 floor indices (x taps then y taps)
 *   valid_or_null (B*h*w, L, (2r+1)^2) u8   utils.py:77 predicate per sample
 * pyr: dtype F32, BF16 or F16.  Floor indices and validity masks do not depend on the dtype.  16-bit pyramids with
 * radius 3 or 4 take the register-tile kernel, whose 3-tap filter multiplies one in-window column by an exact zero
 * weight the reference's 2-tap form never reads: an inf stored in that column (an fp16 correlation beyond +-65504)
 * gives NaN where the reference gives a finite value.
 * ------------------------------------------------------------------------------------- */
int ofb_corr_lookup(const ofb_pyramid* pyr_host, const float* coords, float* out,
                    int32_t* idx_or_null, uint8_t* valid_or_null, int B, int h, int w, int radius,
                    void* stream);
/* ofb_corr_lookup with the output's dtype chosen: out_dtype OFB_DTYPE_F32 (= ofb_corr_lookup), F16 or BF16; anything
 * else is OFB_EINVAL.  Each sample is accumulated in fp32 exactly as for an fp32 output and rounded once to nearest
 * even: the same bits as the fp32 output cast to that dtype (fp16: beyond +-65504 is inf).  Under the reference's
 * `precision: 16` the lookup's only consumer, BasicMotionEncoder.convc1 (methods/raft/model/update.py:114), receives
 * the output autocast to half precision; writing it in that precision saves the cast and half the output bytes.
 * Indices and masks are unchanged. */
int ofb_corr_lookup_to(const ofb_pyramid* pyr_host, const float* coords, void* out, int out_dtype,
                       int32_t* idx_or_null, uint8_t* valid_or_null, int B, int h, int w, int radius, void* stream);

/* Backward of ofb_corr_lookup with respect to the pyramid (autograd through corr.py:56-77 /
 * utils.py:64-80; the coordinates get no gradient -- RAFT detaches them, raft.py:127).
 * d_pyr: fp32, OFB_LAYOUT_ROWS (ofb_pyramid_layout mode 0 or 1), ACCUMULATED into -- zero it before the
 * first of the refinement iterations, then call once per lookup.  d_out (B, L*(2r+1)^2, h, w). */
int ofb_corr_lookup_backward_f32(const ofb_pyramid* d_pyr, const float* coords, const float* d_out,
                                 int B, int h, int w, int radius, void* stream);
/* The same backward reading d_out in d_out_dtype OFB_DTYPE_F32 (= ofb_corr_lookup_backward_f32), F16 or BF16 (the
 * gradient of an ofb_corr_lookup_to output); anything else is OFB_EINVAL.  Each element is widened exactly to fp32;
 * the arithmetic, its order and the fp32 gradient pyramid are those of the fp32 form. */
int ofb_corr_lookup_backward(const ofb_pyramid* d_pyr, const float* coords, const void* d_out, int d_out_dtype,
                             int B, int h, int w, int radius, void* stream);

/* Backward of ofb_corr_lookup with respect to the coordinates: what autograd computes for coords through
 * CorrBlock.__call__ (methods/raft/model/corr.py:56-77) and bilinear_sampler = grid_sample(align_corners=True, zeros
 * padding) (methods/raft/model/utils.py:64-80), ATen's d grid with the normalise / un-normalise chain factors applied
 * as exactly 1.  pyr: the STORED pyramid the forward read (exactly the pyramids ofb_corr_lookup accepts, same argument
 * checks); d_out (B, L*(2r+1)^2, h, w) fp32; d_coords (B,2,h,w) fp32 is OVERWRITTEN.  Taps on the floors and weights of
 * the forward (integer coordinates: the one-sided derivative the reference's fp32 floor picks).  Taps outside the
 * image read 0; a level with a tap outside the floor guard, a non-finite or far coordinate, or a width or height of 1,
 * contributes 0 (ATen: NaN for NaN coordinates).  Row padding is never read into the result.  Deterministic: the same
 * bits on every run. */
int ofb_corr_lookup_coords_backward(const ofb_pyramid* pyr, const float* coords, const float* d_out, float* d_coords,
                                    int B, int h, int w, int radius, void* stream);
/* The same backward reading d_out in d_out_dtype OFB_DTYPE_F32 (= ofb_corr_lookup_coords_backward), F16 or BF16,
 * widened exactly to fp32 on load; anything else is OFB_EINVAL.  d_coords stays fp32. */
int ofb_corr_lookup_coords_backward_from(const ofb_pyramid* pyr, const float* coords, const void* d_out,
                                         int d_out_dtype, float* d_coords, int B, int h, int w, int radius,
                                         void* stream);

/* The two GEMMs behind d CorrBlock / d fmap (autograd through corr.py:45-54,79-87), on the tensor cores:
 *   D[b] (M x N, fp32, row pitch ldd) = alpha * A[b] (M x K) . B[b]^T (N x K)  (+ D[b] when accumulate != 0)
 * A, B bf16, K-major (row pitches lda, ldb and batch strides in elements, multiples of 8); N a multiple of 32,
 * <= 256; all bases 16-byte aligned.  With dP_l the fp32 gradient of pyramid level l:
 *   d fmap1^T = sum_l dP_l . pool_l(fmap2)        A = bf16(dP_l) (queries x targets),   B = pool_l(fmap2) (C x targets)
 *   d pool_l(fmap2)^T = dP_l^T . fmap1^T          A = bf16(dP_l)^T (targets x queries), B = fmap1 (C x queries)
 * ofb_cast_bf16 produces both A operands from the fp32 level in one pass: a bf16 copy (row pitch
 * pitch_dst >= cols) and / or the bf16 transpose (row pitch pitch_dst_t >= rows); pitches at most the next
 * multiple of 32, padding zero-filled. */
int ofb_gemm_nt_bf16(const void* A, const void* B, float* D, int batch, int M, int N, int K,
                     long long lda, long long ldb, long long ldd, long long strideA, long long strideB,
                     long long strideD, float alpha, int accumulate, void* stream);
int ofb_cast_bf16(const float* src, void* dst_or_null, void* dst_t_or_null, int batch, int rows, int cols,
                  long long pitch_dst, long long pitch_dst_t, void* stream);

/* bilinear_sampler (utils.py:64-80) for arbitrary images: img (N,C,H,W), coords (N,Ho,Wo,2)
 * pixel units -> out (N,C,Ho,Wo) [+ mask (N,Ho,Wo) fp32 0/1]. */
int ofb_bilinear_sampler_f32(const float* img, const float* coords, float* out, float* mask_or_null,
                             int N, int C, int H, int W, int Ho, int Wo, void* stream);

/* ---------------------------------------------------------------------------------------
 * The two passes around the backward GEMMs of CorrBlock (torch-optical-flow_b200/csrc/pool_ops.cu).
 * ofb_pool_cast_bf16: fmap (B,C,h,w) in in_dtype -> (B, C, pitch_k) bf16, element k < (h/pool)*(w/pool) = mean of the
 *   complete pool x pool block k (what the avg_pool2d chain of corr.py:52-54 makes of fmap2), the padding up to
 *   pitch_k zero: the K-long B operand of ofb_gemm_nt_bf16.
 * ofb_pool_adjoint_f32: d_levels[l] (B, (h>>l)*(w>>l), C) fp32 -> d_fmap (B,C,h,w) fp32 (overwritten):
 *   d_fmap[b,c,y,x] = sum_l d_levels[l][b, (y>>l)*(w>>l) + (x>>l), c] / 4^l over the levels whose floor-cropped image
 *   contains the pixel -- the adjoint of that pooling chain, fused with the (B,N,C) -> (B,C,h,w) transpose
 *   (levels = 1: the transpose alone).
 * ------------------------------------------------------------------------------------- */
int ofb_pool_cast_bf16(const void* fmap_nchw, int in_dtype, void* out_bck_bf16, int B, int C, int h, int w, int pool,
                       int pitch_k, void* stream);
int ofb_pool_adjoint_f32(const float* const* d_levels_bnc_host, float* d_fmap_nchw, int B, int C, int h, int w, int levels,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OFB200_H_ */
