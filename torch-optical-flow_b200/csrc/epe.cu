// epe.cu -- K4c: end-point-error map, masked EPE sum/count and outlier (F1) count reductions.
//
// Replaces torch.norm(pred-target, p=2, dim=1) + boolean select + sum/numel in
// AverageEndPointError.update (reference optical_flow/metrics/epe.py:25-35,58).
// One streaming pass: float4 loads of both flow components, per-thread fp64 partial sums,
// warp shuffle -> shared -> ONE atomicAdd(double) pair per CTA into acc[2] = {sum, count}.
// The cross-rank reduction (dist_reduce_fx="sum", epe.py:22-23) is a single all-reduce of
// that 16-byte buffer, issued by the host (see optical_flow/metrics/epe.py in this repo).
// HBM roofline: 16 bytes per pixel (+4 with a validity map).
// end_point_error's backward (epe_bwd_kernel) is one more streaming pass of the same shape: 16 bytes read per pixel
// (+4 for a map gradient), 8 written per requested gradient.
#include "common.cuh"

namespace {

constexpr int NT = 256;

__device__ __forceinline__ float epe1(float px, float py, float tx, float ty) {
    const float dx = __fsub_rn(px, tx), dy = __fsub_rn(py, ty);
    return sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
}

// per-pixel contribution: MODE 0 = the end-point error (epe.py:28-35), MODE 1 = 1 if the pixel is an outlier,
// epe > abs_thr and epe / |target| > rel_thr (reference optical_flow/metrics/f1.py:36-41), else 0
template <int MODE>
__device__ __forceinline__ float contribution(float px, float py, float tx, float ty, float abs_thr, float rel_thr) {
    const float e = epe1(px, py, tx, ty);
    if (MODE == 0) return e;
    const float mag = sqrtf(__fadd_rn(__fmul_rn(tx, tx), __fmul_rn(ty, ty)));
    return (e > abs_thr && __fdiv_rn(e, mag) > rel_thr) ? 1.0f : 0.0f;
}

template <int MODE>
__global__ void __launch_bounds__(NT) epe_reduce_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                        const float* __restrict__ valid, double* __restrict__ acc,
                                                        int B, int64_t HW, int vec, float abs_thr, float rel_thr) {
    double sum = 0.0;
    unsigned long long cnt = 0;
    if (vec) {
        const int64_t HW4 = HW >> 2;
        const int64_t total = (int64_t)B * HW4;
        for (int64_t t = (int64_t)blockIdx.x * NT + threadIdx.x; t < total; t += (int64_t)gridDim.x * NT) {
            const int64_t b = t / HW4, q = t - b * HW4;
            const float4 px = __ldg(reinterpret_cast<const float4*>(pred + (b * 2 + 0) * HW) + q);
            const float4 py = __ldg(reinterpret_cast<const float4*>(pred + (b * 2 + 1) * HW) + q);
            const float4 tx = __ldg(reinterpret_cast<const float4*>(target + (b * 2 + 0) * HW) + q);
            const float4 ty = __ldg(reinterpret_cast<const float4*>(target + (b * 2 + 1) * HW) + q);
            float4 v = make_float4(1.f, 1.f, 1.f, 1.f);
            if (valid) v = __ldg(reinterpret_cast<const float4*>(valid + b * HW) + q);
            if (v.x >= 0.5f) { sum += (double)contribution<MODE>(px.x, py.x, tx.x, ty.x, abs_thr, rel_thr); ++cnt; }
            if (v.y >= 0.5f) { sum += (double)contribution<MODE>(px.y, py.y, tx.y, ty.y, abs_thr, rel_thr); ++cnt; }
            if (v.z >= 0.5f) { sum += (double)contribution<MODE>(px.z, py.z, tx.z, ty.z, abs_thr, rel_thr); ++cnt; }
            if (v.w >= 0.5f) { sum += (double)contribution<MODE>(px.w, py.w, tx.w, ty.w, abs_thr, rel_thr); ++cnt; }
        }
    } else {
        const int64_t total = (int64_t)B * HW;
        for (int64_t t = (int64_t)blockIdx.x * NT + threadIdx.x; t < total; t += (int64_t)gridDim.x * NT) {
            const int64_t b = t / HW, q = t - b * HW;
            if (valid && !(__ldg(valid + t) >= 0.5f)) continue;
            sum += (double)contribution<MODE>(__ldg(pred + (b * 2 + 0) * HW + q), __ldg(pred + (b * 2 + 1) * HW + q),
                                              __ldg(target + (b * 2 + 0) * HW + q), __ldg(target + (b * 2 + 1) * HW + q),
                                              abs_thr, rel_thr);
            ++cnt;
        }
    }
    __shared__ double s_sum[NT / 32];
    __shared__ double s_cnt[NT / 32];
    double c = (double)cnt;
    sum = ofb::warp_sum(sum);
    c = ofb::warp_sum(c);
    if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = sum; s_cnt[threadIdx.x >> 5] = c; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0.0, tc = 0.0;
#pragma unroll
        for (int k = 0; k < NT / 32; ++k) { ts += s_sum[k]; tc += s_cnt[k]; }
        atomicAdd(acc + 0, ts);
        atomicAdd(acc + 1, tc);
    }
}

__global__ void __launch_bounds__(NT) epe_map_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                     float* __restrict__ out, int B, int64_t HW) {
    const int64_t total = (int64_t)B * HW;
    for (int64_t t = (int64_t)blockIdx.x * NT + threadIdx.x; t < total; t += (int64_t)gridDim.x * NT) {
        const int64_t b = t / HW, q = t - b * HW;
        out[t] = epe1(__ldg(pred + (b * 2 + 0) * HW + q), __ldg(pred + (b * 2 + 1) * HW + q),
                      __ldg(target + (b * 2 + 0) * HW + q), __ldg(target + (b * 2 + 1) * HW + q));
    }
}

// d end_point_error / d pred of one pixel, ATen's norm backward op for op: g * ((p - t) / n).masked_fill(n == 0, 0)
// with n the forward's own end-point error.  Not (p - t) * (g / n): that rounds differently.
__device__ __forceinline__ float2 epe_grad1(float px, float py, float tx, float ty, float g) {
    const float n = epe1(px, py, tx, ty);
    const float qx = n == 0.0f ? 0.0f : __fdiv_rn(__fsub_rn(px, tx), n);
    const float qy = n == 0.0f ? 0.0f : __fdiv_rn(__fsub_rn(py, ty), n);
    return make_float2(__fmul_rn(g, qx), __fmul_rn(g, qy));
}

// One streaming pass, lane <-> pixel (VEC: 4 consecutive pixels, float4 loads and stores), both gradients written;
// d_target = -d_pred (the subtraction's backward).  d_epe is the (B,H,W) map, or with `scalar` the mean's one
// upstream gradient, divided by B*H*W on the device as ATen's mean backward divides it.
template <bool VEC>
__global__ void __launch_bounds__(NT) epe_bwd_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                     const float* __restrict__ d_epe, int scalar,
                                                     float* __restrict__ d_pred, float* __restrict__ d_target, int B,
                                                     int64_t HW) {
    constexpr int V = VEC ? 4 : 1;
    const int64_t per_b = HW / V;
    const int64_t total = (int64_t)B * per_b;
    const float g0 = scalar ? __fdiv_rn(__ldg(d_epe), (float)((int64_t)B * HW)) : 0.0f;
    for (int64_t t = (int64_t)blockIdx.x * NT + threadIdx.x; t < total; t += (int64_t)gridDim.x * NT) {
        const int64_t b = t / per_b, q = (t - b * per_b) * V;
        const int64_t ox = (b * 2 + 0) * HW + q, oy = (b * 2 + 1) * HW + q;
        float px[V], py[V], tx[V], ty[V], g[V], dx[V], dy[V];
        if constexpr (VEC) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(pred + ox));
            const float4 c = __ldg(reinterpret_cast<const float4*>(pred + oy));
            const float4 e = __ldg(reinterpret_cast<const float4*>(target + ox));
            const float4 f = __ldg(reinterpret_cast<const float4*>(target + oy));
            const float4 h = scalar ? make_float4(g0, g0, g0, g0) : __ldg(reinterpret_cast<const float4*>(d_epe + b * HW + q));
            px[0] = a.x; px[1] = a.y; px[2] = a.z; px[3] = a.w;
            py[0] = c.x; py[1] = c.y; py[2] = c.z; py[3] = c.w;
            tx[0] = e.x; tx[1] = e.y; tx[2] = e.z; tx[3] = e.w;
            ty[0] = f.x; ty[1] = f.y; ty[2] = f.z; ty[3] = f.w;
            g[0] = h.x; g[1] = h.y; g[2] = h.z; g[3] = h.w;
        } else {
            px[0] = __ldg(pred + ox); py[0] = __ldg(pred + oy);
            tx[0] = __ldg(target + ox); ty[0] = __ldg(target + oy);
            g[0] = scalar ? g0 : __ldg(d_epe + t);
        }
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const float2 d = epe_grad1(px[k], py[k], tx[k], ty[k], g[k]);
            dx[k] = d.x; dy[k] = d.y;
        }
        if constexpr (VEC) {
            if (d_pred) {
                *reinterpret_cast<float4*>(d_pred + ox) = make_float4(dx[0], dx[1], dx[2], dx[3]);
                *reinterpret_cast<float4*>(d_pred + oy) = make_float4(dy[0], dy[1], dy[2], dy[3]);
            }
            if (d_target) {
                *reinterpret_cast<float4*>(d_target + ox) = make_float4(-dx[0], -dx[1], -dx[2], -dx[3]);
                *reinterpret_cast<float4*>(d_target + oy) = make_float4(-dy[0], -dy[1], -dy[2], -dy[3]);
            }
        } else {
            if (d_pred) { d_pred[ox] = dx[0]; d_pred[oy] = dy[0]; }
            if (d_target) { d_target[ox] = -dx[0]; d_target[oy] = -dy[0]; }
        }
    }
}


// ---------------------------------------------------------------------------------- sequence loss
// sequence_loss (reference methods/raft/model/raft.py:231-260) in one pass over the ground truth:
//   keep = (valid >= 0.5) & (|gt| < max_flow)
//   loss = sum_i gamma^(n-1-i) * mean(keep * |pred_i - gt|)     (mean over ALL B*2*H*W elements)
//   epe  = |pred_{n-1} - gt|_2 over kept pixels -> fractions below 1 / 3 / 5 px
// The reference makes 4 elementwise passes per prediction plus the metric passes; here the ground truth and
// validity map are read once and every prediction once (8 bytes per pixel per prediction).
constexpr int MAX_PREDS = OFB_MAX_PREDICTIONS;
struct PredList {
    const float* p[MAX_PREDS];
    double w[MAX_PREDS];
};

struct SeqAcc {
    double loss, epe;
    unsigned long long keep, n1, n3, n5;
};

__global__ void __launch_bounds__(NT) sequence_loss_kernel(const __grid_constant__ PredList preds, int n,
                                                           const float* __restrict__ gt, const float* __restrict__ valid,
                                                           double* __restrict__ acc, int B, int64_t HW, int vec,
                                                           float max_flow) {
    SeqAcc a{0.0, 0.0, 0ull, 0ull, 0ull, 0ull};
    const int64_t step = vec ? 4 : 1;
    const int64_t per_b = HW / step;
    const int64_t total = (int64_t)B * per_b;
    for (int64_t t = (int64_t)blockIdx.x * NT + threadIdx.x; t < total; t += (int64_t)gridDim.x * NT) {
        const int64_t b = t / per_b, q = (t - b * per_b) * step;
        const int64_t ox = (b * 2 + 0) * HW + q, oy = (b * 2 + 1) * HW + q, ov = b * HW + q;
        float gx[4], gy[4], m[4];
        if (vec) {
            const float4 x = __ldg(reinterpret_cast<const float4*>(gt + ox)), y = __ldg(reinterpret_cast<const float4*>(gt + oy));
            const float4 v = __ldg(reinterpret_cast<const float4*>(valid + ov));
            gx[0] = x.x; gx[1] = x.y; gx[2] = x.z; gx[3] = x.w;
            gy[0] = y.x; gy[1] = y.y; gy[2] = y.z; gy[3] = y.w;
            m[0] = v.x; m[1] = v.y; m[2] = v.z; m[3] = v.w;
        } else {
            gx[0] = __ldg(gt + ox); gy[0] = __ldg(gt + oy); m[0] = __ldg(valid + ov);
        }
        const int cnt = vec ? 4 : 1;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k >= cnt) break;
            const float mag = sqrtf(__fadd_rn(__fmul_rn(gx[k], gx[k]), __fmul_rn(gy[k], gy[k])));
            m[k] = (m[k] >= 0.5f && mag < max_flow) ? 1.0f : 0.0f;
            a.keep += m[k] != 0.0f;
        }
        for (int i = 0; i < n; ++i) {
            float px[4], py[4];
            if (vec) {
                const float4 x = __ldg(reinterpret_cast<const float4*>(preds.p[i] + ox));
                const float4 y = __ldg(reinterpret_cast<const float4*>(preds.p[i] + oy));
                px[0] = x.x; px[1] = x.y; px[2] = x.z; px[3] = x.w;
                py[0] = y.x; py[1] = y.y; py[2] = y.z; py[3] = y.w;
            } else {
                px[0] = __ldg(preds.p[i] + ox); py[0] = __ldg(preds.p[i] + oy);
            }
            float part = 0.0f;                            // keep * |d|: a NaN under a dropped pixel stays NaN, as there
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k >= cnt) break;
                const float dx = __fsub_rn(px[k], gx[k]), dy = __fsub_rn(py[k], gy[k]);
                part += __fmul_rn(m[k], fabsf(dx)) + __fmul_rn(m[k], fabsf(dy));
                if (i == n - 1 && m[k] != 0.0f) {
                    const float e = sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
                    a.epe += (double)e;
                    a.n1 += e < 1.0f; a.n3 += e < 3.0f; a.n5 += e < 5.0f;
                }
            }
            a.loss += preds.w[i] * (double)part;
        }
    }
    __shared__ double s_red[NT / 32][6];
    double v[6] = {a.loss, a.epe, (double)a.keep, (double)a.n1, (double)a.n3, (double)a.n5};
#pragma unroll
    for (int k = 0; k < 6; ++k) v[k] = ofb::warp_sum(v[k]);
    if ((threadIdx.x & 31) == 0)
        for (int k = 0; k < 6; ++k) s_red[threadIdx.x >> 5][k] = v[k];
    __syncthreads();
    if (threadIdx.x < 6) {
        double tsum = 0.0;
#pragma unroll
        for (int wv = 0; wv < NT / 32; ++wv) tsum += s_red[wv][threadIdx.x];
        atomicAdd(acc + threadIdx.x, tsum);
    }
}

// Backward of sequence_loss: d loss / d pred_i = grad * gamma^(n-1-i) / (B*2*H*W) * keep * sign(pred_i - gt)
// (autograd of raft.py:247-250: abs -> sign, mean -> 1/numel, the mask multiplies).  One elementwise pass that
// reads the ground truth / validity once and writes all n gradients.
struct GradList {
    float* p[MAX_PREDS];
};

__global__ void __launch_bounds__(NT) sequence_loss_bwd_kernel(const __grid_constant__ PredList preds,
                                                               const __grid_constant__ GradList grads, int n,
                                                               const float* __restrict__ gt, const float* __restrict__ valid,
                                                               const float* __restrict__ grad_loss, int B, int64_t HW,
                                                               float max_flow, double inv_numel) {
    const double g0 = (double)__ldg(grad_loss) * inv_numel;
    const int64_t total = (int64_t)B * HW;
    for (int64_t t = (int64_t)blockIdx.x * NT + threadIdx.x; t < total; t += (int64_t)gridDim.x * NT) {
        const int64_t b = t / HW, q = t - b * HW;
        const int64_t ox = (b * 2 + 0) * HW + q, oy = (b * 2 + 1) * HW + q;
        const float gx = __ldg(gt + ox), gy = __ldg(gt + oy);
        const float mag = sqrtf(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)));
        const bool keep = __ldg(valid + t) >= 0.5f && mag < max_flow;
        for (int i = 0; i < n; ++i) {
            if (!grads.p[i]) continue;
            float dx = 0.0f, dy = 0.0f;
            if (keep) {
                const float w = (float)(g0 * preds.w[i]);
                const float ex = __ldg(preds.p[i] + ox) - gx, ey = __ldg(preds.p[i] + oy) - gy;
                dx = ex > 0.0f ? w : (ex < 0.0f ? -w : 0.0f);
                dy = ey > 0.0f ? w : (ey < 0.0f ? -w : 0.0f);
            }
            grads.p[i][ox] = dx;
            grads.p[i][oy] = dy;
        }
    }
}

}  // namespace

namespace {
template <int MODE>
int launch_reduce(const float* pred, const float* target, const float* valid_or_null, double* acc, int B, int H, int W,
                  float abs_thr, float rel_thr, void* stream) {
    if (B == 0 || H == 0 || W == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!pred || !target || !acc || B < 0 || H < 0 || W < 0) return OFB_EINVAL;
    const int64_t HW = (int64_t)H * W;
    if ((int64_t)B * HW == 0) return OFB_OK;
    const uintptr_t al = reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(target) |
                         reinterpret_cast<uintptr_t>(valid_or_null);
    const int vec = (HW % 4 == 0) && ((al & 15) == 0);
    const int64_t work = vec ? (int64_t)B * (HW / 4) : (int64_t)B * HW;
    int64_t blocks = (work + NT - 1) / NT;
    const int cap = ofb_num_sms() * 8;   // few CTAs -> few atomics; 8 x 256 threads fill an SM
    if (blocks > cap) blocks = cap;
    epe_reduce_kernel<MODE><<<(int)blocks, NT, 0, (cudaStream_t)stream>>>(pred, target, valid_or_null, acc, B, HW, vec,
                                                                         abs_thr, rel_thr);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
}  // namespace

OFB_API int ofb_epe_reduce_f32(const float* pred, const float* target, const float* valid_or_null, double* acc, int B,
                               int H, int W, void* stream) {
    return launch_reduce<0>(pred, target, valid_or_null, acc, B, H, W, 0.0f, 0.0f, stream);
}

OFB_API int ofb_outlier_reduce_f32(const float* pred, const float* target, const float* valid_or_null, double* acc, int B,
                                   int H, int W, float abs_threshold, float rel_threshold, void* stream) {
    return launch_reduce<1>(pred, target, valid_or_null, acc, B, H, W, abs_threshold, rel_threshold, stream);
}

OFB_API int ofb_epe_map_f32(const float* pred, const float* target, float* out, int B, int H, int W, void* stream) {
    if (B == 0 || H == 0 || W == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!pred || !target || !out || B < 0 || H < 0 || W < 0) return OFB_EINVAL;
    const int64_t HW = (int64_t)H * W;
    if ((int64_t)B * HW == 0) return OFB_OK;
    int64_t blocks = ((int64_t)B * HW + NT - 1) / NT;
    const int cap = ofb_num_sms() * 32;
    if (blocks > cap) blocks = cap;
    epe_map_kernel<<<(int)blocks, NT, 0, (cudaStream_t)stream>>>(pred, target, out, B, HW);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_epe_backward_f32(const float* pred, const float* target, const float* d_epe, int d_epe_is_scalar,
                                 float* d_pred_or_null, float* d_target_or_null, int B, int H, int W, void* stream) {
    if (B == 0 || H == 0 || W == 0) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!pred || !target || !d_epe || B < 0 || H < 0 || W < 0) return OFB_EINVAL;
    if (!d_pred_or_null && !d_target_or_null) return OFB_OK;
    const int64_t HW = (int64_t)H * W;
    const int scalar = d_epe_is_scalar != 0;
    const uintptr_t al = reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(target) |
                         reinterpret_cast<uintptr_t>(d_pred_or_null) | reinterpret_cast<uintptr_t>(d_target_or_null) |
                         (scalar ? 0 : reinterpret_cast<uintptr_t>(d_epe));
    const bool vec = (HW % 4 == 0) && ((al & 15) == 0);
    const int64_t work = vec ? (int64_t)B * (HW / 4) : (int64_t)B * HW;
    int64_t blocks = (work + NT - 1) / NT;
    const int cap = ofb_num_sms() * 8;   // 8 x 256 threads fill an SM; each thread strides over the rest
    if (blocks > cap) blocks = cap;
    if (vec)
        epe_bwd_kernel<true><<<(int)blocks, NT, 0, (cudaStream_t)stream>>>(pred, target, d_epe, scalar, d_pred_or_null,
                                                                          d_target_or_null, B, HW);
    else
        epe_bwd_kernel<false><<<(int)blocks, NT, 0, (cudaStream_t)stream>>>(pred, target, d_epe, scalar, d_pred_or_null,
                                                                           d_target_or_null, B, HW);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_sequence_loss_f32(const float* const* preds, int n_predictions, const float* flow_gt, const float* valid,
                                  double* acc, int B, int H, int W, double gamma, float max_flow, void* stream) {
    if (n_predictions >= 1 && (B == 0 || H == 0 || W == 0)) return OFB_OK;   // nothing to do: empty tensors have no storage, their pointers may be null
    if (!preds || !flow_gt || !valid || !acc || B < 0 || H < 0 || W < 0 || n_predictions < 1) return OFB_EINVAL;
    if (n_predictions > MAX_PREDS) return OFB_EUNSUPPORTED;
    const int64_t HW = (int64_t)H * W;
    if ((int64_t)B * HW == 0) return OFB_OK;
    PredList pl;
    uintptr_t al = reinterpret_cast<uintptr_t>(flow_gt) | reinterpret_cast<uintptr_t>(valid);
    for (int i = 0; i < MAX_PREDS; ++i) { pl.p[i] = nullptr; pl.w[i] = 0.0; }
    double wgt = 1.0;                                     // gamma ** (n - 1 - i), as the reference's Python float
    for (int i = n_predictions - 1; i >= 0; --i) {
        if (!preds[i]) return OFB_EINVAL;
        pl.p[i] = preds[i];
        pl.w[i] = wgt;
        wgt *= gamma;
        al |= reinterpret_cast<uintptr_t>(preds[i]);
    }
    const int vec = (HW % 4 == 0) && ((al & 15) == 0);
    const int64_t work = vec ? (int64_t)B * (HW / 4) : (int64_t)B * HW;
    int64_t blocks = (work + NT - 1) / NT;
    const int cap = ofb_num_sms() * 8;
    if (blocks > cap) blocks = cap;
    sequence_loss_kernel<<<(int)blocks, NT, 0, (cudaStream_t)stream>>>(pl, n_predictions, flow_gt, valid, acc, B, HW, vec,
                                                                      max_flow);
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}

OFB_API int ofb_sequence_loss_backward_f32(const float* const* preds, float* const* d_preds, int n_predictions,
                                           const float* flow_gt, const float* valid, const float* grad_loss, int B, int H,
                                           int W, double gamma, float max_flow, void* stream) {
    if (!preds || !d_preds || !flow_gt || !valid || !grad_loss || B < 0 || H < 0 || W < 0 || n_predictions < 1)
        return OFB_EINVAL;
    if (n_predictions > MAX_PREDS) return OFB_EUNSUPPORTED;
    const int64_t HW = (int64_t)H * W;
    if ((int64_t)B * HW == 0) return OFB_OK;
    PredList pl;
    GradList gl;
    for (int i = 0; i < MAX_PREDS; ++i) { pl.p[i] = nullptr; pl.w[i] = 0.0; gl.p[i] = nullptr; }
    double wgt = 1.0;
    for (int i = n_predictions - 1; i >= 0; --i) {
        if (!preds[i]) return OFB_EINVAL;
        pl.p[i] = preds[i];
        pl.w[i] = wgt;
        gl.p[i] = d_preds[i];
        wgt *= gamma;
    }
    int64_t blocks = ((int64_t)B * HW + NT - 1) / NT;
    const int cap = ofb_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    sequence_loss_bwd_kernel<<<(int)blocks, NT, 0, (cudaStream_t)stream>>>(
        pl, gl, n_predictions, flow_gt, valid, grad_loss, B, HW, max_flow, 1.0 / ((double)B * 2.0 * (double)HW));
    OFB_LAUNCH_CHECK();
    return OFB_OK;
}
