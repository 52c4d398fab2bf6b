"""RAFT's convex flow upsampling (reference methods/raft/model/raft.py:73-85) on the K4b kernel and the forward
value of `sequence_loss` (raft.py:231-260) as one fused streaming reduction.

Only the hot-path static methods / functions of the reference's `raft` module are provided; the network itself
(encoders, GRU, training loop) is out of scope and keeps running from the reference."""
import ctypes
from typing import Dict, Sequence, Tuple

import torch
from torch import Tensor

import ofb200
from ofb200.ops.operator import _check_f32, _run, aligned16
from ofb200.ops.sampling import coords_grid


_MASK_DTYPES = {torch.float32: ofb200.DTYPE_F32, torch.bfloat16: ofb200.DTYPE_BF16, torch.float16: ofb200.DTYPE_F16}


def upsample_flow(flow: Tensor, mask: Tensor) -> Tensor:
    """Upsample flow field [H/8, W/8, 2] -> [H, W, 2] using convex combination (reference raft.py:73-85).

    flow (N, 2, h, w) fp32, mask (N, 576, h, w) -> (N, 2, 8h, 8w) fp32.  The mask may be fp32, bf16 or fp16 (the mask
    head's output under `precision: 16`) and is read as it is, in both directions: the backward keeps the caller's mask
    and writes its gradient in the mask's dtype, the bits of the fp32 gradient cast to it (what autocast's cast around
    the reference's fp32 softmax, raft.py:78, hands the mask head)."""
    n, _, h, w = flow.shape
    if flow.shape[1] != 2 or tuple(mask.shape) != (n, 576, h, w):
        raise RuntimeError(f"upsample_flow: expected flow (N,2,h,w) and mask (N,576,h,w), got "
                           f"{tuple(flow.shape)} and {tuple(mask.shape)}")
    _check_f32(flow)
    if mask.dtype not in _MASK_DTYPES:
        raise NotImplementedError(f"upsample_flow: mask must be fp32, bf16 or fp16, got {mask.dtype}")

    def run(flow_d: Tensor, mask_d: Tensor):
        flow_d, mask_d = flow_d.contiguous(), aligned16(mask_d)
        out = torch.empty((n, 2, 8 * h, 8 * w), dtype=torch.float32, device=flow_d.device)
        rc = ofb200.load().ofb_convex_upsample(
            ofb200.ptr(flow_d), ofb200.ptr(mask_d), _MASK_DTYPES[mask_d.dtype], ofb200.ptr(out), n, h, w, ofb200.stream_ptr()
        )
        ofb200.check(rc, "ofb_convex_upsample")
        return out

    def backward(saved, grad_out: Tensor, needs):
        """d up / d flow and d up / d mask: autograd through softmax, unfold and the weighted sum (raft.py:77-85)."""
        flow_d, mask_d = saved
        with torch.cuda.device(flow_d.device):
            flow_c, mask_c, grad_c = flow_d.contiguous(), aligned16(mask_d), aligned16(grad_out)
            d_flow = torch.zeros((n, 2, h, w), dtype=torch.float32, device=flow_c.device) if needs[0] else None
            d_mask = torch.empty((n, 576, h, w), dtype=mask_c.dtype, device=flow_c.device) if needs[1] else None
            rc = ofb200.load().ofb_convex_upsample_backward(
                ofb200.ptr(flow_c), ofb200.ptr(mask_c), _MASK_DTYPES[mask_c.dtype], ofb200.ptr(grad_c), ofb200.ptr(d_flow),
                ofb200.ptr(d_mask), n, h, w, ofb200.stream_ptr(),
            )
            ofb200.check(rc, "ofb_convex_upsample_backward")
        return d_flow, d_mask

    return _run(run, "upsample_flow", flow, mask, bwd=backward)


def sequence_loss(
    flow_preds: Sequence[Tensor],
    flow_gt: Tensor,
    valid: Tensor,
    gamma: float = 0.8,
    max_flow: float = 400.0,
) -> Tuple[Tensor, Dict[str, float]]:
    """Loss function defined over sequence of flow predictions (reference raft.py:231-260), forward value.

    flow_preds: n tensors (B, 2, H, W); flow_gt (B, 2, H, W); valid (B, H, W).  Returns the gamma-weighted L1 loss
    (0-dim fp32 tensor on the inputs' device) and the reference's {"1px", "3px", "5px"} metrics of the last
    prediction.  The ground truth and validity map are read once and every prediction once; the reference makes
    four elementwise passes per prediction.  Differentiable with respect to the predictions."""
    n = len(flow_preds)
    if n < 1:
        raise ValueError("sequence_loss: need at least one flow prediction")
    if n > ofb200.MAX_PREDICTIONS:
        raise NotImplementedError(f"sequence_loss: at most {ofb200.MAX_PREDICTIONS} predictions, got {n}")
    b, two, h, w = flow_gt.shape
    if two != 2 or tuple(valid.shape) != (b, h, w) or any(tuple(p.shape) != (b, 2, h, w) for p in flow_preds):
        raise RuntimeError(f"sequence_loss: expected predictions / flow_gt (B,2,H,W) and valid (B,H,W), got "
                           f"{[tuple(p.shape) for p in flow_preds]}, {tuple(flow_gt.shape)}, {tuple(valid.shape)}")
    _check_f32(flow_gt, *flow_preds)

    numel = float(b * 2 * h * w)

    def run(gt_d: Tensor, valid_d: Tensor, *preds_d: Tensor):
        gt_d, valid_d = gt_d.contiguous(), valid_d.float().contiguous()
        preds_d = [p.contiguous() for p in preds_d]
        acc = torch.zeros(6, dtype=torch.float64, device=gt_d.device)
        ptrs = (ctypes.c_void_p * n)(*[p.data_ptr() for p in preds_d])
        rc = ofb200.load().ofb_sequence_loss_f32(ptrs, n, ofb200.ptr(gt_d), ofb200.ptr(valid_d), ofb200.ptr(acc),
                                                 b, h, w, float(gamma), float(max_flow), ofb200.stream_ptr())
        ofb200.check(rc, "ofb_sequence_loss_f32")
        return (acc[0] / numel).to(torch.float32), acc

    def backward(saved, grad_loss: Tensor, needs):
        """d loss / d pred_i = grad * gamma^(n-1-i) / numel * keep * sign(pred_i - gt) (autograd of raft.py:247-250);
        the ground truth and the validity map get no gradient."""
        gt_d, valid_d, *preds_d = saved
        with torch.cuda.device(gt_d.device):
            gt_c, valid_c = gt_d.contiguous(), valid_d.float().contiguous()
            preds_c = [p.contiguous() for p in preds_d]
            grads = [torch.empty_like(p) if needs[2 + i] else None for i, p in enumerate(preds_c)]
            ptrs = (ctypes.c_void_p * n)(*[p.data_ptr() for p in preds_c])
            gptrs = (ctypes.c_void_p * n)(*[(g.data_ptr() if g is not None else None) for g in grads])
            gl = grad_loss.to(torch.float32).contiguous()
            rc = ofb200.load().ofb_sequence_loss_backward_f32(ptrs, gptrs, n, ofb200.ptr(gt_c), ofb200.ptr(valid_c),
                                                              ofb200.ptr(gl), b, h, w, float(gamma), float(max_flow),
                                                              ofb200.stream_ptr())
            ofb200.check(rc, "ofb_sequence_loss_backward_f32")
        return (None, None, *grads)

    loss, acc = _run(run, "sequence_loss", flow_gt, valid, *flow_preds, bwd=backward)
    host = acc.detach().cpu()                               # one 48-byte read-back, as the reference's .item() calls
    kept = float(host[2])
    # an empty selection is mean() of an empty tensor in the reference: NaN
    metrics = {name: (float(host[k]) / kept if kept > 0 else float("nan")) for name, k in (("1px", 3), ("3px", 4), ("5px", 5))}
    return loss, metrics


class RAFT:
    """Namespace for the static hot-path methods of the reference's RAFT LightningModule."""

    upsample_flow = staticmethod(upsample_flow)

    @staticmethod
    def initialize_flow(img: Tensor) -> Tuple[Tensor, Tensor]:
        """flow = coords1 - coords0 on the 1/8 grid (reference raft.py:64-71)."""
        n, c, h, w = img.shape
        coords0 = coords_grid(n, h // 8, w // 8).to(img.device)
        coords1 = coords_grid(n, h // 8, w // 8).to(img.device)
        return coords0, coords1
