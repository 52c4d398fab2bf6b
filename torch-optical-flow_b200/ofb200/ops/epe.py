"""End-point error with the reference's interface (reference optical_flow/metrics/epe.py), computed
by the K4c streaming-reduction kernel.  torchmetrics is not required: the two metric states
(`sum_epe`, `total`) live in one 16-byte device buffer and one all-reduce sums it across ranks -- the
semantics of `dist_reduce_fx="sum"` (reference epe.py:22-23)."""
from typing import Optional

import torch
from torch import Tensor

import ofb200
from ofb200.ops.operator import aligned16


def _prep(pred: Tensor, target: Tensor, dim: int, keep_graph: bool = False):
    """Device, fp32, contiguous, viewed as (L, 2, T, 1): `dim` may be any dimension holding the two flow components
    (reference epe.py:41-61 takes any dim); the dimensions before it fold into L, those after it into T -- a free view
    of a contiguous tensor, (B, 2, H, W) with dim=1 being the usual case.  Detached unless `keep_graph`: then the
    staging, the copy and the view stay on the autograd path and carry gradients back to the inputs' shapes,
    strides and devices."""
    if pred.shape != target.shape:
        raise RuntimeError(f"pred {tuple(pred.shape)} and target {tuple(target.shape)} differ in shape")
    nd = pred.dim()
    if not (-nd <= dim < nd):
        raise IndexError(f"dim {dim} out of range for a {nd}-dimensional flow")
    d = dim % nd
    if pred.shape[d] != 2:
        raise NotImplementedError(f"end-point error kernel expects 2 flow components along dim {dim}, got {pred.shape[d]}")
    for t in (pred, target):
        if t.dtype != torch.float32:
            raise NotImplementedError(f"ofb200 kernels are fp32 only, got {t.dtype}")
    lead = 1
    for n in pred.shape[:d]:
        lead *= int(n)
    trail = 1
    for n in pred.shape[d + 1:]:
        trail *= int(n)
    view = (lead, 2, trail, 1)

    def flat(t: Tensor) -> Tensor:
        t = ofb200.to_device(t)
        return (t if keep_graph else t.detach()).contiguous().view(view)

    return flat(pred), flat(target)


def _prep_valid(valid: Optional[Tensor], b: int, h: int, w: int) -> Optional[Tensor]:
    if valid is None:
        return None
    valid = ofb200.to_device(valid).detach()
    if valid.numel() != b * h * w:
        raise RuntimeError("valid must have B*H*W elements")
    return valid.reshape(b, h, w).to(torch.float32).contiguous()


def _accumulate(acc: Tensor, pred: Tensor, target: Tensor, valid: Optional[Tensor]) -> None:
    b, _, h, w = pred.shape
    valid = _prep_valid(valid, b, h, w)
    with torch.cuda.device(pred.device):
        rc = ofb200.load().ofb_epe_reduce_f32(
            ofb200.ptr(pred), ofb200.ptr(target), ofb200.ptr(valid), ofb200.ptr(acc), b, h, w, ofb200.stream_ptr()
        )
    ofb200.check(rc, "ofb_epe_reduce_f32")


class SumCountMetric:
    """A streaming ratio metric whose two states -- a running sum and a running count -- live in one `double[2]`
    device buffer (exact for counts < 2^53).  Mirrors what torchmetrics does for states declared with
    `dist_reduce_fx="sum"` (reference epe.py:22-23, f1.py:30-31):

      * `update` accumulates into the LOCAL state only (one kernel launch, no synchronisation);
      * `compute` returns sum / count over ALL ranks when `torch.distributed` is initialised: it all-reduces a COPY
        of the state, so the local state is untouched and `compute` / `sync` may be called any number of times;
      * every rank takes part in that collective, also one that never saw an `update` (empty shard): its state is
        created as zeros on the current device;
      * `metric(pred, target, valid)` accumulates and returns the value of THIS batch, like `Metric.forward`."""

    def __init__(self) -> None:
        self._acc: Optional[Tensor] = None   # double[2] on the device: (sum, count)

    def _state(self, device=None) -> Tensor:
        if self._acc is None:
            if device is None:
                device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
            self._acc = torch.zeros(2, dtype=torch.float64, device=device)
        return self._acc

    def _accumulate(self, acc: Tensor, pred: Tensor, target: Tensor, valid: Optional[Tensor]) -> None:
        raise NotImplementedError

    def update(self, pred: Tensor, target: Tensor, valid: Optional[Tensor] = None) -> None:
        pred_d, target_d = _prep(pred, target, self.dim)
        self._accumulate(self._state(pred_d.device), pred_d, target_d, valid)

    def __call__(self, pred: Tensor, target: Tensor, valid: Optional[Tensor] = None) -> Tensor:
        pred_d, target_d = _prep(pred, target, self.dim)
        batch = torch.zeros(2, dtype=torch.float64, device=pred_d.device)
        self._accumulate(batch, pred_d, target_d, valid)
        self._state(pred_d.device).add_(batch)
        return (batch[0] / batch[1]).to(torch.float32)

    def sync(self, group=None) -> Tensor:
        """(sum, count) summed over all ranks -- one 16-byte all-reduce of a copy; the local state is not modified.
        Without an initialised process group this is just a copy of the local state."""
        import torch.distributed as dist

        acc = self._state().clone()
        if dist.is_available() and dist.is_initialized():
            dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
        return acc

    def compute(self, sync: bool = True) -> Tensor:
        """sum / count; over all ranks when `torch.distributed` is initialised (sync=False: this rank only)."""
        import torch.distributed as dist

        if sync and dist.is_available() and dist.is_initialized():
            acc = self.sync()
        elif self._acc is None:
            return torch.tensor(float("nan"))
        else:
            acc = self._acc
        return (acc[0] / acc[1]).to(torch.float32)

    def reset(self) -> None:
        if self._acc is not None:
            self._acc.zero_()


class AverageEndPointError(SumCountMetric):
    """Average End-to-end Point Error (reference epe.py:8-38): streaming mean of ||pred - target||_2.

    Args:
        dim: the dimension along which to compute the end-point-error (it must hold the 2 flow components)
    """

    def __init__(self, dim: int = 1) -> None:
        super().__init__()
        self.dim = dim

    def _accumulate(self, acc: Tensor, pred: Tensor, target: Tensor, valid: Optional[Tensor]) -> None:
        _accumulate(acc, pred, target, valid)

    @property
    def sum_epe(self) -> Tensor:
        return self._acc[0].to(torch.float32) if self._acc is not None else torch.tensor(0.0)

    @property
    def total(self) -> Tensor:
        return self._acc[1].to(torch.int64) if self._acc is not None else torch.tensor(0)


def end_point_error(pred: Tensor, target: Tensor, dim: int = 1, reduce: bool = True) -> Tensor:
    """End-to-end Point Error (reference epe.py:41-61): mean EPE, or the (B, H, W) map with reduce=False.

    Differentiable with respect to `pred` and `target` as the reference's `torch.norm(pred - target, p=2, dim=dim)`
    [`.mean()`] is: d pred = g * ((pred - target) / epe), 0 where epe == 0, and d target = -d pred, with g the map's
    gradient or the mean's divided by the number of pixels (`ofb_epe_backward_f32`)."""
    on_host = not pred.is_cuda
    grad = torch.is_grad_enabled() and (pred.requires_grad or target.requires_grad)
    pred_d, target_d = _prep(pred, target, dim, keep_graph=grad)
    b, _, h, w = pred_d.shape
    map_shape = tuple(pred.shape[:dim % pred.dim()]) + tuple(pred.shape[dim % pred.dim() + 1:])

    def run(p: Tensor, t: Tensor) -> Tensor:
        if reduce:
            acc = torch.zeros(2, dtype=torch.float64, device=p.device)
            _accumulate(acc, p, t, None)
            return (acc[0] / acc[1]).to(torch.float32)
        out = torch.empty((b, h, w), dtype=torch.float32, device=p.device)
        rc = ofb200.load().ofb_epe_map_f32(ofb200.ptr(p), ofb200.ptr(t), ofb200.ptr(out), b, h, w, ofb200.stream_ptr())
        ofb200.check(rc, "ofb_epe_map_f32")
        return out

    def backward(saved, grad_out: Tensor, needs):
        """Both gradients from one kernel launch; the mean's upstream gradient stays on the device."""
        p, t = saved
        with torch.cuda.device(p.device):
            g = grad_out.contiguous() if reduce else aligned16(grad_out)
            d_p = torch.empty_like(p) if needs[0] else None
            d_t = torch.empty_like(t) if needs[1] else None
            rc = ofb200.load().ofb_epe_backward_f32(
                ofb200.ptr(p), ofb200.ptr(t), ofb200.ptr(g), int(reduce), ofb200.ptr(d_p), ofb200.ptr(d_t), b, h, w,
                ofb200.stream_ptr(),
            )
            ofb200.check(rc, "ofb_epe_backward_f32")
        return d_p, d_t

    with torch.cuda.device(pred_d.device):
        out = ofb200.differentiable(run, backward, "end_point_error", pred_d, target_d)
    if not reduce:
        out = out.view(map_shape)
    return out.cpu() if on_host else out
