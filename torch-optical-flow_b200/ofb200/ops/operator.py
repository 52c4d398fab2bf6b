"""Flow operators with the reference's names, arguments and assertion behaviour
(reference optical_flow/operator/operator.py), computed by the K1 / K4a kernels of libofb200.

Tensors may live on the host or on the GPU: host tensors are staged through the device and the
result is returned on the host (the reference's tests/operator build CPU tensors).  fp32 only, except `scale` /
`normalize` / `denormalize` (dtype-preserving) and `warp` (fp32, fp16 or bf16 frames and flows).
"""
import warnings
from typing import Optional, Tuple, Union

import torch
from torch import Tensor

import ofb200


def aligned16(t: Tensor) -> Tensor:
    """`t.contiguous()`, re-allocated when its first byte is not 16-byte aligned: a contiguous VIEW with a storage
    offset (a sliced upstream gradient, say) is legal autograd input, and the vectorised kernels need the alignment."""
    t = t.contiguous()
    return t.clone() if t.data_ptr() % 16 else t


def _check_f32(*tensors: Tensor) -> None:
    for t in tensors:
        if t.dtype != torch.float32:
            raise NotImplementedError(f"ofb200 kernels are fp32 only, got {t.dtype}")


_WARP_DTYPES = {torch.float32: ofb200.DTYPE_F32, torch.float16: ofb200.DTYPE_F16, torch.bfloat16: ofb200.DTYPE_BF16}


def alert_not_deterministic(caller: str) -> None:
    """What ATen's `alertNotDeterministic` does for its own order-dependent kernels: under
    `torch.use_deterministic_algorithms(True)` raise RuntimeError, with `warn_only=True` warn instead."""
    if not torch.are_deterministic_algorithms_enabled():
        return
    if torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(f"{caller} does not have a deterministic implementation, but you set "
                      "'torch.use_deterministic_algorithms(True, warn_only=True)'.", stacklevel=3)
        return
    raise RuntimeError(f"{caller} does not have a deterministic implementation, but you set "
                       "'torch.use_deterministic_algorithms(True)'. You can turn off determinism just for this "
                       "operation, or you can use the 'warn_only=True' option, if that's acceptable for your "
                       "application.")


def _run(fn, name: str, *tensors: Tensor, bwd=None) -> Tensor:
    """Stage inputs on the device, run the kernel (forward-only unless a backward kernel is given), return on
    the inputs' device."""
    on_host = not tensors[0].is_cuda
    dev = [ofb200.to_device(t) for t in tensors]
    with torch.cuda.device(dev[0].device):
        out = ofb200.differentiable(fn, bwd, name, *dev) if bwd else ofb200.forward_only(fn, name, *dev)
    if on_host:
        out = tuple(o.cpu() for o in out) if isinstance(out, tuple) else out.cpu()
    return out


def warp(
    frame: Tensor,
    flow: Tensor,
    mode: str = "bilinear",
    padding_mode: str = "border",
    align_corners: bool = False,
    return_mask: bool = False,
    variant: int = 0,
    pixel_flow: bool = False,
) -> Union[Tensor, Tuple[Tensor, Tensor]]:
    """Inverse warping with optical flow (reference operator.py:8-33).

    Args:
        frame: the image tensor of shape (B, C, H, W); contiguous or channels_last
        flow: the optical flow tensor of shape (B, 2, H, W), normalised units (see :func:`normalize`)
        mode: "bilinear" or "nearest" ("bicubic" raises NotImplementedError)
        padding_mode: "zeros", "border" or "reflection"
        align_corners: as :func:`torch.nn.functional.grid_sample`
        return_mask: extension (default off): also return the (B, H, W) bool validity mask -- the
            predicate of ``bilinear_sampler(mask=True)`` (reference methods/raft/model/utils.py:76-78)
            evaluated on the warp grid: True where the source position lies strictly inside the frame
        variant: kernel selection, 0 = auto, 1 = direct gather, 2 = cp.async-staged, 3 = row kernel, 4 = TMA-staged
        pixel_flow: extension (default off): `flow` is in pixel units and :func:`normalize` is fused into
            the kernel -- ``warp(f, flow, pixel_flow=True)`` equals ``warp(f, normalize(flow))`` bit for bit for an
            fp32 flow, and ``warp(f.float(), normalize(flow.float()))`` for a half one.  It does not equal
            ``warp(f, normalize(flow))`` for a half flow: `normalize` keeps the flow's dtype and rounds the product
            to it, the fused multiply is one fp32 rounding.

    The frame and the flow may each be fp32, fp16 or bf16.  Half-precision inputs are read directly, each element
    widened exactly, so the result is always fp32 and bit for bit ``warp(frame.float(), flow.float(), ...)``: what
    the reference returns under CUDA autocast, where grid_sample runs in fp32.  Outside autocast ATen raises for a
    half frame; this computes the same fp32 result instead.  The gradients arrive in the inputs' dtypes, the fp32
    gradients rounded once (what autocast's cast, or type promotion's, hands them).

    Returns:
        The warped image (B, C, H, W), contiguous fp32; with ``return_mask`` a tuple (warped, mask).
    """
    if mode not in ofb200.MODE:
        if mode == "bicubic":
            raise NotImplementedError("warp: mode='bicubic' has no B200 kernel")
        raise ValueError(f"warp: unknown mode {mode!r}")
    if padding_mode not in ofb200.PAD:
        raise ValueError(f"warp: unknown padding_mode {padding_mode!r}")
    if frame.dim() != 4 or flow.dim() != 4:
        raise ValueError("warp: frame must be (B, C, H, W) and flow (B, 2, H, W)")
    b, c, h, w = frame.shape
    if tuple(flow.shape) != (b, 2, h, w):
        raise RuntimeError(f"warp: flow shape {tuple(flow.shape)} does not match frame {tuple(frame.shape)}")
    for t in (frame, flow):
        if t.dtype not in _WARP_DTYPES:
            raise NotImplementedError(f"ofb200 warp kernels are fp32, fp16 or bf16 only, got {t.dtype}")
    mul_x, mul_y = (2.0 / max(w - 1, 1), 2.0 / max(h - 1, 1)) if pixel_flow else (1.0, 1.0)

    def run(frame_d: Tensor, flow_d: Tensor):
        lib = ofb200.load()
        channels_last = (
            c > 1 and not frame_d.is_contiguous() and frame_d.is_contiguous(memory_format=torch.channels_last)
        )
        if not channels_last:
            frame_d = frame_d.contiguous()
        flow_d = flow_d.contiguous()
        out = torch.empty((b, c, h, w), dtype=torch.float32, device=frame_d.device)
        mask = torch.empty((b, h, w), dtype=torch.uint8, device=frame_d.device) if return_mask else None
        rc = lib.ofb_warp(
            ofb200.ptr(frame_d), _WARP_DTYPES[frame_d.dtype], ofb200.ptr(flow_d), _WARP_DTYPES[flow_d.dtype],
            ofb200.ptr(out), ofb200.ptr(mask), b, c, h, w, ofb200.MODE[mode], ofb200.PAD[padding_mode],
            int(bool(align_corners)), int(channels_last), int(variant), mul_x, mul_y, ofb200.stream_ptr(),
        )
        ofb200.check(rc, "ofb_warp")
        return (out, mask.view(torch.bool)) if return_mask else out     # the kernel writes 0 / 1 bytes: zero-copy view

    def backward(saved, grad_out: Tensor, needs):
        """d warp / d frame (scatter-add of the bilinear weights) and d warp / d flow, as F.grid_sample's backward
        through warp_grid (reference operator.py:28-33,56).  d_frame is accumulated in fp32 and rounded once to the
        frame's dtype; d_flow is written in the flow's dtype.  d_frame's atomic adds run in no fixed order, so its
        bits may differ between runs: under `torch.use_deterministic_algorithms(True)` a frame gradient raises, as
        F.grid_sample's backward does.  d_flow is one store per element and always reproducible."""
        if mode != "bilinear":
            raise NotImplementedError("warp: backward exists for mode='bilinear' only")
        if needs[0]:
            alert_not_deterministic("ofb200 warp backward with respect to the frame (ofb_warp_backward d_frame)")
        frame_d, flow_d = saved
        with torch.cuda.device(frame_d.device):
            frame_c, flow_c = frame_d.contiguous(), flow_d.contiguous()
            grad_c = grad_out.contiguous()
            d_frame = torch.zeros((b, c, h, w), dtype=torch.float32, device=frame_c.device) if needs[0] else None
            d_flow = torch.empty((b, 2, h, w), dtype=flow_c.dtype, device=frame_c.device) if needs[1] else None
            rc = ofb200.load().ofb_warp_backward(
                ofb200.ptr(frame_c), _WARP_DTYPES[frame_c.dtype], ofb200.ptr(flow_c), _WARP_DTYPES[flow_c.dtype],
                ofb200.ptr(grad_c), ofb200.ptr(d_frame), ofb200.ptr(d_flow), b, c, h, w, ofb200.PAD[padding_mode],
                int(bool(align_corners)), mul_x, mul_y, ofb200.stream_ptr(),
            )
            ofb200.check(rc, "ofb_warp_backward")
        return (d_frame.to(frame_c.dtype) if d_frame is not None else None), d_flow

    return _run(run, "warp", frame, flow, bwd=backward)


def warp_grid(flow: Tensor) -> Tensor:
    """Warping grid of a normalised flow map, (B, H, W, 2) -> (B, H, W, 2) (reference operator.py:36-56).

    `warp` never materialises this grid; the function exists for API parity.  Differentiable: the grid is the base
    grid plus the flow, so the flow's gradient is the grid's gradient itself.
    """
    b, h, w, _ = flow.shape
    _check_f32(flow)

    def run(flow_d: Tensor):
        flow_d = flow_d.contiguous()
        grid = torch.empty_like(flow_d)
        rc = ofb200.load().ofb_warp_grid_f32(ofb200.ptr(flow_d), ofb200.ptr(grid), b, h, w, ofb200.stream_ptr())
        ofb200.check(rc, "ofb_warp_grid_f32")
        return grid

    def backward(saved, grad_out: Tensor, needs):
        return (grad_out,)

    return _run(run, "warp_grid", flow, bwd=backward)


_SCALE_DTYPES = {torch.float32: ofb200.DTYPE_F32, torch.float64: ofb200.DTYPE_F64, torch.float16: ofb200.DTYPE_F16,
                 torch.bfloat16: ofb200.DTYPE_BF16}


def scale(flow: Tensor, factor: Union[float, Tuple[float, float]] = 1.0) -> Tensor:
    """Scales the optical flow by a constant in X- and Y-direction (reference operator.py:59-82).

    Dtype-preserving like the reference (fp32, fp64, fp16, bf16): the factor is rounded to the flow's dtype, then one
    multiply in that dtype."""
    assert flow.size(1) == 2
    if isinstance(factor, (float, int)):
        factor = (factor, factor)
    assert len(factor) == 2
    if flow.dtype not in _SCALE_DTYPES:
        raise NotImplementedError(f"scale: no B200 kernel for {flow.dtype} flows (fp32, fp64, fp16, bf16)")
    dt = _SCALE_DTYPES[flow.dtype]
    b = flow.shape[0]
    hw = flow[0, 0].numel() if b > 0 else 0
    fx, fy = float(factor[0]), float(factor[1])

    def run(flow_d: Tensor):
        flow_d = flow_d.contiguous()
        out = torch.empty_like(flow_d)
        rc = ofb200.load().ofb_scale_flow(ofb200.ptr(flow_d), ofb200.ptr(out), dt, b, hw, fx, fy, ofb200.stream_ptr())
        ofb200.check(rc, "ofb_scale_flow")
        return out

    def backward(saved, grad_out: Tensor, needs):
        """d scale / d flow is the same per-channel multiply applied to the incoming gradient."""
        with torch.cuda.device(grad_out.device):
            return (run(grad_out),)

    return _run(run, "scale", flow, bwd=backward)


def _resize_raw(x: Tensor, size: Tuple[int, int], align_corners: bool, mul_x: float, mul_y: float, name: str) -> Tensor:
    n, c, h, w = x.shape
    ho, wo = int(size[0]), int(size[1])

    def run(x_d: Tensor):
        x_d = x_d.contiguous()
        out = torch.empty((n, c, ho, wo), dtype=torch.float32, device=x_d.device)
        rc = ofb200.load().ofb_resize_bilinear_f32(
            ofb200.ptr(x_d), ofb200.ptr(out), n, c, h, w, ho, wo, int(align_corners), float(mul_x), float(mul_y),
            ofb200.stream_ptr(),
        )
        ofb200.check(rc, "ofb_resize_bilinear_f32")
        return out

    def backward(saved, grad_out: Tensor, needs):
        """Adjoint of the bilinear resize: scatter the output gradient with the forward weights."""
        with torch.cuda.device(grad_out.device):
            d_in = torch.zeros((n, c, h, w), dtype=torch.float32, device=grad_out.device)
            rc = ofb200.load().ofb_resize_bilinear_backward_f32(
                ofb200.ptr(grad_out.contiguous()), ofb200.ptr(d_in), n, c, h, w, ho, wo, int(align_corners), float(mul_x),
                float(mul_y), ofb200.stream_ptr(),
            )
            ofb200.check(rc, "ofb_resize_bilinear_backward_f32")
        return (d_in,)

    return _run(run, name, x, bwd=backward)


def resize(
    flow: Tensor,
    size: Optional[Tuple[int, int]] = None,
    scale_factor: Optional[float] = None,
    mode: str = "bilinear",
) -> Tensor:
    """Resizes the flow spatially and re-scales its magnitude accordingly (reference operator.py:85-114)."""
    assert flow.size(1) == 2
    assert flow.ndimension() == 4
    if mode != "bilinear":
        raise NotImplementedError(f"resize: mode={mode!r} has no B200 kernel (bilinear only)")
    _check_f32(flow)
    in_h, in_w = flow.shape[-2:]
    if scale_factor:                                     # Python's round: banker's rounding, as the reference (:109)
        size = (round(in_h * scale_factor), round(in_w * scale_factor))
    out_h, out_w = int(size[0]), int(size[1])
    # the flow vectors are measured in pixels of the new grid: x scales with the width ratio, y with the height ratio
    return _resize_raw(flow, (out_h, out_w), False, out_w / in_w, out_h / in_h, "resize")


def _half_extent(flow: Tensor) -> Tuple[float, float]:
    """(W-1)/2, (H-1)/2 with the reference's guard for single-pixel dimensions (operator.py:129,145)."""
    rows, cols = flow.shape[-2:]
    return max(cols - 1, 1) / 2, max(rows - 1, 1) / 2


def normalize(flow: Tensor) -> Tensor:
    """Pixel units -> normalised [-1, 1] units (reference operator.py:117-130)."""
    assert flow.size(1) == 2
    half_w, half_h = _half_extent(flow)
    return scale(flow, (1.0 / half_w, 1.0 / half_h))


def denormalize(flow: Tensor) -> Tensor:
    """Normalised units -> pixel units (reference operator.py:133-146)."""
    assert flow.size(1) == 2
    return scale(flow, _half_extent(flow))


def integrate(*flows: Tensor) -> Tensor:
    """Integrates a sequence of flow maps into one (reference operator.py:149-165): a right fold,
    total_k = flow_k + warp(total_{k+1}, flow_k), starting from the last flow."""
    assert len(flows) >= 2
    assert all(f.shape == flows[0].shape for f in flows), "integrate: the flows differ in shape"
    accumulated = flows[-1]
    for step in range(len(flows) - 2, -1, -1):
        accumulated = flows[step] + warp(accumulated, flows[step])
    return accumulated
