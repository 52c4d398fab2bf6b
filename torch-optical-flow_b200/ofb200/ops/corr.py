"""RAFT correlation block with the reference's interface (reference methods/raft/model/corr.py),
built by the K2 tcgen05 kernel and sampled by the K3 lookup kernel of libofb200.

Differences a caller can observe, all deliberate (DESIGN.md):
  * `corr_pyramid[l]` keeps the reference's shape (B*h*w, 1, h_l, w_l) but is a strided view of a
    padded buffer (row pitch rounded up to 8 elements for TMA) and is stored in bf16 by default;
    pass `pyramid_dtype=torch.float16` for the precision the reference's shipped configs store it in
    (`precision: 16`: an fp16 pyramid, the same bytes and tensor-core path as bf16, 3 more significand
    bits, but correlations beyond +-65504 become inf), or `torch.float32` for an fp32 pyramid (CUDA-core builder).
  * differentiable with respect to the feature maps (K3 backward kernel + two library GEMMs per level) and, as
    bilinear_sampler's grid_sample is in the reference (utils.py:64-80), with respect to the lookup coordinates (one
    K3 coordinate-backward launch per lookup, only when the coordinates require grad; RAFT itself detaches them,
    raft.py:127).  A coordinate whose window leaves the floor guard, or is non-finite, gets gradient 0 at that level
    (the reference: NaN for NaN).  Forward-only, as before: `return_index=True` lookups and `on_demand=True` blocks.
  * the lookup's output is fp32, as the reference's (corr.py:77), unless `lookup_dtype` (or OFB200_LOOKUP_DTYPE) asks
    for fp16 or bf16: each fp32 sample rounded once, the same bits as the fp32 output cast to that dtype.  "autocast"
    picks the dtype CUDA autocast would cast the output to before its only consumer, BasicMotionEncoder.convc1
    (update.py:114), so that cast and its backward disappear while convc1 receives the same bits; the gradient is then
    read back in that dtype, widened exactly.
"""
import ctypes
import math
import os
from typing import List, Optional

import torch
from torch import Tensor

import ofb200


def _default_pyramid_dtype() -> torch.dtype:
    name = os.environ.get("OFB200_PYRAMID_DTYPE", "bf16").lower()
    if name in ("fp32", "f32", "float32"):
        return torch.float32
    if name in ("fp16", "f16", "float16", "half"):
        return torch.float16
    return torch.bfloat16


_LOOKUP_DTYPES = {"fp32": torch.float32, "f32": torch.float32, "float32": torch.float32, "fp16": torch.float16,
                  "f16": torch.float16, "float16": torch.float16, "half": torch.float16, "bf16": torch.bfloat16,
                  "bfloat16": torch.bfloat16, "autocast": "autocast"}


def _default_lookup_dtype():
    """OFB200_LOOKUP_DTYPE=fp32|fp16|bf16|autocast; unset means fp32."""
    name = os.environ.get("OFB200_LOOKUP_DTYPE", "").lower() or "fp32"
    if name not in _LOOKUP_DTYPES:
        raise ValueError(f"OFB200_LOOKUP_DTYPE must be fp32, fp16, bf16 or autocast, got {name!r}")
    return _LOOKUP_DTYPES[name]


# optional ofb200.runner.KernelTimers: when set (bench.py), the prep launches and the pyramid kernel get their own
# CUDA-event brackets on the launching stream
TIMERS = None


class _NullSpan:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def _span(name: str, launches: int):
    return TIMERS.span(name, launches) if TIMERS is not None else _NullSpan()


_IN_DTYPES = {torch.float32: ofb200.DTYPE_F32, torch.bfloat16: ofb200.DTYPE_BF16, torch.float16: ofb200.DTYPE_F16}


def prepare_operands(fmap1: Tensor, fmap2: Tensor, num_levels: int, dtype: torch.dtype = torch.bfloat16):
    """K-major operands of the tcgen05 builder in `dtype` (bf16 or fp16): fmap1, fmap2, and (for pyramids with more
    than two levels) fmap2 averaged over complete 4x4 blocks.  (B, C, h, w) CUDA inputs in fp32, bf16 or fp16:
    half-precision maps (autocast callers) are read as they are, without an fp32 round trip.

    bf16 operands carry the 1/sqrt(C) of corr.py:87 folded into fmap1 (build with scale 1.0).  fp16 operands do not:
    the fp16 builder applies it to its fp32 accumulators, the reference's order under autocast (an fp16 matmul of the
    rounded maps, then the scale), and fmap1/sqrt(C) stays out of fp16 subnormals.  `operand_scale` says which."""
    if dtype not in (torch.bfloat16, torch.float16):
        raise NotImplementedError("prepare_operands: the tcgen05 builder's operands are bf16 or fp16")
    b, c, h, w = fmap1.shape
    dt1, dt2 = _IN_DTYPES[fmap1.dtype], _IN_DTYPES[fmap2.dtype]
    out_dt = _IN_DTYPES[dtype]
    lib = ofb200.load()
    st = ofb200.stream_ptr()
    dev = fmap1.device
    a_km = torch.empty((b, h * w, c), dtype=dtype, device=dev)
    b_km = torch.empty((b, h * w, c), dtype=dtype, device=dev)
    q_km = torch.empty((b, (h // 4) * (w // 4), c), dtype=dtype, device=dev) if num_levels > 2 else None
    scale = operand_scale(c, dtype)
    ofb200.check(lib.ofb_corr_prep_to(ofb200.ptr(fmap1), dt1, ofb200.ptr(a_km), out_dt, b, c, h, w, 1, scale, st),
                 "ofb_corr_prep_to")
    ofb200.check(lib.ofb_corr_prep_to(ofb200.ptr(fmap2), dt2, ofb200.ptr(b_km), out_dt, b, c, h, w, 1, 1.0, st),
                 "ofb_corr_prep_to")
    if q_km is not None:
        ofb200.check(lib.ofb_corr_prep_to(ofb200.ptr(fmap2), dt2, ofb200.ptr(q_km), out_dt, b, c, h, w, 4, 1.0, st),
                     "ofb_corr_prep_to")
    return a_km, b_km, q_km


def operand_scale(c: int, dtype: torch.dtype = torch.bfloat16) -> float:
    """The factor prepare_operands folds into fmap1: 1/sqrt(C) for bf16 operands, 1 for fp16 ones."""
    return 1.0 / math.sqrt(float(c)) if dtype == torch.bfloat16 else 1.0


def build_pyramid(ops, pyr, b: int, c: int, h: int, w: int, dtype: torch.dtype = torch.bfloat16, cta_group: int = 0) -> int:
    """Run the tcgen05 builder of `dtype` on prepare_operands' output; returns the library's status code."""
    lib = ofb200.load()
    fn = lib.ofb_corr_pyramid_f16 if dtype == torch.float16 else lib.ofb_corr_pyramid_bf16
    scale = (1.0 / math.sqrt(float(c))) / operand_scale(c, dtype)     # what the operands do not carry yet
    return fn(ofb200.ptr(ops[0]), ofb200.ptr(ops[1]), ofb200.ptr(ops[2]), ctypes.byref(pyr), b, c, h, w, scale,
              int(cta_group), ofb200.stream_ptr())


def level_images(buf: Tensor, layout: int, q: int, pitch: int) -> Tensor:
    """One pyramid level's buffer in `layout` (OFB_LAYOUT_*, include/ofb200.h) -> its (q, rows, pitch) images, rows =
    buf.numel() // (q * pitch): a view of the buffer for rows, a copy that unfolds the 8x4 blocks otherwise.  The inverse
    of level_buffer."""
    rows = buf.numel() // (q * pitch)
    if layout == ofb200.LAYOUT_ROWS:
        return buf.view(q, rows, pitch)
    if layout == ofb200.LAYOUT_QMINOR8X4:
        return buf.view(rows // 4, pitch // 8, q, 4, 8).permute(2, 0, 3, 1, 4).reshape(q, rows, pitch)   # (by, bx, q, y, x)
    return buf.view(q, rows // 4, pitch // 8, 4, 8).permute(0, 1, 3, 2, 4).reshape(q, rows, pitch)       # (q, by, bx, y, x)


def level_buffer(img: Tensor, layout: int) -> Tensor:
    """(q, rows, pitch) images -> one pyramid level's contiguous buffer in `layout` (8x4 blocks: rows a multiple of 4,
    pitch a multiple of 8).  The inverse of level_images."""
    q, rows, pitch = img.shape
    if layout == ofb200.LAYOUT_ROWS:
        return img.contiguous()
    order = (1, 3, 0, 2, 4) if layout == ofb200.LAYOUT_QMINOR8X4 else (0, 1, 3, 2, 4)   # (by, bx, q, y, x) / (q, by, bx, y, x)
    return img.reshape(q, rows // 4, 4, pitch // 8, 8).permute(*order).contiguous()


class _GradState:
    """What the backward nodes of one CorrBlock share: the dense fp32 gradient pyramid the lookups' backwards
    accumulate into, and the few scalars needed to allocate and consume it.  The autograd contexts hold THIS object,
    never the CorrBlock: block -> handle tensor -> grad_fn -> ctx -> block would be a reference cycle that keeps the
    pyramid buffers (2.8 GB per 1080p pair) alive until Python's cyclic collector runs."""

    def __init__(self, shape, dev, num_levels: int, radius: int, pyr_dtype: int) -> None:
        self.shape, self.dev, self.num_levels, self.radius, self.pyr_dtype = shape, dev, num_levels, radius, pyr_dtype
        self.dpyr: Optional[List[Optional[Tensor]]] = None
        self.dpyr_desc = None
        self.task = None                      # autograd graph task the gradient pyramid belongs to

    def grad_pyramid(self):
        """The gradient pyramid of the CURRENT backward pass.  A pyramid left behind by another pass (a backward that
        raised, or never reached the handle node) is dropped, not accumulated into."""
        task = torch._C._current_graph_task_id() if hasattr(torch._C, "_current_graph_task_id") else None
        if self.dpyr is None or any(t is None for t in self.dpyr) or task != self.task:
            self.alloc()
            self.task = task
        return self.dpyr_desc

    def alloc(self) -> None:
        """Dense fp32 gradient levels (B*h*w, h_l*w_l), tight rows, zero-filled."""
        b, c, h, w = self.shape
        desc = ofb200.Pyramid()
        elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
        ofb200.check(ofb200.load().ofb_pyramid_layout(h, w, self.num_levels, 0, ctypes.byref(desc), ctypes.byref(elems)),
                     "ofb_pyramid_layout")
        desc.dtype = ofb200.DTYPE_F32
        self.dpyr = []
        for lvl in range(self.num_levels):
            buf = torch.zeros(b * h * w * int(elems[lvl]), dtype=torch.float32, device=self.dev)
            self.dpyr.append(buf)
            desc.base[lvl] = buf.data_ptr()
        self.dpyr_desc = desc

    def release(self) -> None:
        self.dpyr, self.dpyr_desc, self.task = None, None, None


class _PyramidHandle(torch.autograd.Function):
    """Graph node standing for "the pyramid built from (fmap1, fmap2)".  Its output is a dummy scalar every
    lookup depends on; autograd therefore runs this backward after all the lookups' backwards, when the gradient
    pyramid is complete, and turns it into feature-map gradients:
        pyr_l = fmap1^T . pool_l(fmap2) / sqrt(C)        (pooling is linear, reference corr.py:45-54)
        d fmap1 = sum_l pool_l(fmap2) . dP_l^T / sqrt(C);  d pool_l(fmap2) = fmap1 . dP_l / sqrt(C)
    With a bf16 pyramid (default) all of it runs on this library's kernels: pooled bf16 operands, the long-K tcgen05
    GEMMs, and a fused pooling-adjoint + layout pass; with an fp32 pyramid (the parity configuration) the GEMMs are fp32
    library GEMMs and the pooling adjoint goes through autograd."""

    @staticmethod
    def forward(ctx, state, fmap1, fmap2):
        ctx.state = state
        ctx.save_for_backward(fmap1.detach(), fmap2.detach())
        return torch.zeros(1, dtype=torch.float32, device=fmap1.device)

    @staticmethod
    def backward(ctx, _grad_handle):
        blk = ctx.state
        fmap1, fmap2 = ctx.saved_tensors
        b, c, h, w = fmap1.shape
        d1 = d2 = None
        task = torch._C._current_graph_task_id() if hasattr(torch._C, "_current_graph_task_id") else None
        if blk.dpyr is not None and blk.task == task:
            scale = 1.0 / math.sqrt(float(c))
            # The two GEMMs per level.  "tcgen05" (default with a bf16 or fp16 pyramid): bf16 operands, fp32
            # accumulation, this library's long-K tensor-core kernel fed by one cast / transpose pass over the fp32
            # gradient level -- the precision of a `precision: 16` run of the reference.  It reads only the fp32 gradient
            # pyramid and the feature maps, never the stored pyramid, and bf16 keeps the gradients' fp32 range (fp16
            # operands would underflow without loss scaling).  "fp32" (default with an fp32 pyramid; matches the
            # reference's fp32 autograd to 1e-5) and "bf16" go through the library bmm.  OFB200_BWD_GEMM overrides.
            tc_ok = c % 32 == 0 and c <= 256
            half_pyr = blk.pyr_dtype in (ofb200.DTYPE_BF16, ofb200.DTYPE_F16)
            mode = os.environ.get("OFB200_BWD_GEMM", "").lower() or ("tcgen05" if half_pyr and tc_ok else "fp32")
            if mode == "tcgen05" and not tc_ok:
                raise NotImplementedError("CorrBlock backward: the tcgen05 GEMM needs C to be a multiple of 32, at most 256")
            d_levels = []
            if mode == "tcgen05":
                # everything on this library's kernels: pooled bf16 operands (ofb_pool_cast_bf16), one cast / transpose
                # pass per gradient level (ofb_cast_bf16), the two long-K tcgen05 GEMMs (ofb_gemm_nt_bf16), and one
                # pooling-adjoint + layout pass per feature map (ofb_pool_adjoint_f32)
                lib, st = ofb200.load(), ofb200.stream_ptr()
                dev = fmap1.device
                n = h * w
                pn = (n + 7) // 8 * 8
                f1c, f2c = fmap1.contiguous(), fmap2.contiguous()
                d1t = torch.zeros((b, n, c), dtype=torch.float32, device=dev)                  # d fmap1^T, summed over levels
                f1_16 = torch.empty((b, c, pn), dtype=torch.bfloat16, device=dev)
                ofb200.check(lib.ofb_pool_cast_bf16(ofb200.ptr(f1c), _IN_DTYPES[f1c.dtype], ofb200.ptr(f1_16), b, c, h, w, 1, pn, st),
                             "ofb_pool_cast_bf16")
                d2_levels = []
                for lvl in range(blk.num_levels):
                    hl, wl = h >> lvl, w >> lvl
                    nl = hl * wl
                    pk = (nl + 7) // 8 * 8
                    a16 = torch.empty((b, n, pk), dtype=torch.bfloat16, device=dev)            # bf16(dP_l)
                    a16_t = torch.empty((b, nl, pn), dtype=torch.bfloat16, device=dev)         # bf16(dP_l)^T
                    ofb200.check(lib.ofb_cast_bf16(ofb200.ptr(blk.dpyr[lvl]), ofb200.ptr(a16), ofb200.ptr(a16_t), b, n, nl,
                                                   pk, pn, st), "ofb_cast_bf16")
                    blk.dpyr[lvl] = None                                                        # free level by level
                    f2_16 = torch.empty((b, c, pk), dtype=torch.bfloat16, device=dev)          # bf16(avgpool_l(fmap2)), K-padded
                    ofb200.check(lib.ofb_pool_cast_bf16(ofb200.ptr(f2c), _IN_DTYPES[f2c.dtype], ofb200.ptr(f2_16), b, c, h, w,
                                                        1 << lvl, pk, st), "ofb_pool_cast_bf16")
                    ofb200.check(lib.ofb_gemm_nt_bf16(ofb200.ptr(a16), ofb200.ptr(f2_16), ofb200.ptr(d1t), b, n, c, nl, pk, pk, c,
                                                      n * pk, c * pk, n * c, scale, 1, st), "ofb_gemm_nt_bf16")
                    d2t = torch.empty((b, nl, c), dtype=torch.float32, device=dev)
                    ofb200.check(lib.ofb_gemm_nt_bf16(ofb200.ptr(a16_t), ofb200.ptr(f1_16), ofb200.ptr(d2t), b, nl, c, n, pn, pn, c,
                                                      nl * pn, c * pn, nl * c, scale, 0, st), "ofb_gemm_nt_bf16")
                    d2_levels.append(d2t)
                d1 = torch.empty((b, c, h, w), dtype=torch.float32, device=dev)
                d2 = torch.empty((b, c, h, w), dtype=torch.float32, device=dev)
                one = (ctypes.c_void_p * ofb200.MAX_LEVELS)(d1t.data_ptr())
                ofb200.check(lib.ofb_pool_adjoint_f32(one, ofb200.ptr(d1), b, c, h, w, 1, st), "ofb_pool_adjoint_f32")
                ptrs = (ctypes.c_void_p * ofb200.MAX_LEVELS)(*[t.data_ptr() for t in d2_levels])
                ofb200.check(lib.ofb_pool_adjoint_f32(ptrs, ofb200.ptr(d2), b, c, h, w, blk.num_levels, st), "ofb_pool_adjoint_f32")
                d1 = d1.to(fmap1.dtype)
                d2 = d2.to(fmap2.dtype)
            else:
                f1 = fmap1.float().reshape(b, c, h * w)
                with torch.enable_grad():
                    leaf = fmap2.float().detach().requires_grad_(True)
                    levels, cur = [leaf], leaf
                    for _ in range(blk.num_levels - 1):
                        cur = torch.nn.functional.avg_pool2d(cur, 2, stride=2)
                        levels.append(cur)
                gemm_dt = torch.bfloat16 if mode == "bf16" else torch.float32
                f1g = f1.to(gemm_dt)
                d1 = torch.zeros_like(f1)
                for lvl, f2l in enumerate(levels):
                    hl, wl = f2l.shape[-2:]
                    dp = blk.dpyr[lvl].view(b, h * w, hl * wl).to(gemm_dt)               # (B, N, N_l), tight rows
                    f2g = f2l.detach().reshape(b, c, hl * wl).to(gemm_dt)
                    d1.add_(torch.bmm(f2g, dp.transpose(1, 2)).float(), alpha=scale)
                    d_levels.append((torch.bmm(f1g, dp).float() * scale).view(b, c, hl, wl))
                    blk.dpyr[lvl] = None                                                # free level by level
                d2 = torch.autograd.grad(levels, leaf, d_levels)[0]
                d1 = d1.view(b, c, h, w).to(fmap1.dtype)
                d2 = d2.to(fmap2.dtype)
        blk.release()                                                            # free the gradient pyramid
        need1, need2 = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        return None, (d1 if need1 else None), (d2 if need2 else None)


class _LookupFn(torch.autograd.Function):
    """One CorrBlock.__call__: forward = the K3 kernel; backward = the coordinate gradient (when `coords_d` requires
    grad) and the scatter into the block's gradient pyramid (when there is a handle, i.e. the feature maps require
    grad).  The context never keeps the CorrBlock (see _GradState).  Only a lookup whose coordinates require grad keeps
    the stored pyramid's buffers, which its backward reads: with detached coordinates the multi-GB pyramid is freed as
    soon as the block is dropped, while the graph lives on.  The output gradient is read in its own dtype."""

    @staticmethod
    def forward(ctx, block, coords_d, handle, out_dtype):
        ctx.state = block._grad
        if ctx.needs_input_grad[1]:
            ctx.pyr, ctx.buffers = block._pyr, block._buffers
        ctx.shape, ctx.dev, ctx.radius = block._shape, block._dev, block.radius
        ctx.save_for_backward(coords_d)
        return block._lookup(coords_d.detach(), None, None, None, out_dtype)

    @staticmethod
    def backward(ctx, grad_out):
        st = ctx.state
        (coords_d,) = ctx.saved_tensors
        b, c, h, w = ctx.shape
        g = grad_out.contiguous()
        g_dt = _IN_DTYPES[g.dtype]
        d_coords = None
        with torch.cuda.device(ctx.dev):
            if ctx.needs_input_grad[1]:
                d_coords = torch.empty((b, 2, h, w), dtype=torch.float32, device=ctx.dev)
                rc = ofb200.load().ofb_corr_lookup_coords_backward_from(
                    ctypes.byref(ctx.pyr), ofb200.ptr(coords_d), ofb200.ptr(g), g_dt, ofb200.ptr(d_coords), b, h, w,
                    ctx.radius, ofb200.stream_ptr())
                ofb200.check(rc, "ofb_corr_lookup_coords_backward_from")
            if st is not None:
                desc = st.grad_pyramid()
                rc = ofb200.load().ofb_corr_lookup_backward(
                    ctypes.byref(desc), ofb200.ptr(coords_d), ofb200.ptr(g), g_dt, b, h, w, st.radius, ofb200.stream_ptr())
                ofb200.check(rc, "ofb_corr_lookup_backward")
        handle_grad = torch.zeros(1, dtype=torch.float32, device=ctx.dev) if st is not None else None
        return None, d_coords, handle_grad, None


class CorrBlock:
    def __init__(
        self,
        fmap1: Tensor,
        fmap2: Tensor,
        num_levels: int = 4,
        radius: int = 4,
        *,
        pyramid_dtype: Optional[torch.dtype] = None,
        builder: str = "auto",
        cta_group: int = 0,
        on_demand: Optional[bool] = None,
        lookup_dtype=None,
    ) -> None:
        """fmap1, fmap2 (B, C, h, w) in fp32 / bf16 / fp16 (reference corr.py:38-54).

        Extensions (keyword-only, defaults keep the reference's behaviour): `pyramid_dtype` (bf16 default; fp16 is the
        precision the reference stores its pyramid in under `precision: 16`; fp32 selects the CUDA-core builder;
        OFB200_PYRAMID_DTYPE=bf16|fp16|fp32 sets the default; ignored with `on_demand`), `builder`, `cta_group` (K2
        launch mode), and `on_demand=True` (or OFB200_CORR_ON_DEMAND=1): nothing is materialised -- every lookup
        evaluates the correlation values of its own windows from the operand maps (ofb_corr_lookup_ondemand; 22 MB
        instead of 2.83 GB per 1080p pair, slower per lookup; forward-only).  `lookup_dtype`: the dtype of every lookup's
        output -- torch.float32 (default, the reference's), torch.float16, torch.bfloat16, or "autocast", resolved at
        each call to torch.get_autocast_dtype("cuda") while CUDA autocast is enabled and to fp32 otherwise;
        OFB200_LOOKUP_DTYPE=fp32|fp16|bf16|autocast sets the default."""
        self.num_levels = num_levels
        self.radius = radius
        if lookup_dtype is None:
            lookup_dtype = _default_lookup_dtype()
        if not (lookup_dtype == "autocast" or lookup_dtype in _IN_DTYPES):
            raise NotImplementedError('CorrBlock: lookup_dtype must be torch.float32, torch.float16, torch.bfloat16 or '
                                      '"autocast"')
        self.lookup_dtype = lookup_dtype
        if fmap1.shape != fmap2.shape or fmap1.dim() != 4:
            raise RuntimeError("CorrBlock: fmap1 and fmap2 must both be (B, C, h, w)")
        if not (1 <= num_levels <= ofb200.MAX_LEVELS):
            raise NotImplementedError(f"CorrBlock: num_levels must be in [1, {ofb200.MAX_LEVELS}]")
        if pyramid_dtype is None:
            pyramid_dtype = _default_pyramid_dtype()
        if pyramid_dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise NotImplementedError("CorrBlock: pyramid_dtype must be torch.float32, torch.bfloat16 or torch.float16")
        self._on_host = not fmap1.is_cuda
        # training: keep the differentiable feature maps behind a handle node the lookups depend on
        self._handle = None
        self._grad: Optional[_GradState] = None
        diff_maps = None
        if torch.is_grad_enabled() and (fmap1.requires_grad or fmap2.requires_grad):
            diff_maps = (ofb200.to_device(fmap1), ofb200.to_device(fmap2))
        fmap1 = ofb200.to_device(fmap1).detach()
        fmap2 = ofb200.to_device(fmap2).detach()
        if fmap1.dtype not in _IN_DTYPES or fmap2.dtype not in _IN_DTYPES:
            raise NotImplementedError(f"CorrBlock: feature maps must be fp32, bf16 or fp16, got {fmap1.dtype} / {fmap2.dtype}")
        fmap1, fmap2 = fmap1.contiguous(), fmap2.contiguous()
        b, c, h, w = fmap1.shape
        if (h >> (num_levels - 1)) == 0 or (w >> (num_levels - 1)) == 0:
            # F.avg_pool2d in the reference: "Output size is too small" (corr.py:53)
            raise RuntimeError("CorrBlock: feature map too small for the requested number of pyramid levels")
        self._shape = (b, c, h, w)
        self._dev = fmap1.device
        lib = ofb200.load()
        if on_demand is None:
            on_demand = os.environ.get("OFB200_CORR_ON_DEMAND", "0") not in ("", "0")
        self._on_demand = None
        if on_demand:
            if diff_maps is not None:
                raise NotImplementedError("CorrBlock(on_demand=True) is forward-only: the feature maps must not require grad")
            if c not in (64, 128, 256) or radius > 4:
                raise NotImplementedError("CorrBlock(on_demand=True) needs C in {64, 128, 256} and radius <= 4")
            self.builder = "on_demand"
            self._buffers, self._views, self._pyr = [], None, None
            scale = 1.0 / math.sqrt(float(c))
            st = ofb200.stream_ptr()
            with torch.cuda.device(self._dev):
                a_km = torch.empty((b, h * w, c), dtype=torch.bfloat16, device=self._dev)
                ofb200.check(lib.ofb_corr_prep_from(ofb200.ptr(fmap1), _IN_DTYPES[fmap1.dtype], ofb200.ptr(a_km), b, c, h, w, 1,
                                                    scale, st), "ofb_corr_prep_from")
                levels = []
                for lvl in range(num_levels):
                    f2l = torch.empty((b, (h >> lvl) * (w >> lvl), c), dtype=torch.bfloat16, device=self._dev)
                    ofb200.check(lib.ofb_corr_prep_from(ofb200.ptr(fmap2), _IN_DTYPES[fmap2.dtype], ofb200.ptr(f2l), b, c, h, w,
                                                        1 << lvl, 1.0, st), "ofb_corr_prep_from")
                    levels.append(f2l)
            self._on_demand = (a_km, levels)
            return
        tc_ok = pyramid_dtype in (torch.bfloat16, torch.float16) and c % 64 == 0 and c <= 256
        if builder == "auto":
            builder = "tcgen05" if tc_ok else "simt"
        if builder == "tcgen05" and not tc_ok:
            raise NotImplementedError("CorrBlock: the tcgen05 builder needs a bf16 or fp16 pyramid and C in {64,128,192,256}")
        self.builder = builder
        if builder != "tcgen05":
            # the CUDA-core builder reads fp32; the tcgen05 prep reads bf16 / fp16 maps (autocast callers) as they are.
            # An fp16 pyramid is the correlation of the fp16-rounded maps, whichever builder makes it (autocast's matmul
            # operands, corr.py:85)
            if pyramid_dtype == torch.float16 and fmap1.dtype != torch.float16:
                fmap1, fmap2 = fmap1.half(), fmap2.half()
            if fmap1.dtype != torch.float32:
                fmap1, fmap2 = fmap1.float(), fmap2.float()

        pyr = ofb200.Pyramid()
        elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
        # tcgen05 builder: 8x4-blocked 16-bit levels (what the lookup kernel reads with the fewest DRAM atoms),
        # query-minor by default (OFB200_PYRAMID_LAYOUT=blocked|qminor); CUDA-core builder: padded rows
        blocked_mode = 2 if os.environ.get("OFB200_PYRAMID_LAYOUT", "qminor").lower() == "blocked" else 3
        mode = blocked_mode if (builder == "tcgen05" and radius in (3, 4)) else 1
        ofb200.check(lib.ofb_pyramid_layout(h, w, num_levels, mode, ctypes.byref(pyr), ctypes.byref(elems)), "ofb_pyramid_layout")
        pyr.dtype = _IN_DTYPES[pyramid_dtype]
        n = h * w
        self._buffers = []
        self._views: Optional[List[Tensor]] = None
        with torch.cuda.device(self._dev):
            for lvl in range(num_levels):
                # the tcgen05 builder writes the row padding itself (zeros); the CUDA-core builder does not,
                # and the lookup kernel requires finite values there
                alloc = torch.empty if builder == "tcgen05" else torch.zeros
                buf = alloc(b * n * int(elems[lvl]), dtype=pyramid_dtype, device=self._dev)
                self._buffers.append(buf)
                pyr.base[lvl] = buf.data_ptr()
            self._pyr = pyr
            if diff_maps is not None:
                self._grad = _GradState(self._shape, self._dev, num_levels, radius, int(pyr.dtype))
                self._handle = _PyramidHandle.apply(self._grad, *diff_maps)
            scale = 1.0 / math.sqrt(float(c))
            if builder == "tcgen05":
                with _span("corr_prep", 3 if num_levels > 2 else 2):
                    ops = prepare_operands(fmap1, fmap2, num_levels, pyramid_dtype)
                with _span("corr_pyramid_kernel", 2 if num_levels > 2 else 1):
                    rc = build_pyramid(ops, pyr, b, c, h, w, pyramid_dtype, cta_group)
                ofb200.check(rc, "ofb_corr_pyramid_f16" if pyramid_dtype == torch.float16 else "ofb_corr_pyramid_bf16")
                # keep the operands alive until the stream has consumed them
                for t in ops:
                    if t is not None:
                        t.record_stream(torch.cuda.current_stream())
            elif builder == "simt":
                rc = lib.ofb_corr_pyramid_simt_f32(ofb200.ptr(fmap1), ofb200.ptr(fmap2), ctypes.byref(pyr), b, c, h, w,
                                                   scale, ofb200.stream_ptr())
                ofb200.check(rc, "ofb_corr_pyramid_simt_f32")
            else:
                raise ValueError(f"CorrBlock: unknown builder {builder!r}")

    @property
    def corr_pyramid(self) -> List[Tensor]:
        """The levels with the reference's shapes (B*h*w, 1, h_l, w_l) (reference corr.py:48-54).

        Row layout: strided views of the padded buffers.  8x4-blocked layouts (tcgen05 builder): the
        blocks are unfolded into a copy on first access (level_images) -- the lookup never needs this, only callers
        that inspect the volume do."""
        if self._on_demand is not None:
            raise NotImplementedError("CorrBlock(on_demand=True) does not materialise the correlation pyramid")
        if self._views is None:
            b, _, h, w = self._shape
            n = h * w
            views = []
            for lvl, buf in enumerate(self._buffers):
                hl, wl = int(self._pyr.lvl_h[lvl]), int(self._pyr.lvl_w[lvl])
                img = level_images(buf, self._pyr.layout, b * n, int(self._pyr.row_pitch[lvl]))
                views.append(img[:, :hl, :wl].unsqueeze(1))
            self._views = views
        return self._views

    def out_dtype(self) -> torch.dtype:
        """The dtype a lookup made now returns: `lookup_dtype`, with "autocast" resolved."""
        if self.lookup_dtype != "autocast":
            return self.lookup_dtype
        if not torch.is_autocast_enabled("cuda"):
            return torch.float32
        dt = torch.get_autocast_dtype("cuda")
        if dt not in _IN_DTYPES:
            raise NotImplementedError(f"CorrBlock: no lookup output in the autocast dtype {dt}")
        return dt

    def __call__(self, coords: Tensor, return_index: bool = False, out: Optional[Tensor] = None):
        """Index the pyramid (reference corr.py:56-77): coords (B, 2, h, w) -> (B, L*(2r+1)^2, h, w) in out_dtype()
        (fp32 unless `lookup_dtype` says otherwise).

        Differentiable with respect to `coords` when they require grad (host coordinates get a host gradient) and to
        the feature maps when those did at construction.  `return_index=True` (extension) also returns the floor
        indices (B*h*w, L, 2, 2r+1) int32 and the validity mask (B*h*w, L, (2r+1)^2) uint8 the kernel used; such a
        call, and every lookup of an `on_demand=True` block, is forward-only: its output carries no gradient.  `out`
        (extension) is an optional preallocated contiguous CUDA tensor of the output shape and dtype; on the
        differentiable path it receives the values and the returned tensor carries the graph."""
        b, c, h, w = self._shape
        if tuple(coords.shape) != (b, 2, h, w):
            raise RuntimeError(f"CorrBlock: coords must be {(b, 2, h, w)}, got {tuple(coords.shape)}")
        if coords.dtype != torch.float32:
            raise NotImplementedError("CorrBlock: coords must be fp32")
        on_host = not coords.is_cuda
        diff_coords = (torch.is_grad_enabled() and coords.requires_grad and not return_index
                       and self._on_demand is None)
        coords_d = ofb200.to_device(coords).contiguous()           # differentiable: a host leaf gets a host gradient
        if not diff_coords:
            coords_d = coords_d.detach()
        d = 2 * self.radius + 1
        lvls = self.num_levels
        oshape = (b, lvls * d * d, h, w)
        out_dtype = self.out_dtype()
        if out is not None and (tuple(out.shape) != oshape or out.dtype != out_dtype or not out.is_cuda
                                or not out.is_contiguous()):
            raise RuntimeError(f"CorrBlock: out must be a contiguous {out_dtype} CUDA tensor of shape {oshape}")
        idx = valid = None
        if diff_coords or (self._handle is not None and torch.is_grad_enabled() and not return_index):
            res = _LookupFn.apply(self, coords_d, self._handle, out_dtype)
            if out is not None:
                out.copy_(res.detach())                       # the preallocated buffer is filled, the graph keeps `res`
            out = res
        else:
            with torch.cuda.device(self._dev):
                if return_index:
                    idx = torch.empty((b * h * w, lvls, 2, d), dtype=torch.int32, device=self._dev)
                    valid = torch.empty((b * h * w, lvls, d * d), dtype=torch.uint8, device=self._dev)
            out = self._lookup(coords_d, out, idx, valid, out_dtype)
        if on_host:
            out = out.cpu()
            idx = idx.cpu() if idx is not None else None
            valid = valid.cpu() if valid is not None else None
        return (out, idx, valid) if return_index else out

    def _lookup(self, coords_d: Tensor, out: Optional[Tensor], idx: Optional[Tensor], valid: Optional[Tensor],
                out_dtype: torch.dtype = torch.float32) -> Tensor:
        b, c, h, w = self._shape
        d = 2 * self.radius + 1
        out_dt = _IN_DTYPES[out_dtype]
        with torch.cuda.device(self._dev):
            if out is None:
                out = torch.empty((b, self.num_levels * d * d, h, w), dtype=out_dtype, device=self._dev)
            if self._on_demand is not None:
                if idx is not None or valid is not None:
                    raise NotImplementedError("CorrBlock(on_demand=True): return_index is not available")
                a_km, levels = self._on_demand
                ptrs = (ctypes.c_void_p * ofb200.MAX_LEVELS)(*[t.data_ptr() for t in levels])
                rc = ofb200.load().ofb_corr_lookup_ondemand_to(ofb200.ptr(a_km), ptrs, ofb200.ptr(coords_d), ofb200.ptr(out),
                                                               out_dt, b, c, h, w, self.num_levels, self.radius,
                                                               ofb200.stream_ptr())
                ofb200.check(rc, "ofb_corr_lookup_ondemand_to")
                return out
            rc = ofb200.load().ofb_corr_lookup_to(
                ctypes.byref(self._pyr), ofb200.ptr(coords_d), ofb200.ptr(out), out_dt, ofb200.ptr(idx), ofb200.ptr(valid),
                b, h, w, self.radius, ofb200.stream_ptr(),
            )
        ofb200.check(rc, "ofb_corr_lookup_to")
        return out

    @staticmethod
    def corr(fmap1: Tensor, fmap2: Tensor, **kwargs) -> Tensor:
        """All-pairs correlation volume (B, h, w, 1, h, w) / sqrt(C) (reference corr.py:79-87).

        The reference's static method is an exact matmul in the inputs' precision, so the default here is the fp32
        CUDA-core builder (`pyramid_dtype=torch.bfloat16` or `torch.float16` selects the tcgen05 builder and a volume
        rounded to that type; fp16 is what the reference's matmul returns under autocast).
        Forward-only: the training path goes through the constructor (reference raft.py:112), which is
        differentiable; inputs that require grad raise instead of silently returning a detached volume."""
        if torch.is_grad_enabled() and (fmap1.requires_grad or fmap2.requires_grad):
            raise NotImplementedError("CorrBlock.corr: the static volume is forward-only; build CorrBlock(fmap1, fmap2) "
                                      "for the differentiable path, or call it under torch.no_grad()")
        kwargs.setdefault("pyramid_dtype", torch.float32)
        blk = CorrBlock(fmap1, fmap2, num_levels=1, radius=0, **kwargs)
        b, c, h, w = blk._shape
        vol = blk.corr_pyramid[0].reshape(b, h, w, 1, h, w).to(fmap1.dtype)
        return vol.cpu() if blk._on_host else vol
