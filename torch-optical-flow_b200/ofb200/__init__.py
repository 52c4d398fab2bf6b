"""ctypes binding of libofb200.so -- the C ABI declared in include/ofb200.h.

This is the only bridge between the Python call surface (optical_flow/, model/) and the
hand-written sm_100a kernels.  There is no CPU compute path and no fallback: if the shared
library is missing or no CUDA device is present, every op raises.
"""
import ctypes
import os
import subprocess
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libofb200.so")
CSRC = os.path.join(os.path.dirname(_HERE), "csrc")

MODE = {"bilinear": 0, "nearest": 1}
PAD = {"zeros": 0, "border": 1, "reflection": 2}
DTYPE_F32, DTYPE_BF16, DTYPE_F16, DTYPE_F64 = 0, 1, 2, 3
LAYOUT_ROWS, LAYOUT_BLOCK8X4, LAYOUT_QMINOR8X4 = 0, 1, 2
MAX_LEVELS = 4

_vp = ctypes.c_void_p
_i = ctypes.c_int
_i64 = ctypes.c_int64
_f = ctypes.c_float
MAX_PREDICTIONS = 24      # OFB_MAX_PREDICTIONS (include/ofb200.h)


class Pyramid(ctypes.Structure):
    """struct ofb_pyramid (include/ofb200.h)."""

    _fields_ = [
        ("base", _vp * MAX_LEVELS),
        ("q_stride", _i64 * MAX_LEVELS),
        ("row_pitch", ctypes.c_int32 * MAX_LEVELS),
        ("lvl_h", ctypes.c_int32 * MAX_LEVELS),
        ("lvl_w", ctypes.c_int32 * MAX_LEVELS),
        ("levels", ctypes.c_int32),
        ("dtype", ctypes.c_int32),
        ("layout", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
    ]


# name -> (restype, argtypes); must list every symbol include/ofb200.h declares
SIGNATURES = {
    "ofb_version": (_i, []),
    "ofb_strerror": (ctypes.c_char_p, [_i]),
    "ofb_launch_count": (_i64, []),
    "ofb_warp_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _vp]),
    "ofb_warp_backward_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _f, _vp]),
    "ofb_warp_grid_f32": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "ofb_scale_flow_f32": (_i, [_vp, _vp, _i, _i64, _f, _f, _vp]),
    "ofb_scale_flow": (_i, [_vp, _vp, _i, _i, _i64, ctypes.c_double, ctypes.c_double, _vp]),
    "ofb_resize_bilinear_backward_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _f, _vp]),
    "ofb_resize_bilinear_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _f, _vp]),
    "ofb_convex_upsample_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "ofb_convex_upsample": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _vp]),
    "ofb_epe_reduce_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "ofb_epe_map_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "ofb_outlier_reduce_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _vp]),
    "ofb_sequence_loss_backward_f32": (_i, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), _i, _vp, _vp, _vp, _i, _i, _i,
                                            ctypes.c_double, _f, _vp]),
    "ofb_convex_upsample_backward_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "ofb_convex_upsample_backward": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "ofb_sequence_loss_f32": (_i, [ctypes.POINTER(_vp), _i, _vp, _vp, _vp, _i, _i, _i, ctypes.c_double, _f, _vp]),
    "ofb_pyramid_layout": (_i, [_i, _i, _i, _i, ctypes.POINTER(Pyramid), ctypes.POINTER(_i64 * MAX_LEVELS)]),
    "ofb_corr_prep_bf16": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "ofb_corr_prep_from": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "ofb_corr_prep_to": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "ofb_corr_pyramid_bf16": (_i, [_vp, _vp, _vp, ctypes.POINTER(Pyramid), _i, _i, _i, _i, _f, _i, _vp]),
    "ofb_corr_pyramid_f16": (_i, [_vp, _vp, _vp, ctypes.POINTER(Pyramid), _i, _i, _i, _i, _f, _i, _vp]),
    "ofb_corr_pyramid_bf16_profile": (_i, [_vp, _vp, _vp, ctypes.POINTER(Pyramid), _i, _i, _i, _i, _f, _i, _vp, _vp]),
    "ofb_corr_pyramid_simt_f32": (_i, [_vp, _vp, ctypes.POINTER(Pyramid), _i, _i, _i, _i, _f, _vp]),
    "ofb_gemm_nt_bf16": (_i, [_vp, _vp, _vp, _i, _i, _i, _i] + [ctypes.c_longlong] * 6 + [_f, _i, _vp]),
    "ofb_cast_bf16": (_i, [_vp, _vp, _vp, _i, _i, _i, ctypes.c_longlong, ctypes.c_longlong, _vp]),
    "ofb_pool_cast_bf16": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "ofb_pool_adjoint_f32": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_backward_f32": (_i, [ctypes.POINTER(Pyramid), _vp, _vp, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_backward": (_i, [ctypes.POINTER(Pyramid), _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_coords_backward": (_i, [ctypes.POINTER(Pyramid), _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_coords_backward_from": (_i, [ctypes.POINTER(Pyramid), _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup": (_i, [ctypes.POINTER(Pyramid), _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_to": (_i, [ctypes.POINTER(Pyramid), _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_ondemand": (_i, [_vp, ctypes.POINTER(_vp), _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "ofb_corr_lookup_ondemand_to": (_i, [_vp, ctypes.POINTER(_vp), _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "ofb_bilinear_sampler_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
}

_lib = None
_lock = threading.Lock()


class OfbError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libofb200.so in-tree with nvcc for sm_100a (csrc/Makefile)."""
    res = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0:
        raise OfbError("building libofb200.so failed")
    return LIB_PATH


def load():
    """Load libofb200.so and bind every entry point.  Raises if the library is missing."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise OfbError(
                    f"{LIB_PATH} not found: build it with `make -C {CSRC}` (nvcc, sm_100a). "
                    "There is no CPU or PyTorch fallback for these ops."
                )
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().ofb_strerror(rc).decode()
        raise OfbError(f"{what} failed: {msg} (code {rc})")


def require_cuda():
    if not torch.cuda.is_available():
        raise OfbError("ofb200 kernels need a CUDA device (B200, sm_100a); there is no CPU compute path")


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def launch_count():
    return int(load().ofb_launch_count())


def to_device(t):
    """Stage a host tensor through the GPU (the ops themselves only run on CUDA)."""
    if t is None or t.is_cuda:
        return t
    require_cuda()
    return t.cuda(non_blocking=False)


class _NoBackward(torch.autograd.Function):
    """Forward-only kernels: differentiable inputs are accepted, backward raises."""

    @staticmethod
    def forward(ctx, fn, name, *tensors):
        ctx.op_name = name
        return fn(*[t.detach() for t in tensors])

    @staticmethod
    def backward(ctx, *grads):
        raise NotImplementedError(f"{ctx.op_name}: backward is not implemented (forward-only B200 kernels)")


class _WithBackward(torch.autograd.Function):
    """A forward kernel with a hand-written backward kernel: `bwd(saved_inputs, grad_out, needs_input_grad)`
    returns one gradient (or None) per input tensor.  Extra outputs (masks, indices) are non-differentiable."""

    @staticmethod
    def forward(ctx, fn, bwd, name, *tensors):
        ctx.bwd, ctx.op_name = bwd, name
        det = [t.detach() for t in tensors]
        out = fn(*det)
        ctx.save_for_backward(*det)
        if isinstance(out, tuple):
            ctx.mark_non_differentiable(*out[1:])
        return out

    @staticmethod
    def backward(ctx, *grads):
        res = ctx.bwd(ctx.saved_tensors, grads[0], ctx.needs_input_grad[3:])
        return (None, None, None) + tuple(res)


def differentiable(fn, bwd, name, *tensors):
    if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
        return _WithBackward.apply(fn, bwd, name, *tensors)
    return fn(*tensors)


def forward_only(fn, name, *tensors):
    if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
        return _NoBackward.apply(fn, name, *tensors)
    return fn(*tensors)


def patch_reference(*args, **kwargs):
    """Rebind the hot-path names of an already-imported reference checkout to these kernels (ofb200/overlay.py)."""
    from ofb200.overlay import patch_reference as _patch

    return _patch(*args, **kwargs)


def unpatch_reference():
    from ofb200.overlay import unpatch_reference as _unpatch

    return _unpatch()
