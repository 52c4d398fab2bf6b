"""The warp's sampling contract, kernel by kernel, element by element: every K1 forward variant (`ofb_warp_f32`: direct,
staged, row and TMA kernels, NCHW and channels_last, the fused pixel-flow normalize, nearest mode), the warp backward
(`ofb_warp_backward_f32`) and `bilinear_sampler`, in every padding mode x align_corners, at the source coordinates
where the tap arithmetic has edges.

All of them take their source coordinate from `ofb::warp_source` and their taps from `ofb::bilinear_taps`
(csrc/common.cuh), whose comment states the contract for non-finite and far coordinates:
  zeros       a non-finite (or far) source coordinate samples 0 (ATen's bilinear grid_sample gives NaN for NaN / inf)
  border      NaN and -inf clip to 0, +inf to size - 1
  reflection  every non-finite coordinate becomes 0
and the mask is 0 wherever a grid coordinate is not finite.

Coordinate kinds (flows built in pixels, then normalised as optical_flow.normalize does; every kind runs in every
padding x align_corners):
  int        integer pixel shifts in [-3, 3]
  half       half-pixel shifts
  edge       grid coordinates on -1 and +1 and source positions on the first and last pixel centre
  straddle   source positions whose two taps straddle each edge (-0.5, -0.25, size - 0.75, size - 0.5)
  far        +-1e3 px
  huge       +-1e9 and +-3e9 in normalised units
  nonfinite  NaN, +inf and -inf on x only, on y only and on both

Tolerances:
  mask                                    bit-exact against the oracle, every kind
  forward values, finite kinds            <= 1e-5 * max(1, |ref|_inf) against the oracle (nearest: exact)
  every forward variant                   bit-identical to the row kernel, every kind
  forward values, nonfinite kind          zeros: exactly 0; border / reflection: the oracle on a flow whose non-finite
                                          components are replaced by finite ones that clip to the same pixel, at the
                                          finite-kind tolerance (nearest: exact)
  backward, finite kinds                  d_frame <= 1e-5, d_flow <= 2e-5 * max(1, |ref|_inf) against autograd through
                                          oracle/torch_port.py (as test_gpu_parity.test_warp_backward_vs_oracle)
  backward, pinned cases                  d_flow bit-identical, d_frame <= 1e-5 * max(1, |ref|_inf) (its scatter-add
                                          order varies) against tests/golden/warp_contract.npz, recorded with the
                                          kernels before they shared bilinear_taps: the nonfinite kind, and reflection
                                          x huge, where ATen's CPU grid_sample reflects coordinates beyond ~1e9 px to
                                          other pixels than the fp32 reflection the kernels and the oracle share (its
                                          forward differs there too)
  bilinear_sampler                        mask bit-exact; values as the forward, against oracle.bilinear_sampler
"""
import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

PADS = ("zeros", "border", "reflection")
KINDS = ("int", "half", "edge", "straddle", "far", "huge", "nonfinite")
PINNED = [(p, ac, "nonfinite") for p in PADS for ac in (False, True)]
PINNED += [("reflection", ac, "huge") for ac in (False, True)]
BACKWARD = [(p, ac, k) for p in PADS for ac in (False, True) for k in KINDS if (p, ac, k) not in PINNED]
B, H, W = 2, 12, 16                       # W % 4 == 0: the TMA kernel runs too


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ofb200

    ofb200.load()


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().cpu().numpy()


def tol(ref, eps=1e-5):
    return eps * max(1.0, float(np.abs(ref).max()))


def maxabs(a, b):
    return float(np.max(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))))


def flow_mul(h, w):
    """optical_flow.normalize's factors (pixels -> normalised units)."""
    return np.float32(2.0 / max(w - 1, 1)), np.float32(2.0 / max(h - 1, 1))


def source_to_grid(ix, size, ac):
    """The grid coordinate whose un-normalised source position is ix (GridSampler.h:26-36, inverted in float64)."""
    ix = np.asarray(ix, np.float64)
    return 2.0 * ix / (size - 1) - 1.0 if ac else (2.0 * ix + 1.0) / size - 1.0


def make_flow(kind, ac, b=B, h=H, w=W, seed=0):
    """Pixel-unit flow (b, 2, h, w) float32 of one kind (module docstring)."""
    r = np.random.default_rng(seed)
    shape = (b, h, w)
    mx, my = flow_mul(h, w)
    if kind == "int":
        return r.integers(-3, 4, (b, 2, h, w)).astype(np.float32)
    if kind == "half":
        return (r.integers(-3, 3, (b, 2, h, w)) + 0.5).astype(np.float32)
    if kind == "far":
        return (np.where(r.random((b, 2, h, w)) < 0.5, -1e3, 1e3) + r.standard_normal((b, 2, h, w))).astype(np.float32)
    if kind == "huge":
        g = r.choice(np.array([1e9, -1e9, 3e9, -3e9, 0.0]), (b, 2, h, w))
        return (g / np.array([mx, my]).reshape(1, 2, 1, 1)).astype(np.float32)
    if kind in ("edge", "straddle"):
        flow = np.empty((b, 2, h, w), np.float32)
        for axis, n, m in ((0, w, mx), (1, h, my)):
            if kind == "edge":
                targets = np.concatenate([[-1.0, 1.0], source_to_grid([0.0, n - 1.0], n, ac)])
            else:
                targets = source_to_grid([-0.5, -0.25, n - 0.75, n - 0.5], n, ac)
            g = r.choice(targets, shape)
            lin = oracle.linspace(-1.0, 1.0, n).astype(np.float64)
            lin = lin[None, None, :] if axis == 0 else lin[None, :, None]
            flow[:, axis] = (g - lin) / m
        return flow
    assert kind == "nonfinite", kind
    flow = r.standard_normal((b, 2, h, w)).astype(np.float32)
    # pixel k: (k % 4) picks x only, y only, both or neither; the value cycles through NaN, +inf, -inf
    k = np.arange(b * h * w).reshape(shape)
    special = np.array([np.nan, np.inf, -np.inf], np.float32)
    val = special[(k // 4) % 3]
    valy = special[(k // 12) % 3]
    flow[:, 0] = np.where((k % 4 == 0) | (k % 4 == 2), val, flow[:, 0])
    flow[:, 1] = np.where((k % 4 == 1) | (k % 4 == 2), valy, flow[:, 1])
    return flow


def contract_substitute(flow_n, pad, ac):
    """The normalised flow with each non-finite component replaced by a finite one that the padding clips to the same
    source pixel (common.cuh): border -1e9 for NaN / -inf and +1e9 for +inf; reflection a grid coordinate of about -1
    (source position about 0 with align_corners, about -0.5 without: both land on pixel 0)."""
    sub = flow_n.copy()
    for axis, n in ((0, sub.shape[3]), (1, sub.shape[2])):
        f = sub[:, axis]
        lin = oracle.linspace(-1.0, 1.0, n)
        lin = np.broadcast_to(lin[None, None, :] if axis == 0 else lin[None, :, None], f.shape)
        bad = ~np.isfinite(f)
        if pad == "border":
            f[bad & (f > 0)] = 1e9
            f[bad & ~(f > 0)] = -1e9
        else:
            assert pad == "reflection"
            f[bad] = (np.float32(-1.0) - lin)[bad]
    return sub


def nonfinite_pixels(flow):
    return ~np.isfinite(flow).all(axis=1)             # (b, h, w)


def expected(frame, flow_n, pad, ac, kind, mode="bilinear"):
    """What the contract says `warp` returns: the oracle on finite kinds, the substitution / zero rule on the other."""
    if kind != "nonfinite":
        return oracle.warp(frame, flow_n, mode=mode, padding_mode=pad, align_corners=ac)
    if pad == "zeros":
        ref = oracle.warp(frame, np.where(np.isfinite(flow_n), flow_n, 0).astype(np.float32), mode=mode,
                          padding_mode=pad, align_corners=ac)
        ref[np.broadcast_to(nonfinite_pixels(flow_n)[:, None], ref.shape)] = 0.0
        return ref
    return oracle.warp(frame, contract_substitute(flow_n, pad, ac), mode=mode, padding_mode=pad, align_corners=ac)


def check_values(out, ref, kind, exact=False):
    assert np.isfinite(out).all()
    if exact or (kind == "nonfinite" and not np.any(ref)):
        assert np.array_equal(out, ref)
    else:
        assert maxabs(out, ref) <= tol(ref)


# =============================================================================== forward
def warp_variants(w):
    return (1, 2, 3, 4) if w % 4 == 0 else (1, 2, 3)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("ac", [False, True])
@pytest.mark.parametrize("pad", PADS)
def test_warp_forward_contract(pad, ac, kind):
    """Every bilinear variant, channels_last (C = 3: scalar path, C = 8: float4 path), the fused pixel-flow normalize
    and nearest mode, against the oracle / the contract, and bit-identical to the row kernel."""
    from optical_flow import warp

    r = np.random.default_rng(7)
    flow_px = make_flow(kind, ac)
    flow_n = oracle.normalize(flow_px).astype(np.float32)
    frame = (r.random((B, 8, H, W)) - 0.5).astype(np.float32)
    ref = expected(frame, flow_n, pad, ac, kind)
    _, ref_mask = oracle.warp(frame, flow_n, padding_mode=pad, align_corners=ac, return_mask=True)

    rows = None
    for variant in (3,) + tuple(v for v in warp_variants(W) if v != 3):
        out, mask = warp(T(frame), T(flow_n), padding_mode=pad, align_corners=ac, return_mask=True, variant=variant)
        out = N(out)
        assert np.array_equal(N(mask).astype(np.uint8), ref_mask), variant
        check_values(out, ref, kind)
        if rows is None:
            rows = out
            if kind == "nonfinite" and pad == "zeros":
                assert not np.any(out[np.broadcast_to(nonfinite_pixels(flow_n)[:, None], out.shape)])
        assert np.array_equal(out, rows), variant
    for c in (3, 8):
        cl = T(frame[:, :c]).contiguous(memory_format=torch.channels_last)
        assert not cl.is_contiguous()
        out = N(warp(cl, T(flow_n), padding_mode=pad, align_corners=ac))
        assert np.array_equal(out, rows[:, :c]), c
    fused, fmask = warp(T(frame), T(flow_px), padding_mode=pad, align_corners=ac, return_mask=True, pixel_flow=True)
    assert np.array_equal(N(fused), rows) and np.array_equal(N(fmask).astype(np.uint8), ref_mask)

    near = N(warp(T(frame), T(flow_n), mode="nearest", padding_mode=pad, align_corners=ac))
    check_values(near, expected(frame, flow_n, pad, ac, kind, mode="nearest"), kind, exact=True)


# =============================================================================== backward
def warp_backward(frame, flow_n, weight, pad, ac):
    from optical_flow import warp

    gf, gw = T(frame).requires_grad_(True), T(flow_n).requires_grad_(True)
    (warp(gf, gw, padding_mode=pad, align_corners=ac) * T(weight)).sum().backward()
    return N(gf.grad), N(gw.grad)


def backward_inputs(kind, ac):
    r = np.random.default_rng(11)
    frame = r.random((B, 3, H, W), dtype=np.float32)
    weight = r.standard_normal((B, 3, H, W)).astype(np.float32)
    return frame, oracle.normalize(make_flow(kind, ac, seed=3)).astype(np.float32), weight


@pytest.mark.parametrize("pad,ac,kind", BACKWARD)
def test_warp_backward_contract(pad, ac, kind):
    from oracle import torch_port as tp

    frame, flow_n, weight = backward_inputs(kind, ac)
    cf, cw = torch.from_numpy(frame).requires_grad_(True), torch.from_numpy(flow_n).requires_grad_(True)
    (tp.warp(cf, cw, padding_mode=pad, align_corners=ac) * torch.from_numpy(weight)).sum().backward()
    want_f, want_w = cf.grad.numpy(), cw.grad.numpy()
    got_f, got_w = warp_backward(frame, flow_n, weight, pad, ac)
    assert maxabs(got_f, want_f) <= tol(want_f) and maxabs(got_w, want_w) <= tol(want_w, 2e-5)


@pytest.mark.parametrize("pad,ac,kind", PINNED)
def test_warp_backward_pinned(golden, pad, ac, kind):
    """Both gradients against the recorded result.  What it holds for non-finite flows: under zeros padding such a pixel
    adds nothing to d_frame and its d_flow is 0; under border / reflection a NaN coordinate (the backward's clip keeps
    NaN, as ATen's does) reaches no tap, and a clipped +-inf one scatters into the clipped taps."""
    frame, flow_n, weight = backward_inputs(kind, ac)
    got_f, got_w = warp_backward(frame, flow_n, weight, pad, ac)
    g = golden("warp_contract")
    want_f = g[f"dframe_{pad}_{int(ac)}_{kind}"]
    assert maxabs(got_f, want_f) <= tol(want_f)
    assert np.array_equal(got_w, g[f"dflow_{pad}_{int(ac)}_{kind}"])
    if kind == "nonfinite" and pad == "zeros":
        assert not np.any(got_w[np.broadcast_to(nonfinite_pixels(flow_n)[:, None], got_w.shape)])


# =============================================================================== bilinear_sampler
@pytest.mark.parametrize("kind", KINDS)
def test_bilinear_sampler_contract(kind):
    """bilinear_sampler (zeros padding, align_corners=True, pixel coordinates) on the same kinds: source positions
    base grid + flow."""
    from model.utils import bilinear_sampler

    r = np.random.default_rng(5)
    img = (r.random((B, 3, H, W)) - 0.5).astype(np.float32)
    coords = (oracle.coords_grid(B, H, W) + make_flow(kind, True, seed=9)).transpose(0, 2, 3, 1)
    coords = np.ascontiguousarray(coords, dtype=np.float32)
    ref, ref_mask = oracle.bilinear_sampler(img, coords, mask=True)
    out, mask = bilinear_sampler(T(img), T(coords), mask=True)
    out = N(out)
    assert np.array_equal(N(mask), ref_mask)
    if kind == "nonfinite":
        bad = np.broadcast_to(~np.isfinite(coords).all(axis=-1)[:, None], out.shape)
        assert np.array_equal(out[bad], np.zeros(int(bad.sum()), np.float32))
        out, ref = out[~bad], ref[~bad]
    check_values(out, ref, kind)
