"""The correlation lookup's gradient with respect to its coordinates (`ofb_corr_lookup_coords_backward`, and
`CorrBlock.__call__` when the coordinates require grad), element by element against float64 references.

The reference's lookup (CorrBlock.__call__ + bilinear_sampler, corr.py:56-77, utils.py:64-80) is grid_sample, so
autograd gives the coordinates ATen's d grid: for level l, window cell (i, j) with the replayed taps (x0, wx0, wx1),
(y0, wy0, wy1) of `test_lookup_contract.replay_taps` and v the level value (0 outside the image)
    gx_ij = wy0 (v(y0, x0+1) - v(y0, x0)) + wy1 (v(y0+1, x0+1) - v(y0+1, x0))
    gy_ij = wx0 (v(y0+1, x0) - v(y0, x0)) + wx1 (v(y0+1, x0+1) - v(y0, x0+1))
    d coords = sum_l 2^-l sum_ij d_out[l, i, j] (gx_ij, gy_ij)
`coords_grad_f64` evaluates this in float64 from the fp32 floors and weights; A is the same sum over
|d_out| w (|v_a| + |v_b|), one term per difference w (v_b - v_a).  A sample with a tap outside the floor guard
contributes 0 (such a tap puts every tap of its axis outside the image; the weights may be NaN).

Bound (u = 2^-24).  Every intermediate the kernel rounds is a partial sum of terms each bounded by its share of A:
  per window row and tap, the difference v_b - v_a or the horizontal sample wx0 v_a + wx1 v_b (<= 2 roundings); per
  sample row using the window row, the D <= 9 products with d_out summed (9 roundings), then scaled by wy or +-1 and
  added to the row's sum (<= 3 samples: 3 roundings); the D + 2 <= 11 rows summed (11 roundings); <= 4 levels summed
  (3 roundings), the 2^-l scale exact.  That is <= 28 roundings, each adding at most u times a quantity <= A:
  28 u A = 1.7e-6 A.
The reference's own fp32 path (ATen's gix / giy, the (W-1)/2 and 2/(W-1) chain factors, the window and level sums of
autograd) stays below the same order.  Tested: |got - ref| <= 1e-5 A per element; A == 0 gives exactly 0.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_lookup_contract import (FWD_LAYOUTS, FWD_SHAPES, KINDS, OFB_EALIGN, OFB_EINVAL, OFB_EUNSUPPORTED,  # noqa: E402
                                  OFB_OK, REPLAY_GEOMS, TORCH_DT, N, T, dead_queries, in_guard, level_shapes_of,
                                  level_taps, lookup_pyramid, make_coords)

from oracle import torch_port  # noqa: E402

gpu = pytest.mark.gpu
FINITE_KINDS = ("int", "half", "noise", "edge")     # kinds where the reference's grid_sample gradient is finite
TOL = 1e-5


# =============================================================================== reference (CPU)
def coords_grad_levels(levels, coords, d_out, radius):
    """Per level l: (grad, A), each (B, 2, h, w) float64 and already scaled by 2^-l.  levels: (Q, 1, h_l, w_l) float32
    arrays (the stored values); d_out (B, >= L*(2r+1)^2, h, w)."""
    b, _, h, w = coords.shape
    q, d = b * h * w, 2 * radius + 1
    lv = len(levels)
    g = d_out.reshape(b, -1, d, d, h * w)[:, :lv].transpose(0, 4, 1, 2, 3).reshape(q, lv, d, d).astype(np.float64)
    rows = np.arange(q)[:, None, None]
    out = []
    for l, lvl in enumerate(levels):
        hl, wl = lvl.shape[-2:]
        img = lvl.reshape(q, hl, wl).astype(np.float64)
        tx, ty = level_taps(coords, l, radius, hl, wl)
        ok = in_guard(tx[0]).all(1)[:, None, None] & in_guard(ty[0]).all(1)[:, None, None]   # (q, 1, 1)

        def v(dx, dy):
            with np.errstate(invalid="ignore"):
                xi, yi = tx[0] + np.float32(dx), ty[0] + np.float32(dy)
                inx, iny = (xi >= 0) & (xi < wl), (yi >= 0) & (yi < hl)
            xi = np.where(inx, xi, 0).astype(np.int64)
            yi = np.where(iny, yi, 0).astype(np.int64)
            val = img[rows, yi[:, None, :], xi[:, :, None]]                                     # (q, i, j)
            return np.where(inx[:, :, None] & iny[:, None, :], val, 0.0)

        v00, v01, v10, v11 = v(0, 0), v(1, 0), v(0, 1), v(1, 1)                                 # v<dy><dx>
        f = lambda a: np.where(ok, a.astype(np.float64), 0.0)                                   # noqa: E731
        wx0, wx1 = f(tx[1][:, :, None]), f(tx[2][:, :, None])
        wy0, wy1 = f(ty[1][:, None, :]), f(ty[2][:, None, :])
        gl = np.where(ok, g[:, l], 0.0)
        s = 2.0 ** -l
        gx = (gl * (wy0 * (v01 - v00) + wy1 * (v11 - v10))).sum((1, 2)) * s
        gy = (gl * (wx0 * (v10 - v00) + wx1 * (v11 - v01))).sum((1, 2)) * s
        ax = (np.abs(gl) * (wy0 * (abs(v01) + abs(v00)) + wy1 * (abs(v11) + abs(v10)))).sum((1, 2)) * s
        ay = (np.abs(gl) * (wx0 * (abs(v10) + abs(v00)) + wx1 * (abs(v11) + abs(v01)))).sum((1, 2)) * s
        grad = np.stack([gx, gy]).reshape(2, b, h, w).transpose(1, 0, 2, 3)
        amag = np.stack([ax, ay]).reshape(2, b, h, w).transpose(1, 0, 2, 3)
        out.append((grad, amag))
    return out


def coords_grad_f64(levels, coords, d_out, radius):
    """d coords (B, 2, h, w) float64 of the lookup of `levels` at `coords` with output gradient d_out, and A (module
    docstring)."""
    parts = coords_grad_levels(levels, coords, d_out, radius)
    return sum(p[0] for p in parts), sum(p[1] for p in parts)


def autograd_coords_grad(levels, coords, d_out, radius):
    """coords.grad through oracle/torch_port.corr_lookup (the reference's ATen op sequence), fp32, on the CPU."""
    c = torch.tensor(coords, requires_grad=True)
    out = torch_port.corr_lookup([torch.tensor(x) for x in levels], c, radius=radius)
    out.backward(torch.tensor(np.ascontiguousarray(d_out[:, :out.shape[1]])))
    return c.grad.double().numpy()


def assert_within(got, ref, amag, what):
    err = np.abs(got - ref)
    bad = ~(err <= TOL * amag)                                   # NaN fails
    assert not bad.any(), (what, int(bad.sum()), float(err.max()), np.argwhere(bad)[:4].tolist())


@pytest.mark.parametrize("geom", REPLAY_GEOMS)
@pytest.mark.parametrize("radius", range(5))
def test_f64_reference_matches_torch_autograd(geom, radius):
    """coords_grad_f64 == autograd of the coordinates through torch_port.corr_lookup within 1e-5 A per element, for
    every finite coordinate kind and 1-4 levels.  At `int` (most taps on integers) this shows that the reference takes
    the one-sided derivative the replayed fp32 floors pick."""
    h, w = geom
    b, d = 2, 2 * radius + 1
    r = np.random.default_rng(900 + radius + h)
    levels = [r.standard_normal((b * h * w, 1, hl, wl)).astype(np.float32) for hl, wl in level_shapes_of(h, w, 4)]
    for kind in FINITE_KINDS:
        coords = make_coords(kind, b, h, w, 910 + radius)
        d_out = r.standard_normal((b, 4 * d * d, h, w)).astype(np.float32)
        for nl in range(1, 5):
            ref, amag = coords_grad_f64(levels[:nl], coords, d_out, radius)
            got = autograd_coords_grad(levels[:nl], coords, d_out, radius)
            assert_within(got, ref, amag, (kind, nl))


# =============================================================================== ABI (CPU: every call is rejected)
@pytest.fixture(scope="module")
def lib():
    import ofb200

    if not os.path.exists(ofb200.LIB_PATH):
        ofb200.build()
    return ofb200.load()


@pytest.fixture
def cuda_lib(lib):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return lib


def test_coords_backward_validates_arguments_without_launch(lib):
    """Zero-size calls return OK and bad arguments are rejected, all before any launch."""
    import ofb200

    fake = ctypes.c_void_p(1 << 20)                      # never dereferenced: every call below returns before a launch

    def pyr(levels=4, dtype=ofb200.DTYPE_F32, mode=1, base=1 << 20):
        p = ofb200.Pyramid()
        elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
        assert lib.ofb_pyramid_layout(16, 24, 4, mode, ctypes.byref(p), ctypes.byref(elems)) == 0
        for l in range(4):
            p.base[l] = base
        p.levels, p.dtype = levels, dtype
        return p

    def call(p, coords=fake, d_out=fake, d_coords=fake, b=1, h=16, w=24, radius=4):
        return lib.ofb_corr_lookup_coords_backward(ctypes.byref(p) if p is not None else None, coords, d_out, d_coords,
                                                   b, h, w, radius, None)

    before = lib.ofb_launch_count()
    assert call(None, b=0) == OFB_OK
    assert call(None) == OFB_EINVAL
    assert call(pyr(), coords=None) == OFB_EINVAL
    assert call(pyr(), d_out=None) == OFB_EINVAL
    assert call(pyr(), d_coords=None) == OFB_EINVAL
    assert call(pyr(), b=-1) == OFB_EINVAL
    assert call(pyr(), h=0) == OFB_EINVAL
    assert call(pyr(), w=0) == OFB_EINVAL
    assert call(pyr(), radius=5) == OFB_EUNSUPPORTED
    assert call(pyr(), radius=-1) == OFB_EUNSUPPORTED
    assert call(pyr(dtype=3)) == OFB_EINVAL
    p = pyr()
    p.layout = 3
    assert call(p) == OFB_EINVAL
    assert call(pyr(levels=0)) == OFB_EINVAL
    assert call(pyr(levels=5)) == OFB_EINVAL
    p = pyr()
    p.row_pitch[2] = p.lvl_w[2] - 1
    assert call(p) == OFB_EINVAL
    p = pyr()
    p.base[3] = None
    assert call(p) == OFB_EINVAL
    p = pyr()
    p.lvl_w[0] = p.row_pitch[0] = 70000
    assert call(p) == OFB_EUNSUPPORTED
    # 16-bit rows: 4-byte aligned bases and even pitches / strides (as ofb_corr_lookup)
    assert call(pyr(dtype=ofb200.DTYPE_BF16, base=(1 << 20) + 2)) == OFB_EALIGN
    p = pyr(dtype=ofb200.DTYPE_F16)
    p.row_pitch[1] = p.row_pitch[1] + 1
    assert call(p) == OFB_EALIGN
    # blocked layouts: 16-bit, radius 3 or 4, 16-byte aligned levels (where ofb_corr_lookup reads them)
    for mode in (2, 3):
        assert call(pyr(mode=mode)) == OFB_EUNSUPPORTED
        assert call(pyr(dtype=ofb200.DTYPE_BF16, mode=mode), radius=2) == OFB_EUNSUPPORTED
        assert call(pyr(dtype=ofb200.DTYPE_F16, mode=mode, base=(1 << 20) + 4)) == OFB_EUNSUPPORTED
    assert lib.ofb_launch_count() == before


# =============================================================================== C ABI (GPU)
def run_coords_backward(pyr, coords_d, d_out_d, radius):
    """ofb_corr_lookup_coords_backward into a NaN-prefilled buffer -> (rc, d_coords (B, 2, h, w) or None)."""
    import ofb200

    b, _, h, w = coords_d.shape
    d_coords = torch.full((b, 2, h, w), float("nan"), device="cuda")
    rc = ofb200.load().ofb_corr_lookup_coords_backward(ctypes.byref(pyr), ofb200.ptr(coords_d), ofb200.ptr(d_out_d),
                                                       ofb200.ptr(d_coords), b, h, w, radius, ofb200.stream_ptr())
    return rc, (N(d_coords) if rc == OFB_OK else None)


# FWD_SHAPES plus a level of height 1 (9 >> 3), which contributes 0
ABI_SHAPES = FWD_SHAPES + [(1, 9, 17)]


@gpu
@pytest.mark.parametrize("shape", ABI_SHAPES)
@pytest.mark.parametrize("dtype", ["fp32", "bf16", "fp16"])
def test_coords_backward_matches_float64(cuda_lib, dtype, shape):
    """ofb_corr_lookup_coords_backward on every pyramid layout ofb_corr_lookup reads (padding poisoned: NaN in fp32,
    the largest finite value in 16-bit), radius 0-4, 1-4 levels, every coordinate kind: |got - ref| <= 1e-5 A per
    element against coords_grad_f64 on the stored level values; A == 0 and dead queries give exactly 0; no NaN; a second
    run gives the same bits.  Blocked layouts where the forward has no kernel (fp32, radius <= 2) are rejected."""
    b, h, w = shape
    tdt = TORCH_DT[dtype]
    q = b * h * w
    r = np.random.default_rng(1000 + h)
    shapes = level_shapes_of(h, w, 4)
    levels = [T(8 * r.standard_normal((q, 1, hl, wl)).astype(np.float32)).to(tdt).float().cpu().numpy()
              for hl, wl in shapes]
    pyrs = {layout: lookup_pyramid(levels, tdt, layout, b, h, w) for layout in FWD_LAYOUTS}
    for radius in range(5):
        d = 2 * radius + 1
        for kind in KINDS:
            coords = make_coords(kind, b, h, w, 1010 + radius)
            d_out = r.standard_normal((b, 4 * d * d, h, w)).astype(np.float32)
            parts = coords_grad_levels(levels, coords, d_out, radius)
            coords_d = T(coords)
            for nl in range(1, 5):
                ref = sum(p[0] for p in parts[:nl])
                amag = sum(p[1] for p in parts[:nl])
                dead = dead_queries(coords, shapes[:nl], radius).reshape(b, h, w)
                d_sub = T(d_out[:, :nl * d * d])
                for layout, (pyr, _) in pyrs.items():
                    what = (kind, radius, layout, nl)
                    pyr.levels = nl
                    rc, got = run_coords_backward(pyr, coords_d, d_sub, radius)
                    if layout.startswith(("block", "qminor")) and (dtype == "fp32" or radius <= 2):
                        assert rc == OFB_EUNSUPPORTED, what
                        continue
                    assert rc == OFB_OK, what
                    assert not np.isnan(got).any(), what
                    assert_within(got.astype(np.float64), ref, amag, what)
                    assert not got[amag == 0].any(), what
                    assert not got.transpose(1, 0, 2, 3)[:, dead].any(), what
                    _, again = run_coords_backward(pyr, coords_d, d_sub, radius)
                    assert np.array_equal(got.view(np.int32), again.view(np.int32)), what
                for pyr, _ in pyrs.values():
                    pyr.levels = 4


# =============================================================================== CorrBlock (GPU)
def corr_block(b, c, h, w, seed, maps_grad=False, device="cuda", **kw):
    from ofb200.ops.corr import CorrBlock

    gen = torch.Generator().manual_seed(seed)
    f1 = torch.randn((b, c, h, w), generator=gen).to(device).requires_grad_(maps_grad)
    f2 = torch.randn((b, c, h, w), generator=gen).to(device).requires_grad_(maps_grad)
    return CorrBlock(f1, f2, **kw), f1, f2


def stored_levels(blk):
    return [N(v.float()) for v in blk.corr_pyramid]


@gpu
@pytest.mark.parametrize("radius", range(5))
def test_corrblock_fp32_coords_grad_matches_torch_autograd(cuda_lib, radius):
    """CorrBlock with an fp32 pyramid and feature maps that do not require grad: coords.grad equals autograd of the
    coordinates through torch_port.corr_lookup on the same stored levels within 1e-5 A.  The reference autograd runs on
    the CPU: on CUDA, ATen divides by the Python scalar W - 1 of utils.py:70 as a multiply by its reciprocal, which can
    move the un-normalised tap coordinate by an ulp -- the lookup's tap contract (and the forward's bit-exact indices)
    follows the reference's exact division, as ATen's CPU kernels compute it."""
    b, c, h, w = 2, 32, 19, 37
    d = 2 * radius + 1
    blk, _, _ = corr_block(b, c, h, w, 1100 + radius, radius=radius, pyramid_dtype=torch.float32)
    assert blk._handle is None
    levels = stored_levels(blk)
    gen = torch.Generator(device="cuda").manual_seed(1110 + radius)
    for kind in FINITE_KINDS:
        coords_np = make_coords(kind, b, h, w, 1120 + radius)
        coords = T(coords_np).requires_grad_(True)
        g = torch.randn((b, 4 * d * d, h, w), device="cuda", generator=gen)
        blk(coords).backward(g)
        want = autograd_coords_grad(levels, coords_np, N(g), radius)
        _, amag = coords_grad_f64(levels, coords_np, N(g), radius)
        assert_within(N(coords.grad).astype(np.float64), want, amag, kind)


@gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("radius", [2, 4])
def test_corrblock_half_pyramid_coords_grad(cuda_lib, dtype, radius):
    """The tensor-core pyramids (bf16 default, fp16; query-minor 8x4 blocks at radius 4, padded rows at radius 2):
    coords.grad matches coords_grad_f64 on the block's stored levels, every coordinate kind."""
    b, c, h, w = 2, 64, 19, 37
    d = 2 * radius + 1
    blk, _, _ = corr_block(b, c, h, w, 1200 + radius, radius=radius, pyramid_dtype=dtype)
    assert blk.builder == "tcgen05"
    levels = stored_levels(blk)
    gen = torch.Generator(device="cuda").manual_seed(1210 + radius)
    for kind in KINDS:
        coords_np = make_coords(kind, b, h, w, 1220 + radius)
        coords = T(coords_np).requires_grad_(True)
        g = torch.randn((b, 4 * d * d, h, w), device="cuda", generator=gen)
        blk(coords).backward(g)
        ref, amag = coords_grad_f64(levels, coords_np, N(g), radius)
        assert_within(N(coords.grad).astype(np.float64), ref, amag, kind)


def refinement_loop(blk, base, leaf, grads):
    """Three lookups at coordinates base + leaf + k * 0.37 (k = 0, 1, 2): sum_k <lookup_k, grads[k]>."""
    loss = 0.0
    for k, g in enumerate(grads):
        loss = loss + (blk(base + leaf + 0.37 * k) * g).sum()
    return loss


@gpu
@pytest.mark.parametrize("maps_grad", [False, True])
def test_corrblock_coords_grad_accumulates_over_iterations(cuda_lib, maps_grad):
    """A three-iteration loop whose coordinates depend on a leaf: leaf.grad is the sum of the three lookups' coordinate
    gradients (coords_grad_f64, 1e-5 of the summed A).  With feature maps that require grad, their gradients are the
    same bits as those of the same loop with detached coordinates."""
    b, c, h, w, radius = 2, 64, 19, 37, 4
    d = 2 * radius + 1
    base_np = make_coords("noise", b, h, w, 1300)
    base = T(base_np)
    gen = torch.Generator(device="cuda").manual_seed(1310)
    grads = [torch.randn((b, 4 * d * d, h, w), device="cuda", generator=gen) for _ in range(3)]
    leaf = torch.zeros((b, 2, h, w), device="cuda", requires_grad=True)
    blk, f1, f2 = corr_block(b, c, h, w, 1320, maps_grad=maps_grad, radius=radius)
    refinement_loop(blk, base, leaf, grads).backward()
    levels = stored_levels(blk)
    ref, amag = 0.0, 0.0
    for k, g in enumerate(grads):
        ck = (base + leaf.detach() + 0.37 * k).cpu().numpy()
        rk, ak = coords_grad_f64(levels, ck, N(g), radius)
        ref, amag = ref + rk, amag + ak
    assert_within(N(leaf.grad).astype(np.float64), ref, amag, maps_grad)
    if maps_grad:
        blk2, e1, e2 = corr_block(b, c, h, w, 1320, maps_grad=True, radius=radius)
        refinement_loop(blk2, base, leaf.detach(), grads).backward()
        assert torch.equal(f1.grad, e1.grad) and torch.equal(f2.grad, e2.grad)


@gpu
def test_corrblock_coords_grad_on_host_tensors(cuda_lib):
    """Host feature maps and host coordinates: coords.grad arrives on the host, the same bits as on the device."""
    b, c, h, w, radius = 1, 64, 24, 16, 4
    d = 2 * radius + 1
    coords_np = make_coords("noise", b, h, w, 1400)
    g = torch.randn((b, 4 * d * d, h, w), generator=torch.Generator().manual_seed(1410))
    grads = {}
    for device in ("cpu", "cuda"):
        blk, _, _ = corr_block(b, c, h, w, 1420, device=device, radius=radius)
        coords = torch.from_numpy(coords_np).to(device).requires_grad_(True)
        out = blk(coords)
        assert out.device.type == device
        out.backward(g.to(device))
        assert coords.grad is not None and coords.grad.device.type == device
        grads[device] = coords.grad.cpu()
    assert torch.equal(grads["cpu"], grads["cuda"])


@gpu
def test_corrblock_launches(cuda_lib):
    """Lookups whose coordinates do not require grad launch what they launched before (one kernel forward; with
    differentiable feature maps, one backward kernel per lookup); coordinates that require grad add exactly one
    backward launch per lookup and none forward."""
    import ofb200

    b, c, h, w, radius = 2, 64, 19, 37, 4
    d = 2 * radius + 1
    coords = T(make_coords("noise", b, h, w, 1500))
    g = torch.randn((b, 4 * d * d, h, w), device="cuda")

    blk, _, _ = corr_block(b, c, h, w, 1510, radius=radius)            # forward-only maps, plain coordinates
    n0 = ofb200.launch_count()
    out = blk(coords)
    assert ofb200.launch_count() - n0 == 1 and out.grad_fn is None

    counts = {}
    for coords_grad in (False, True):
        blk, _, _ = corr_block(b, c, h, w, 1510, maps_grad=True, radius=radius)
        x = coords.clone().requires_grad_(coords_grad)
        n0 = ofb200.launch_count()
        loss = (blk(x) * g).sum() + (blk(x + 0.5) * g).sum()
        n1 = ofb200.launch_count()
        loss.backward()
        torch.cuda.synchronize()
        counts[coords_grad] = (n1 - n0, ofb200.launch_count() - n1)
    assert counts[True][0] == counts[False][0] == 2
    assert counts[True][1] == counts[False][1] + 2


@gpu
def test_corrblock_pyramid_lifetime(cuda_lib):
    """With coordinates that do not require grad, the autograd graph does not keep the stored pyramid: dropping the
    block frees it at once, as before coordinates became differentiable.  A lookup whose coordinates require grad keeps
    it until its backward has run (that backward reads it), and the graph works without the block."""
    b, c, h, w, radius = 2, 64, 19, 37, 4
    d = 2 * radius + 1
    coords = T(make_coords("noise", b, h, w, 1600))
    g = torch.randn((b, 4 * d * d, h, w), device="cuda")
    for coords_grad in (False, True):
        blk, f1, _ = corr_block(b, c, h, w, 1610, maps_grad=True, radius=radius)
        pyr_bytes = sum(t.numel() * t.element_size() for t in blk._buffers)
        x = coords.clone().requires_grad_(coords_grad)
        out = blk(x)
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        del blk
        freed = before - torch.cuda.memory_allocated()
        if coords_grad:
            assert freed < pyr_bytes, (freed, pyr_bytes)
        else:
            assert freed >= pyr_bytes, (freed, pyr_bytes)
        (out * g).sum().backward()
        assert f1.grad is not None and (x.grad is not None) == coords_grad
        if coords_grad:
            torch.cuda.synchronize()
            before = torch.cuda.memory_allocated()
            del out
            assert before - torch.cuda.memory_allocated() >= pyr_bytes
