"""The correlation lookup's half-precision output and gradient: `ofb_corr_lookup_to`, `ofb_corr_lookup_ondemand_to`,
`ofb_corr_lookup_backward`, `ofb_corr_lookup_coords_backward_from` and `CorrBlock(..., lookup_dtype=...)`.

Every check is bit-exact, against the fp32 kernels themselves:
  forward      the fp16 / bf16 output equals the fp32 output cast by ATen (`out_fp32.to(dtype)`, round to nearest even,
               fp16 beyond +-65504 -> inf) bit for bit, NaN at the same positions; indices and masks equal the fp32
               call's.  The kernels accumulate each sample in fp32 as for an fp32 output and round it once.
  backward     a gradient G representable in the 16-bit type, passed in 16 bits, gives the same bits as the fp32 kernels
               fed G: the kernels widen each element exactly and then run the fp32 arithmetic in the same order.
  autocast     a lookup -> Conv2d(324, 256, 1) -> ReLU -> sum under torch.autocast gives the same loss and gradients with
               lookup_dtype="autocast" as with the fp32 output that autocast casts, and two kernels fewer per lookup.
Coordinate kinds, pyramid packers and reference helpers come from test_lookup_contract.py.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_lookup_contract import (BWD_SHAPES, FWD_LAYOUTS, FWD_SHAPES, KINDS, OD_CASES, OFB_EINVAL,  # noqa: E402
                                  OFB_EUNSUPPORTED, OFB_OK, TORCH_DT, N, T, bits, check_padding, grad_pyramid,
                                  level_shapes_of, lookup_pyramid, make_coords, ondemand_block)

gpu = pytest.mark.gpu
HALF = {"fp16": torch.float16, "bf16": torch.bfloat16}


def dtype_code(dt):
    import ofb200

    return {torch.float32: ofb200.DTYPE_F32, torch.float16: ofb200.DTYPE_F16, torch.bfloat16: ofb200.DTYPE_BF16}[dt]


def assert_cast_equal(got, out32, what):
    """got (16-bit) == out32.to(got.dtype) bit for bit, NaN at the same positions (NaN payloads are not compared)."""
    want = out32.to(got.dtype)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), what
    assert torch.equal(bits(got)[~nan], bits(want)[~nan]), (what, int((bits(got) != bits(want))[~nan].sum()))


# =============================================================================== C ABI (CPU: every call is rejected)
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


BAD_DTYPES = (-1, 3, 4, 99)          # 3 = OFB_DTYPE_F64


def test_dtype_entry_points_validate_arguments_without_launch(lib):
    """Each dtype-aware entry point returns OFB_EINVAL for an unknown dtype (OFB_DTYPE_F64 included) and for null
    pointers; for every malformed pyramid descriptor, and for every descriptor variant the forward lookup and coordinate
    backward test against each other, each returns the code of its fp32 form, for all three dtypes.  Nothing launches."""
    import ofb200

    fake = ctypes.c_void_p(1 << 20)                      # never dereferenced: every call below returns before a launch

    def pyr(mode=1, dtype=ofb200.DTYPE_F32, base=1 << 20):
        p = ofb200.Pyramid()
        elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
        assert lib.ofb_pyramid_layout(16, 24, 4, mode, ctypes.byref(p), ctypes.byref(elems)) == 0
        for l in range(4):
            p.base[l] = base
        p.dtype = dtype
        return p

    def edit(**kw):
        def apply(p):
            for k, v in kw.items():
                if isinstance(v, tuple):
                    getattr(p, k)[v[0]] = v[1]
                else:
                    setattr(p, k, v)
            return p
        return apply

    # One function per entry point: (dtype-aware form, fp32 form).  Each call below is one the checks reject before a
    # launch; a call that passes them would launch on fake pointers, so entry points are called one at a time.
    def lookup(p, dt, b=1, h=16, w=24, radius=4, coords=fake, out=fake):
        r = ctypes.byref(p) if p is not None else None
        return (lib.ofb_corr_lookup_to(r, coords, out, dt, None, None, b, h, w, radius, None),
                lib.ofb_corr_lookup(r, coords, out, None, None, b, h, w, radius, None))

    def coords_bwd(p, dt, b=1, h=16, w=24, radius=4, coords=fake, d_out=fake, d_coords=fake):
        r = ctypes.byref(p) if p is not None else None
        return (lib.ofb_corr_lookup_coords_backward_from(r, coords, d_out, dt, d_coords, b, h, w, radius, None),
                lib.ofb_corr_lookup_coords_backward(r, coords, d_out, d_coords, b, h, w, radius, None))

    def pyr_bwd(p, dt, b=1, h=16, w=24, radius=4, coords=fake, d_out=fake):
        r = ctypes.byref(p) if p is not None else None
        return (lib.ofb_corr_lookup_backward(r, coords, d_out, dt, b, h, w, radius, None),
                lib.ofb_corr_lookup_backward_f32(r, coords, d_out, b, h, w, radius, None))

    def ondemand(dt, c=64, levels=4, radius=4, f1=1 << 20, lvl=(1 << 20,) * 4, h=16, w=24, out=fake, b=1):
        ptrs = (ctypes.c_void_p * 4)(*lvl)
        return (lib.ofb_corr_lookup_ondemand_to(ctypes.c_void_p(f1), ptrs, fake, out, dt, b, c, h, w, levels, radius, None),
                lib.ofb_corr_lookup_ondemand(ctypes.c_void_p(f1), ptrs, fake, out, b, c, h, w, levels, radius, None))

    before = lib.ofb_launch_count()
    good = (ofb200.DTYPE_F32, ofb200.DTYPE_F16, ofb200.DTYPE_BF16)
    # unknown dtypes: rejected first, also for arguments the fp32 form would launch and for an empty call
    for dt in BAD_DTYPES:
        for b in (0, 1):
            r = ctypes.byref(pyr())
            ptrs = (ctypes.c_void_p * 4)(*((1 << 20,) * 4))
            assert lib.ofb_corr_lookup_to(r, fake, fake, dt, None, None, b, 16, 24, 4, None) == OFB_EINVAL, (dt, b)
            assert lib.ofb_corr_lookup_coords_backward_from(r, fake, fake, dt, fake, b, 16, 24, 4, None) == OFB_EINVAL
            assert lib.ofb_corr_lookup_backward(r, fake, fake, dt, b, 16, 24, 4, None) == OFB_EINVAL, (dt, b)
            assert lib.ofb_corr_lookup_ondemand_to(fake, ptrs, fake, fake, dt, b, 64, 16, 24, 4, 4, None) == OFB_EINVAL
    # null pointers
    for dt in good:
        for codes in (lookup(None, dt), lookup(pyr(), dt, coords=None), lookup(pyr(), dt, out=None),
                      coords_bwd(None, dt), coords_bwd(pyr(), dt, coords=None), coords_bwd(pyr(), dt, d_out=None),
                      coords_bwd(pyr(), dt, d_coords=None),
                      pyr_bwd(None, dt), pyr_bwd(pyr(), dt, coords=None), pyr_bwd(pyr(), dt, d_out=None),
                      ondemand(dt, out=None), ondemand(dt, f1=0)):
            assert codes == (OFB_EINVAL, OFB_EINVAL), (dt, codes)
        assert lib.ofb_corr_lookup_ondemand_to(fake, None, fake, fake, dt, 1, 64, 16, 24, 4, 4, None) == OFB_EINVAL
    # malformed descriptors: the code of the fp32 form (OFB_EINVAL), at every entry point and dtype
    broken = [edit(levels=0), edit(levels=5), edit(dtype=3), edit(dtype=-1), edit(layout=3), edit(layout=-1),
              edit(base=(2, None)), edit(lvl_h=(1, 0)), edit(lvl_w=(3, 0)), edit(row_pitch=(2, 5)),
              edit(q_stride=(1, 64))]
    for pdt in (ofb200.DTYPE_F32, ofb200.DTYPE_BF16):
        for k, fault in enumerate(broken):
            for dt in good:
                for fn in (lookup, coords_bwd, pyr_bwd):
                    assert fn(fault(pyr(3, pdt)), dt) == (OFB_EINVAL, OFB_EINVAL), (pdt, k, dt, fn.__name__)
    # descriptors the two readers accept or refuse for their own reasons (test_lookup_contract's variants), with
    # B * h * w = 2^36 queries: more blocks than either launch takes, so an accepted one is refused there
    variants = [edit(), edit(base=(1, (1 << 20) + 2)), edit(base=(2, (1 << 20) + 4)), edit(row_pitch=(1, 13)),
                edit(row_pitch=(1, 14)), edit(lvl_w=(0, 70000), row_pitch=(0, 70000)), edit(q_stride=(3, 64))]
    for mode in range(4):
        for pdt in good:
            for radius in range(5):
                for k, variant in enumerate(variants):
                    for dt in good:
                        for fn in (lookup, coords_bwd):
                            new, old = fn(variant(pyr(mode, pdt)), dt, b=65536, h=1024, w=1024, radius=radius)
                            assert new == old, (mode, pdt, radius, k, dt, fn.__name__, new, old)
    # the on-demand lookup's own checks
    cases = [{"c": 96}, {"radius": 5}, {"levels": 0}, {"levels": 5}, {"f1": (1 << 20) + 8},
             {"lvl": (1 << 20, 1 << 20, (1 << 20) + 4, 1 << 20)}, {"lvl": (1 << 20, None, 1 << 20, 1 << 20)}, {"h": 4},
             {"w": 7}, {"b": 0}]
    for dt in good:
        for kw in cases:
            new, old = ondemand(dt, **kw)
            assert new == old, (dt, kw, new, old)
    assert lib.ofb_launch_count() == before


# =============================================================================== forward (GPU)
def run_lookup_to(pyr, coords_d, radius, dt):
    """ofb_corr_lookup_to with index and mask outputs -> (rc, out, idx, valid)."""
    import ofb200

    b, _, h, w = coords_d.shape
    d, lv = 2 * radius + 1, pyr.levels
    out = torch.full((b, lv * d * d, h, w), float("nan"), dtype=dt, device="cuda")
    idx = torch.full((b * h * w, lv, 2, d), -7, dtype=torch.int32, device="cuda")
    valid = torch.full((b * h * w, lv, d * d), 7, dtype=torch.uint8, device="cuda")
    rc = ofb200.load().ofb_corr_lookup_to(ctypes.byref(pyr), ofb200.ptr(coords_d), ofb200.ptr(out), dtype_code(dt),
                                          ofb200.ptr(idx), ofb200.ptr(valid), b, h, w, radius, ofb200.stream_ptr())
    return rc, out, idx, valid


@gpu
@pytest.mark.parametrize("shape", FWD_SHAPES)
@pytest.mark.parametrize("pyr_dtype", ["fp32", "bf16", "fp16"])
def test_lookup_forward_half_output_is_the_cast_fp32_output(cuda_lib, pyr_dtype, shape):
    """ofb_corr_lookup_to on every pyramid layout of test_lookup_contract (padded rows, rows of pitch = 2 mod 8, both
    8x4-blocked layouts), radius 0-4, 1-4 levels, every coordinate kind: the fp16 and bf16 outputs are the fp32 output
    cast to that dtype, bit for bit; indices and masks equal the fp32 call's.  One query in five has level values scaled
    by 2e4, so that (except on an fp16 pyramid, which cannot hold them) fp16 outputs beyond +-65504 become inf.  Where
    the forward has no kernel (blocked layouts with fp32 or radius <= 2) every output dtype gets OFB_EUNSUPPORTED."""
    b, h, w = shape
    tdt = TORCH_DT[pyr_dtype]
    q = b * h * w
    r = np.random.default_rng(2000 + h)
    shapes = level_shapes_of(h, w, 4)
    scale = np.where(np.arange(q) % 5 == 0, 2e4, 8.0).astype(np.float32)[:, None, None, None]
    levels = []
    for hl, wl in shapes:
        lv = (scale * r.standard_normal((q, 1, hl, wl))).astype(np.float32)
        if tdt == torch.float16:
            lv = np.clip(lv, -6e4, 6e4)
        levels.append(T(lv).to(tdt).float().cpu().numpy())
    pyrs = {layout: lookup_pyramid(levels, tdt, layout, b, h, w) for layout in FWD_LAYOUTS}
    overflow = 0
    for radius in range(5):
        for kind in KINDS:
            coords_d = T(make_coords(kind, b, h, w, 2010 + radius))
            for layout, (pyr, _) in pyrs.items():
                unsupported = layout.startswith(("block", "qminor")) and (pyr_dtype == "fp32" or radius <= 2)
                for nl in range(1, 5):
                    pyr.levels = nl
                    what = (kind, radius, layout, nl)
                    rc, out32, idx32, valid32 = run_lookup_to(pyr, coords_d, radius, torch.float32)
                    if unsupported:
                        assert rc == OFB_EUNSUPPORTED, what
                    for name, dt in HALF.items():
                        rc16, out, idx, valid = run_lookup_to(pyr, coords_d, radius, dt)
                        assert rc16 == rc, (what, name)
                        if rc != OFB_OK:
                            continue
                        assert out.dtype == dt
                        assert_cast_equal(out, out32, (what, name))
                        assert torch.equal(idx, idx32) and torch.equal(valid, valid32), (what, name)
                    if rc == OFB_OK:
                        overflow += int((out32.abs() > 65504).sum())
                pyr.levels = 4
    assert (overflow > 0) == (pyr_dtype != "fp16"), overflow


@gpu
@pytest.mark.parametrize("c,shape", OD_CASES[:3])
def test_ondemand_half_output_is_the_cast_fp32_output(cuda_lib, c, shape):
    """ofb_corr_lookup_ondemand_to at C = 64 / 128 / 256, radius 0-4, 1-4 levels, every coordinate kind: the fp16 and
    bf16 outputs are the fp32 output cast to that dtype, bit for bit."""
    import ofb200

    b, h, w = shape
    _, _, (a_km, f2_levels) = ondemand_block(b, c, h, w, 2100 + c)
    lib = ofb200.load()
    ptrs = (ctypes.c_void_p * ofb200.MAX_LEVELS)(*[t.data_ptr() for t in f2_levels])

    def run(coords_d, levels, radius, dt):
        out = torch.full((b, levels * (2 * radius + 1) ** 2, h, w), float("nan"), dtype=dt, device="cuda")
        rc = lib.ofb_corr_lookup_ondemand_to(ofb200.ptr(a_km), ptrs, ofb200.ptr(coords_d), ofb200.ptr(out),
                                             dtype_code(dt), b, c, h, w, levels, radius, ofb200.stream_ptr())
        assert rc == OFB_OK
        return out

    for radius in range(5):
        for kind in KINDS:
            coords_d = T(make_coords(kind, b, h, w, 2110 + radius))
            for levels in range(1, 5):
                out32 = run(coords_d, levels, radius, torch.float32)
                for name, dt in HALF.items():
                    assert_cast_equal(run(coords_d, levels, radius, dt), out32, (kind, radius, levels, name))


# =============================================================================== backward (GPU)
def representable(g32, dt):
    """An fp32 gradient whose every element is a `dt` value, and the same values in `dt`."""
    g16 = g32.to(dt)
    return g16.float(), g16


def run_pyramid_backward(pyr, coords_d, d_out, radius):
    import ofb200

    b, _, h, w = coords_d.shape
    rc = ofb200.load().ofb_corr_lookup_backward(ctypes.byref(pyr), ofb200.ptr(coords_d), ofb200.ptr(d_out),
                                                dtype_code(d_out.dtype), b, h, w, radius, ofb200.stream_ptr())
    ofb200.check(rc, "ofb_corr_lookup_backward")


def same_pyramid_bits(keep_a, keep_b, what):
    for l, ((wa, _), (wb, _)) in enumerate(zip(keep_a, keep_b)):
        assert torch.equal(bits(wa), bits(wb)), (what, l)


@gpu
@pytest.mark.parametrize("radius", range(5))
@pytest.mark.parametrize("shape", BWD_SHAPES)
def test_pyramid_backward_half_gradient_is_exact(cuda_lib, shape, radius):
    """ofb_corr_lookup_backward with d_out in fp16 / bf16 gives the bits the fp32 kernel gives for the same values in
    fp32: 1-4 levels, tight and padded rows, every coordinate kind; padding columns and guard bands stay untouched."""
    b, h, w = shape
    q, d = b * h * w, 2 * radius + 1
    gen = torch.Generator(device="cuda").manual_seed(2200 + radius + h)
    for kind in KINDS:
        coords_d = T(make_coords(kind, b, h, w, 2210 + radius))
        g = 4 * torch.randn((b, 4 * d * d, h, w), device="cuda", generator=gen)
        for name, dt in HALF.items():
            g32, g16 = representable(g, dt)
            for levels in range(1, 5):
                for mode in (0, 1):
                    what = (kind, name, levels, mode)
                    ref_pyr, ref_keep = grad_pyramid(q, h, w, levels, mode, 0.0)
                    pyr, keep = grad_pyramid(q, h, w, levels, mode, 0.0)
                    run_pyramid_backward(ref_pyr, coords_d, g32[:, :levels * d * d].contiguous(), radius)
                    run_pyramid_backward(pyr, coords_d, g16[:, :levels * d * d].contiguous(), radius)
                    torch.cuda.synchronize()
                    check_padding(keep, pyr, what)
                    same_pyramid_bits(ref_keep, keep, what)


@gpu
@pytest.mark.parametrize("radius", [1, 4])
def test_pyramid_backward_half_gradient_accumulates_exactly(cuda_lib, radius):
    """Two backward calls with 16-bit gradients into a prefilled gradient pyramid (padded rows) leave the same bits as
    the two fp32 calls on the same values."""
    b, h, w, levels = 2, 19, 37, 4
    q, d = b * h * w, 2 * radius + 1
    r = np.random.default_rng(2300 + radius)
    prefill = [r.standard_normal((q, hl, wl)).astype(np.float32) for hl, wl in level_shapes_of(h, w, levels)]
    gen = torch.Generator(device="cuda").manual_seed(2310 + radius)
    for name, dt in HALF.items():
        ref_pyr, ref_keep = grad_pyramid(q, h, w, levels, 1, prefill)
        pyr, keep = grad_pyramid(q, h, w, levels, 1, prefill)
        for call, kind in enumerate(("int", "noise")):
            coords_d = T(make_coords(kind, b, h, w, 2320 + call))
            g32, g16 = representable(torch.randn((b, levels * d * d, h, w), device="cuda", generator=gen), dt)
            run_pyramid_backward(ref_pyr, coords_d, g32, radius)
            run_pyramid_backward(pyr, coords_d, g16, radius)
        torch.cuda.synchronize()
        check_padding(keep, pyr, name)
        same_pyramid_bits(ref_keep, keep, name)


@gpu
@pytest.mark.parametrize("shape", FWD_SHAPES)
@pytest.mark.parametrize("pyr_dtype", ["fp32", "bf16", "fp16"])
def test_coords_backward_half_gradient_is_exact(cuda_lib, pyr_dtype, shape):
    """ofb_corr_lookup_coords_backward_from with d_out in fp16 / bf16 gives the bits the fp32 kernel gives for the same
    values in fp32, on every pyramid layout the forward reads, radius 0-4, 1-4 levels, every coordinate kind."""
    import ofb200

    b, h, w = shape
    tdt = TORCH_DT[pyr_dtype]
    q = b * h * w
    r = np.random.default_rng(2400 + h)
    levels = [T(8 * r.standard_normal((q, 1, hl, wl)).astype(np.float32)).to(tdt).float().cpu().numpy()
              for hl, wl in level_shapes_of(h, w, 4)]
    pyrs = {layout: lookup_pyramid(levels, tdt, layout, b, h, w) for layout in FWD_LAYOUTS}
    gen = torch.Generator(device="cuda").manual_seed(2410 + h)

    def run(pyr, coords_d, g, radius):
        d_coords = torch.full((b, 2, h, w), float("nan"), device="cuda")
        rc = ofb200.load().ofb_corr_lookup_coords_backward_from(
            ctypes.byref(pyr), ofb200.ptr(coords_d), ofb200.ptr(g), dtype_code(g.dtype), ofb200.ptr(d_coords), b, h, w,
            radius, ofb200.stream_ptr())
        return rc, d_coords

    for radius in range(5):
        d = 2 * radius + 1
        for kind in KINDS:
            coords_d = T(make_coords(kind, b, h, w, 2420 + radius))
            g = torch.randn((b, 4 * d * d, h, w), device="cuda", generator=gen)
            for name, dt in HALF.items():
                g32, g16 = representable(g, dt)
                for nl in range(1, 5):
                    for layout, (pyr, _) in pyrs.items():
                        pyr.levels = nl
                        what = (kind, radius, name, nl, layout)
                        rc32, ref = run(pyr, coords_d, g32[:, :nl * d * d].contiguous(), radius)
                        rc, got = run(pyr, coords_d, g16[:, :nl * d * d].contiguous(), radius)
                        assert rc == rc32, what
                        if rc == OFB_OK:
                            assert torch.equal(bits(got), bits(ref)), what
                        pyr.levels = 4


# =============================================================================== CorrBlock (GPU)
def maps(b, c, h, w, seed, device="cuda", grad=False):
    gen = torch.Generator().manual_seed(seed)
    f1 = torch.randn((b, c, h, w), generator=gen).to(device).requires_grad_(grad)
    f2 = torch.randn((b, c, h, w), generator=gen).to(device).requires_grad_(grad)
    return f1, f2


@gpu
@pytest.mark.parametrize("on_demand", [False, True])
def test_corrblock_lookup_dtype_on_every_path(cuda_lib, on_demand):
    """lookup_dtype fp16 / bf16: the plain call, return_index=True (indices and masks as the fp32 call's), `out=` (which
    must have that dtype: an fp32 `out` raises, as a wrong shape does), and host coordinates all return the chosen dtype
    with the bits of the fp32 output cast to it.  On-demand blocks too (no return_index there)."""
    from ofb200.ops.corr import CorrBlock

    b, c, h, w, radius = 2, 64, 19, 37, 4
    d = 2 * radius + 1
    f1, f2 = maps(b, c, h, w, 2500)
    blk = CorrBlock(f1, f2, radius=radius, on_demand=on_demand)
    assert blk.lookup_dtype == torch.float32
    coords = T(make_coords("noise", b, h, w, 2510))
    ref = blk(coords)
    assert ref.dtype == torch.float32
    if not on_demand:
        _, ref_idx, ref_valid = blk(coords, return_index=True)
    for name, dt in HALF.items():
        blk.lookup_dtype = dt
        assert blk.out_dtype() == dt
        out = blk(coords)
        assert out.dtype == dt and out.is_cuda
        assert_cast_equal(out, ref, name)
        host = blk(coords.cpu())
        assert host.dtype == dt and not host.is_cuda
        assert torch.equal(bits(host), bits(out.cpu())), name
        buf = torch.empty((b, 4 * d * d, h, w), dtype=dt, device="cuda")
        assert blk(coords, out=buf) is buf
        assert torch.equal(bits(buf), bits(out)), name
        for wrong in (torch.empty((b, 4 * d * d, h, w), device="cuda"),
                      torch.empty((b, 4 * d * d, h, w + 1), dtype=dt, device="cuda")):
            with pytest.raises(RuntimeError, match="out must be a contiguous"):
                blk(coords, out=wrong)
        if not on_demand:
            got, idx, valid = blk(coords, return_index=True)
            assert got.dtype == dt and torch.equal(bits(got), bits(out))
            assert torch.equal(idx, ref_idx) and torch.equal(valid, ref_valid), name
    blk.lookup_dtype = torch.float32
    with pytest.raises(RuntimeError, match="out must be a contiguous"):
        blk(coords, out=torch.empty((b, 4 * d * d, h, w), dtype=torch.float16, device="cuda"))


@gpu
def test_corrblock_lookup_dtype_on_host_tensors(cuda_lib):
    """Host feature maps and host coordinates: the half-precision output arrives on the host with the device bits; with
    coordinates that require grad their gradient arrives there too, the same bits as from an fp32 output fed the same
    (fp16-representable) gradient."""
    from ofb200.ops.corr import CorrBlock

    b, c, h, w, radius = 1, 64, 24, 16, 4
    d = 2 * radius + 1
    f1, f2 = maps(b, c, h, w, 2600, device="cpu")
    g32, g16 = representable(torch.randn((b, 4 * d * d, h, w), generator=torch.Generator().manual_seed(2610)),
                             torch.float16)
    coords_np = make_coords("noise", b, h, w, 2620)
    res = {}
    for dt, g in ((torch.float32, g32), (torch.float16, g16)):
        blk = CorrBlock(f1, f2, radius=radius, lookup_dtype=dt)
        coords = torch.from_numpy(coords_np).requires_grad_(True)
        out = blk(coords)
        assert out.dtype == dt and out.device.type == "cpu"
        out.backward(g)
        assert coords.grad.device.type == "cpu"
        res[dt] = (out.detach(), coords.grad)
    assert_cast_equal(res[torch.float16][0], res[torch.float32][0], "host")
    assert torch.equal(res[torch.float16][1], res[torch.float32][1])


@gpu
def test_corrblock_lookup_dtype_autocast_and_environment(cuda_lib, monkeypatch):
    """"autocast" is fp32 outside CUDA autocast and the autocast dtype inside it; OFB200_LOOKUP_DTYPE sets the default
    (unset: fp32), the keyword overrides it; anything else is refused."""
    from ofb200.ops.corr import CorrBlock

    b, c, h, w = 1, 64, 16, 24
    f1, f2 = maps(b, c, h, w, 2700)
    coords = T(make_coords("half", b, h, w, 2710))
    blk = CorrBlock(f1, f2, lookup_dtype="autocast")
    assert blk(coords).dtype == torch.float32
    for dt in (torch.float16, torch.bfloat16):
        with torch.autocast("cuda", dtype=dt):
            assert blk.out_dtype() == dt
            assert blk(coords).dtype == dt
        with torch.autocast("cuda", dtype=dt, enabled=False):
            assert blk(coords).dtype == torch.float32
    monkeypatch.delenv("OFB200_LOOKUP_DTYPE", raising=False)
    assert CorrBlock(f1, f2).lookup_dtype == torch.float32
    for env, want in (("fp32", torch.float32), ("fp16", torch.float16), ("bf16", torch.bfloat16),
                      ("autocast", "autocast")):
        monkeypatch.setenv("OFB200_LOOKUP_DTYPE", env)
        blk = CorrBlock(f1, f2)
        assert blk.lookup_dtype == want, env
        assert blk(coords).dtype == (torch.float32 if want == "autocast" else want), env
        assert CorrBlock(f1, f2, lookup_dtype=torch.float32).lookup_dtype == torch.float32
    monkeypatch.setenv("OFB200_LOOKUP_DTYPE", "fp8")
    with pytest.raises(ValueError):
        CorrBlock(f1, f2)
    monkeypatch.delenv("OFB200_LOOKUP_DTYPE")
    with pytest.raises(NotImplementedError):
        CorrBlock(f1, f2, lookup_dtype=torch.float64)


@gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_corrblock_half_output_pyramid_lifetime(cuda_lib, dt):
    """With a half-precision output and coordinates that do not require grad, the graph does not keep the stored
    pyramid: dropping the block frees it at once; the feature-map gradient still arrives."""
    from ofb200.ops.corr import CorrBlock

    b, c, h, w, radius = 2, 64, 19, 37, 4
    d = 2 * radius + 1
    f1, f2 = maps(b, c, h, w, 2800, grad=True)
    blk = CorrBlock(f1, f2, radius=radius, lookup_dtype=dt)
    pyr_bytes = sum(t.numel() * t.element_size() for t in blk._buffers)
    out = blk(T(make_coords("noise", b, h, w, 2810)))
    assert out.dtype == dt and out.grad_fn is not None
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    del blk
    assert before - torch.cuda.memory_allocated() >= pyr_bytes
    (out.float() * torch.randn((b, 4 * d * d, h, w), device="cuda")).sum().backward()
    assert f1.grad is not None and f2.grad is not None


# =============================================================================== autocast equivalence (GPU)
def motion_step(conv, f1, f2, coords, lookup_dtype, dt, iters):
    """Under autocast(dt): a CorrBlock built from f1, f2, then `iters` lookups -> conv -> ReLU -> sum, summed; backward.
    Returns the loss, the gradients, and (forward, backward) counts of CUDA kernels (torch.profiler) and of library
    launches."""
    import ofb200
    from ofb200.ops.corr import CorrBlock
    from torch.profiler import ProfilerActivity, profile

    def cuda_kernels(prof):
        return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)

    for t in (f1, f2, coords, conv.weight, conv.bias):
        t.grad = None
    with torch.autocast("cuda", dtype=dt):
        blk = CorrBlock(f1, f2, radius=4, lookup_dtype=lookup_dtype)
        torch.cuda.synchronize()
        n0 = ofb200.launch_count()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as fwd:
            loss = sum(torch.relu(conv(blk(coords + 0.37 * k))).sum() for k in range(iters))
            torch.cuda.synchronize()
    n1 = ofb200.launch_count()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as bwd:
        loss.backward()
        torch.cuda.synchronize()
    n2 = ofb200.launch_count()
    grads = [t.grad.clone() for t in (f1, f2, coords, conv.weight, conv.bias)]
    return loss.detach(), grads, (cuda_kernels(fwd), cuda_kernels(bwd)), (n1 - n0, n2 - n1)


@gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_autocast_lookup_is_what_convc1_receives(cuda_lib, dt):
    """The promise of lookup_dtype="autocast": a lookup -> Conv2d(324, 256, 1) -> ReLU -> sum under torch.autocast, with
    fp32 feature maps and coordinates that require grad, gives the same loss and the same gradients of fmap1, fmap2,
    the coordinates and the conv's weight and bias, bit for bit, as the fp32 output autocast casts; it runs one CUDA
    kernel fewer per lookup forward (the cast) and one fewer backward (the cast of the gradient), with the same number
    of library launches."""
    b, c, h, w, iters = 2, 64, 19, 37, 3
    torch.manual_seed(2900)
    conv = torch.nn.Conv2d(324, 256, 1).cuda()
    f1, f2 = maps(b, c, h, w, 2910, grad=True)
    coords = T(make_coords("noise", b, h, w, 2920)).requires_grad_(True)
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        for mode in (torch.float32, "autocast"):                     # warm-up: module loads, cuDNN plans
            motion_step(conv, f1, f2, coords, mode, dt, iters)
        ref = motion_step(conv, f1, f2, coords, torch.float32, dt, iters)
        got = motion_step(conv, f1, f2, coords, "autocast", dt, iters)
    finally:
        torch.backends.cudnn.deterministic = det
    assert torch.equal(ref[0], got[0]), (float(ref[0]), float(got[0]))
    for name, a, g in zip(("fmap1", "fmap2", "coords", "weight", "bias"), ref[1], got[1]):
        assert a.dtype == g.dtype and torch.equal(a, g), name
    assert ref[2][0] - got[2][0] == iters, (ref[2], got[2])
    assert ref[2][1] - got[2][1] == iters, (ref[2], got[2])
    assert ref[3] == got[3], (ref[3], got[3])
