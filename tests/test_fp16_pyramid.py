"""The fp16 correlation pyramid: `CorrBlock(..., pyramid_dtype=torch.float16)`, the precision the reference stores its
pyramid in under `precision: 16` (methods/raft/config/train/default.yaml:20; autocast runs the matmul of corr.py:85 on
fp16 operands and avg_pool2d keeps fp16).

CPU part: the C ABI's argument checks for the new entry points and the OFB200_PYRAMID_DTYPE spellings.
GPU part:
  K2 fp16 (tcgen05)   every element within 1 fp16 ulp + 4e-6 * rms(level) of an fp32 recomputation from the builder's
                      own fp16 operands (levels 0-1 from fmap2, levels 2-3 from the fp16 4x4-pooled fmap2);
                      against the exact (fp64) pyramid rel-Frobenius <= 1e-3 and max-abs <= 5e-3 * rms per level;
                      against the reference's autocast chain computed with torch on the same GPU: level 0 <= 1e-4,
                      levels 1-3 <= 1.5e-3 rel-Frobenius
  CUDA-core fp16      level 0 within 1 ulp of the tcgen05 fp16 builder; also at a C the tcgen05 kernel rejects
  K3 on fp16          floor indices and validity masks equal to the fp32 / bf16 lookups' and the oracle's; values
                      <= 1e-5 * max(1, |ref|_inf) against the oracle on the stored levels read back in fp32
  training            feature-map gradients within rel-Frobenius 6e-3 of autograd through oracle/torch_port.py
  live RAFT           final flow within 2e-3 * |stock|_inf of the stock fp32 model (skipped without a reference checkout)
"""
import ctypes
import json
import math
import os

import numpy as np
import pytest
import torch

import oracle

gpu = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().cpu().numpy()


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


# =============================================================================== CPU: ABI and configuration
def test_fp16_entry_points_validate_arguments_without_launch(lib):
    import ofb200

    fake = ctypes.c_void_p(1 << 20)                      # never dereferenced: every call below is rejected first
    assert lib.ofb_corr_prep_to(None, ofb200.DTYPE_F32, fake, ofb200.DTYPE_F16, 1, 64, 8, 8, 1, 1.0, None) == -1
    assert lib.ofb_corr_prep_to(fake, ofb200.DTYPE_F32, fake, ofb200.DTYPE_F32, 1, 64, 8, 8, 1, 1.0, None) == -1
    assert lib.ofb_corr_prep_to(fake, ofb200.DTYPE_F64, fake, ofb200.DTYPE_F16, 1, 64, 8, 8, 1, 1.0, None) == -1
    assert lib.ofb_corr_prep_to(fake, ofb200.DTYPE_F32, fake, ofb200.DTYPE_F16, 1, 63, 8, 8, 1, 1.0, None) == -2
    assert lib.ofb_corr_prep_to(fake, ofb200.DTYPE_F32, fake, ofb200.DTYPE_F16, 1, 64, 8, 8, 3, 1.0, None) == -1
    assert lib.ofb_corr_prep_to(fake, ofb200.DTYPE_F32, fake, ofb200.DTYPE_F16, 0, 64, 8, 8, 1, 1.0, None) == 0
    pyr = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    assert lib.ofb_pyramid_layout(16, 16, 4, 3, ctypes.byref(pyr), ctypes.byref(elems)) == 0
    for lvl in range(4):
        pyr.base[lvl] = 1 << 20
    args = (fake, fake, fake, ctypes.byref(pyr), 1, 64, 16, 16, 0.125, 0, None)
    pyr.dtype = ofb200.DTYPE_BF16
    assert lib.ofb_corr_pyramid_f16(*args) == -2          # each builder writes its own dtype only
    pyr.dtype = ofb200.DTYPE_F16
    assert lib.ofb_corr_pyramid_bf16(*args) == -2
    assert lib.ofb_corr_pyramid_bf16_profile(*args[:-1], fake, None) == -2
    pyr.dtype = ofb200.DTYPE_F32
    assert lib.ofb_corr_pyramid_f16(*args) == -2
    pyr.dtype = ofb200.DTYPE_F16
    assert lib.ofb_corr_pyramid_f16(fake, fake, fake, ctypes.byref(pyr), 1, 48, 16, 16, 0.125, 0, None) == -2   # C % 64
    assert lib.ofb_corr_pyramid_f16(fake, fake, fake, ctypes.byref(pyr), 1, 64, 16, 16, 0.125, 4, None) == -1   # cta_group
    assert lib.ofb_corr_pyramid_f16(fake, fake, None, ctypes.byref(pyr), 1, 64, 16, 16, 0.125, 0, None) == -1   # f2q_km


def test_pyramid_dtype_environment_spellings(monkeypatch):
    from ofb200.ops.corr import _default_pyramid_dtype, operand_scale

    for name, want in [("fp16", torch.float16), ("F16", torch.float16), ("float16", torch.float16), ("half", torch.float16),
                       ("bf16", torch.bfloat16), ("fp32", torch.float32), ("float32", torch.float32)]:
        monkeypatch.setenv("OFB200_PYRAMID_DTYPE", name)
        assert _default_pyramid_dtype() == want, name
    monkeypatch.delenv("OFB200_PYRAMID_DTYPE")
    assert _default_pyramid_dtype() == torch.bfloat16                 # the default does not change
    assert operand_scale(256, torch.bfloat16) == 1.0 / 16 and operand_scale(256, torch.float16) == 1.0


# =============================================================================== GPU helpers
def ulp16(x):
    """fp16 unit in the last place at the magnitude of x (fp32 tensor): 2^(floor(log2|x|) - 10), subnormal spacing
    2^-24 below 2^-14."""
    _, e = torch.frexp(x.abs())
    return torch.ldexp(torch.ones_like(x), (e - 1).clamp(min=-14) - 10)


def pool_rows(rows, k):
    """Means of complete k x k blocks of each query's (h, w) row image."""
    if k == 1:
        return rows
    q, h, w = rows.shape
    hl, wl = h // k, w // k
    return rows[:, : hl * k, : wl * k].reshape(q, hl, k, wl, k).mean(dim=(2, 4))


def rows_from_km(a_km, b_km, q, h, w, scale, dtype=torch.float32):
    """Rows q of a_km . b_km^T * scale (K-major operands (B, n, C)) in `dtype`, as (len(q), h, w)."""
    b, n, c = a_km.shape
    out = torch.empty((q.numel(), b_km.shape[1]), dtype=dtype, device=a_km.device)
    qb, qp = q // n, q % n
    for bi in range(b):
        sel = (qb == bi).nonzero().flatten()
        if sel.numel():
            out[sel] = (a_km[bi, qp[sel]].to(dtype) @ b_km[bi].to(dtype).t()) * scale
    return out.view(-1, h, w)


def sample_queries(b, h, w, gen, count=1024):
    n = h * w
    corners = torch.tensor([0, w - 1, n - w, n - 1, b * n - 1], device="cuda")
    return torch.cat([corners, torch.randint(0, b * n, (count,), device="cuda", generator=gen)]).unique()


def relfro(got, want):
    return float((got.double() - want.double()).norm() / want.double().norm())


# cases: (shape, levels, cta_group, layout); layout "rows" = radius 2 (padded rows), "blocked" / "qminor" = radius 4
K2_CASES = [
    ((2, 256, 136, 240), 4, 0, "qminor"),       # the bench shape, auto launch mode
    ((16, 256, 47, 156), 4, 1, "qminor"),
    ((16, 256, 47, 156), 4, 2, "blocked"),
    ((16, 256, 47, 156), 4, 3, "qminor"),
    ((3, 64, 9, 35), 3, 1, "rows"),
    ((2, 128, 33, 50), 4, 2, "rows"),
    ((1, 192, 19, 37), 2, 3, "qminor"),
    ((2, 64, 24, 40), 1, 1, "blocked"),
    ((1, 128, 40, 72), 4, 2, "blocked"),
    ((2, 192, 23, 31), 3, 3, "qminor"),
]


# =============================================================================== K2 fp16
@gpu
@pytest.mark.parametrize("shape,levels,cta_group,layout", K2_CASES)
def test_fp16_pyramid_tcgen05(cuda_lib, shape, levels, cta_group, layout, monkeypatch):
    from ofb200.ops.corr import CorrBlock, prepare_operands

    b, c, h, w = shape
    monkeypatch.setenv("OFB200_PYRAMID_LAYOUT", "blocked" if layout == "blocked" else "qminor")
    gen = torch.Generator(device="cuda").manual_seed(1601 + c + h)
    f1 = torch.randn(shape, device="cuda", generator=gen)
    f2 = torch.randn(shape, device="cuda", generator=gen)
    blk = CorrBlock(f1, f2, num_levels=levels, radius=2 if layout == "rows" else 4, pyramid_dtype=torch.float16,
                    cta_group=cta_group)
    import ofb200

    assert blk.builder == "tcgen05" and blk._pyr.dtype == ofb200.DTYPE_F16
    assert blk._pyr.layout == {"rows": ofb200.LAYOUT_ROWS, "blocked": ofb200.LAYOUT_BLOCK8X4,
                               "qminor": ofb200.LAYOUT_QMINOR8X4}[layout]
    pyr = blk.corr_pyramid
    assert all(p.dtype == torch.float16 for p in pyr)
    assert [tuple(p.shape) for p in pyr] == [(b * h * w, 1, h >> l, w >> l) for l in range(levels)]

    # the builder's operands: fp16 maps, exact transposes (fmap1 is NOT pre-scaled), and the 4x4-pooled fmap2
    a_km, b_km, q_km = prepare_operands(f1, f2, levels, torch.float16)
    assert torch.equal(a_km, f1.half().reshape(b, c, h * w).transpose(1, 2))
    assert torch.equal(b_km, f2.half().reshape(b, c, h * w).transpose(1, 2))
    if q_km is not None:
        q_ref = torch.nn.functional.avg_pool2d(f2, 4).reshape(b, c, -1).transpose(1, 2)
        assert float((q_km.float() - q_ref).abs().max()) <= float(ulp16(q_ref).max())

    scale = 1.0 / math.sqrt(c)
    q = sample_queries(b, h, w, gen)
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref01 = rows_from_km(a_km, b_km, q, h, w, scale)                                  # fp32 from fp16 operands
        ref23 = rows_from_km(a_km, q_km, q, h >> 2, w >> 2, scale) if q_km is not None else None
        exact0 = rows_from_km(f1.reshape(b, c, -1).transpose(1, 2), f2.reshape(b, c, -1).transpose(1, 2), q, h, w,
                              scale, torch.float64)
        # the reference under autocast: fp16 matmul (fp32 accumulation), fp16 result, / sqrt(C) in fp16, fp16 avg_pool2d
        amp0 = (rows_from_km(a_km, b_km, q, h, w, 1.0).half() / math.sqrt(c)).unsqueeze(1)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    amp = [amp0]
    for _ in range(1, levels):
        amp.append(torch.nn.functional.avg_pool2d(amp[-1], 2))
    for lvl in range(levels):
        got = pyr[lvl][q, 0].float()
        want = pool_rows(ref01, 1 << lvl) if lvl < 2 else pool_rows(ref23, 1 << (lvl - 2))
        rms = float(want.pow(2).mean().sqrt())
        assert bool((got - want).abs().le(ulp16(want) + 4e-6 * rms).all()), (lvl, float((got - want).abs().max()))
        ex = pool_rows(exact0, 1 << lvl)
        ex_rms = float(ex.pow(2).mean().sqrt())
        assert relfro(got, ex) <= 1e-3, (lvl, relfro(got, ex))
        assert float((got.double() - ex).abs().max()) <= 5e-3 * ex_rms, lvl
        if math.log2(c) % 2 == 0:
            # C = 4^k, so 1/sqrt(C) is a power of two: rounding before or after the scale is the same, and level 0 IS
            # the reference's up to fp32 summation order; the pooled levels differ by its re-rounding of each level.
            # For other C the reference rounds twice (fp16 product, then fp16 quotient): ~3.5e-4 apart at level 0
            assert relfro(got, amp[lvl][:, 0].float()) <= (1e-4 if lvl == 0 else 1.5e-3), (lvl, relfro(got, amp[lvl][:, 0].float()))


@gpu
def test_fp16_pyramid_simt_builder(cuda_lib):
    """The CUDA-core builder writes fp16 pyramids too: level 0 within 1 ulp of the tcgen05 fp16 builder where both run
    (same fp16-rounded operands, fp32 accumulation), and it serves C the tcgen05 kernel rejects (C = 48), pooling each
    stored fp16 level like the reference's avg_pool2d under autocast."""
    from ofb200.ops.corr import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(1602)
    for shape in [(2, 64, 24, 40), (1, 256, 19, 37)]:
        b, c, h, w = shape
        f1 = torch.randn(shape, device="cuda", generator=gen)
        f2 = torch.randn(shape, device="cuda", generator=gen)
        tc = CorrBlock(f1, f2, num_levels=2, pyramid_dtype=torch.float16)
        simt = CorrBlock(f1, f2, num_levels=2, pyramid_dtype=torch.float16, builder="simt")
        assert tc.builder == "tcgen05" and simt.builder == "simt"
        a, s = tc.corr_pyramid[0].float(), simt.corr_pyramid[0].float()
        assert simt.corr_pyramid[0].dtype == torch.float16
        assert bool((a - s).abs().le(ulp16(a) + 1e-6 * float(a.pow(2).mean().sqrt())).all()), shape
        assert relfro(simt.corr_pyramid[1].float(), tc.corr_pyramid[1].float()) <= 1e-3
    b, c, h, w = 2, 48, 17, 29
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2, num_levels=3, radius=3, pyramid_dtype=torch.float16)
    assert blk.builder == "simt"
    f1h, f2h = f1.half().double().reshape(b, c, -1), f2.half().double().reshape(b, c, -1)
    l0 = (torch.bmm(f1h.transpose(1, 2), f2h) / math.sqrt(c)).reshape(-1, h, w)
    got0 = blk.corr_pyramid[0][:, 0].float()
    assert bool((got0 - l0).abs().le(ulp16(l0.float()) + 1e-6 * float(l0.pow(2).mean().sqrt())).all())
    stored = got0.half().unsqueeze(1)
    for lvl in range(1, 3):
        stored = torch.nn.functional.avg_pool2d(stored, 2)            # fp16 in, fp16 out: the reference's chain
        assert torch.equal(blk.corr_pyramid[lvl].cpu(), stored.cpu()), lvl
    out = blk(oracle_coords(b, h, w, 1603))
    ref = oracle.corr_lookup([N(p.float()) for p in blk.corr_pyramid], N(oracle_coords(b, h, w, 1603)), radius=3)
    assert float(np.abs(N(out) - ref).max()) <= 1e-5 * max(1.0, float(np.abs(ref).max()))


def oracle_coords(b, h, w, seed, sigma=3.0):
    r = np.random.default_rng(seed)
    return T((oracle.coords_grid(b, h, w) + sigma * r.standard_normal((b, 2, h, w))).astype(np.float32))


@gpu
def test_fp16_static_volume(cuda_lib):
    """CorrBlock.corr with an fp16 pyramid: the reference's torch.matmul under autocast returns fp16 (corr.py:85)."""
    from ofb200.ops.corr import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(1604)
    f1 = torch.randn((1, 64, 8, 24), device="cuda", generator=gen)
    f2 = torch.randn((1, 64, 8, 24), device="cuda", generator=gen)
    vol = CorrBlock.corr(f1.half(), f2.half(), pyramid_dtype=torch.float16)
    assert vol.shape == (1, 8, 24, 1, 8, 24) and vol.dtype == torch.float16
    want = torch.einsum("cp,cq->pq", f1.half().double()[0].reshape(64, -1), f2.half().double()[0].reshape(64, -1)) / 8.0
    got = vol.reshape(192, 192).float()
    assert bool((got - want).abs().le(ulp16(want.float()) + 1e-6).all())


# =============================================================================== K3 on fp16 pyramids
def _fp16_pyramid(levels, layout, pad_value=6.0e4):
    """Device fp16 pyramid of the given fp32 levels (fp16-representable) in `layout`; padding holds a large finite value
    (the lookup contract), so a padding element that leaked into a sample would show."""
    import ofb200
    from ofb200.ops.corr import level_buffer

    q = levels[0].shape[0]
    pyr = ofb200.Pyramid()
    pyr.levels = len(levels)
    pyr.dtype = ofb200.DTYPE_F16
    pyr.layout = {"rows": ofb200.LAYOUT_ROWS, "blocked": ofb200.LAYOUT_BLOCK8X4, "qminor": ofb200.LAYOUT_QMINOR8X4}[layout]
    bufs = []
    for l, lv in enumerate(levels):
        hl, wl = lv.shape[-2:]
        pitch, rows = ((wl + 15) & ~15, hl) if layout == "rows" else ((wl + 7) & ~7, (hl + 3) & ~3)
        img = torch.full((q, rows, pitch), pad_value, dtype=torch.float16, device="cuda")
        img[:, :hl, :wl] = T(lv[:, 0]).half()
        buf = level_buffer(img, pyr.layout)
        bufs.append(buf)
        pyr.base[l] = buf.data_ptr()
        pyr.q_stride[l] = 32 if layout == "qminor" else rows * pitch
        pyr.row_pitch[l] = pitch
        pyr.lvl_h[l] = hl
        pyr.lvl_w[l] = wl
    return pyr, bufs


def _float_pyramid(levels, dtype):
    import ofb200

    q = levels[0].shape[0]
    pyr = ofb200.Pyramid()
    pyr.levels = len(levels)
    pyr.dtype = ofb200.DTYPE_BF16 if dtype == torch.bfloat16 else ofb200.DTYPE_F32
    pyr.layout = ofb200.LAYOUT_ROWS
    bufs = []
    for l, lv in enumerate(levels):
        hl, wl = lv.shape[-2:]
        pitch = (wl + 15) & ~15
        buf = torch.zeros((q, hl, pitch), dtype=dtype, device="cuda")
        buf[:, :, :wl] = T(lv[:, 0]).to(dtype)
        bufs.append(buf)
        pyr.base[l] = buf.data_ptr()
        pyr.q_stride[l] = hl * pitch
        pyr.row_pitch[l] = pitch
        pyr.lvl_h[l] = hl
        pyr.lvl_w[l] = wl
    return pyr, bufs


def _run_lookup(pyr, coords, radius):
    import ofb200

    b, _, h, w = coords.shape
    d = 2 * radius + 1
    lv = pyr.levels
    out = torch.empty((b, lv * d * d, h, w), device="cuda")
    idx = torch.empty((b * h * w, lv, 2, d), dtype=torch.int32, device="cuda")
    valid = torch.empty((b * h * w, lv, d * d), dtype=torch.uint8, device="cuda")
    rc = ofb200.load().ofb_corr_lookup(ctypes.byref(pyr), ofb200.ptr(coords), ofb200.ptr(out), ofb200.ptr(idx),
                                       ofb200.ptr(valid), b, h, w, radius, ofb200.stream_ptr())
    ofb200.check(rc, "ofb_corr_lookup")
    return N(out), N(idx), N(valid)


LOOKUP_CASES = [(4, "qminor"), (4, "blocked"), (4, "rows"), (3, "qminor"), (3, "blocked"), (3, "rows"), (2, "rows")]


@gpu
@pytest.mark.parametrize("radius,layout", LOOKUP_CASES)
@pytest.mark.parametrize("hw", [(47, 156), (24, 40)])
def test_fp16_lookup_vs_oracle(cuda_lib, radius, layout, hw):
    """Radius 3 and 4 run the register-tile kernel, radius 2 the generic kernel.  Integer, sub-pixel, far, half-pixel,
    border-hanging and non-finite coordinates."""
    h, w = hw
    b = 1
    r = np.random.default_rng(1605)
    q = b * h * w
    levels = [(8 * r.standard_normal((q, 1, h >> l, w >> l))).astype(np.float16).astype(np.float32) for l in range(4)]
    pyr, bufs = _fp16_pyramid(levels, layout)
    p32, b32 = _float_pyramid(levels, torch.float32)
    pbf, bbf = _float_pyramid([oracle.round_bf16(lv) for lv in levels], torch.bfloat16)
    grid = oracle.coords_grid(b, h, w)
    for kind in ("int", "noise", "far", "half", "edge", "nonfinite"):
        coords = grid.copy()
        if kind == "noise":
            coords = (coords + 4 * r.standard_normal(coords.shape)).astype(np.float32)
        if kind == "far":
            coords = (coords + 60 * r.standard_normal(coords.shape)).astype(np.float32)
        if kind == "half":
            coords = (coords + 0.5).astype(np.float32)
        if kind == "edge":
            coords[:, 0] = np.where(coords[:, 0] < w / 2, coords[:, 0] * 0.1 - 3.0, w - 1 + coords[:, 0] * 0.05)
            coords[:, 1] = np.where(coords[:, 1] < h / 2, -2.0, h + 1.25)
            coords = coords.astype(np.float32)
        if kind == "nonfinite":
            coords = coords.astype(np.float32)
            coords[:, 0, ::3, ::5] = np.float32(1e9)
            coords[:, 1, 1::4, 2::7] = np.float32(-3e7)
        ref, ridx, rvalid = oracle.corr_lookup(levels, coords, radius=radius, return_index=True)
        out, idx, valid = _run_lookup(pyr, T(coords), radius)
        _, idx32, valid32 = _run_lookup(p32, T(coords), radius)
        _, idxbf, validbf = _run_lookup(pbf, T(coords), radius)
        assert np.array_equal(idx, ridx) and np.array_equal(valid, rvalid), kind
        assert np.array_equal(idx, idx32) and np.array_equal(valid, valid32), kind
        assert np.array_equal(idx, idxbf) and np.array_equal(valid, validbf), kind
        assert float(np.abs(out - ref).max()) <= 1e-5 * max(1.0, float(np.abs(ref).max())), kind


@gpu
@pytest.mark.parametrize("kind", ["int", "noise"])
def test_fp16_lookup_on_built_pyramid_bench_shape(cuda_lib, kind):
    """K3 on what the fp16 tcgen05 builder stored at 136x240 (query-minor blocks), sampled queries against the oracle
    on the stored levels read back in fp32; indices and masks of every query equal the bf16 block's."""
    from ofb200.ops.corr import CorrBlock

    b, c, h, w = 1, 256, 136, 240
    gen = torch.Generator(device="cuda").manual_seed(1606)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2, pyramid_dtype=torch.float16)
    ref_blk = CorrBlock(f1, f2)
    coords = oracle_coords(b, h, w, 1607, 4.0) if kind == "noise" else T(oracle.coords_grid(b, h, w))
    out, idx, valid = blk(coords, return_index=True)
    _, idx_bf, valid_bf = ref_blk(coords, return_index=True)
    assert torch.equal(idx, idx_bf) and torch.equal(valid, valid_bf)
    n = h * w
    sel = torch.cat([torch.tensor([0, w - 1, n - w, n - 1], device="cuda"),
                     torch.randint(0, n, (1020,), device="cuda", generator=gen)]).unique()
    levels = [N(blk.corr_pyramid[l][sel].float()) for l in range(4)]
    csel = N(coords).reshape(1, 2, n)[:, :, N(sel)].reshape(1, 2, 1, sel.numel())
    ref = oracle.corr_lookup(levels, csel, radius=4)
    got = N(out).reshape(324, n)[:, N(sel)]
    assert float(np.abs(got - ref.reshape(324, -1)).max()) <= 1e-5 * max(1.0, float(np.abs(ref).max()))


# =============================================================================== training
@gpu
def test_fp16_pyramid_training_gradients(cuda_lib):
    """12 lookups and loss.backward() through CorrBlock(..., pyramid_dtype=torch.float16): the backward reads the fp32
    gradient pyramid and the feature maps (bf16 tensor-core GEMMs), never the stored fp16 volume."""
    from ofb200.ops.corr import CorrBlock
    from oracle import torch_port as tp

    r = np.random.default_rng(1608)
    for (b, c, h, w, lv, rad) in [(2, 128, 24, 40, 4, 4), (1, 64, 19, 37, 3, 3), (2, 256, 16, 24, 2, 4)]:
        a1 = r.standard_normal((b, c, h, w)).astype(np.float32)
        a2 = r.standard_normal((b, c, h, w)).astype(np.float32)
        base = np.stack(np.meshgrid(np.arange(w), np.arange(h)), 0)[None].astype(np.float32)
        cs = [(base + 2.5 * r.standard_normal((b, 2, h, w))).astype(np.float32) for _ in range(12)]
        ws = [r.standard_normal((b, lv * (2 * rad + 1) ** 2, h, w)).astype(np.float32) for _ in range(12)]
        c1, c2 = torch.from_numpy(a1).requires_grad_(True), torch.from_numpy(a2).requires_grad_(True)
        pyr = tp.corr_pyramid(c1, c2, lv)
        sum((tp.corr_lookup(pyr, torch.from_numpy(x), rad) * torch.from_numpy(y)).sum() for x, y in zip(cs, ws)).backward()
        g1, g2 = T(a1).requires_grad_(True), T(a2).requires_grad_(True)
        blk = CorrBlock(g1, g2, num_levels=lv, radius=rad, pyramid_dtype=torch.float16)
        assert blk.builder == "tcgen05"
        loss = sum((blk(T(x)) * T(y)).sum() for x, y in zip(cs, ws))
        loss.backward()
        for got, want in ((g1.grad, c1.grad), (g2.grad, c2.grad)):
            assert relfro(got.cpu(), want) <= 6e-3, (b, c, h, w, lv, rad, relfro(got.cpu(), want))
        assert blk._grad.dpyr is None


# =============================================================================== live RAFT
@gpu
def test_live_raft_forward_fp16_pyramid(cuda_lib, tmp_path):
    from test_reference_overlay import NO_REFERENCE, reference_root, run_probe

    ref = reference_root()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    run_probe("raft", "stock", ref, str(tmp_path / "stock.pt"))
    up0 = torch.load(tmp_path / "stock.pt")["flow_up"].double()
    scale = float(up0.abs().max())
    report = {}
    for mode in ("patch", "path"):
        out = tmp_path / f"{mode}_fp16.pt"
        r = run_probe("raft", mode, ref, str(out), env={"OFB200_PYRAMID_DTYPE": "fp16"})
        up = torch.load(out)["flow_up"].double()
        err = float((up - up0).abs().max())
        report[mode] = {"rel_err": err / scale, "ofb_launches": r["ofb_launches"]}
        assert r["ofb_launches"] >= 3 * (3 + 12 + 12), r
        assert err <= 2e-3 * scale, (mode, err, scale)
    print(json.dumps(report))
