"""The correlation lookup's contract, kernel by kernel, element by element: the generic and register-tile forward
lookups (`ofb_corr_lookup`), the lookup backward (`ofb_corr_lookup_backward_f32`) and the on-demand lookup
(`ofb_corr_lookup_ondemand`), at every radius 0-4, 1-4 levels and the coordinates where the tap arithmetic has edges.

All four kernels take their taps from `ofb::lookup_tap` (csrc/common.cuh).  `replay_taps` below replays that sequence in
numpy float32, one rounding per operation, and is checked bit for bit against the CPU oracle; the references of the
GPU tests are built from it (the backward's float64 adjoint) or from the oracle itself (forward, on-demand).

Coordinate kinds (every section runs all of them):
  int        coords_grid: RAFT's first refinement iteration (initialize_flow); most backward windows are irregular
  half       grid + 0.5
  noise      grid + 4 N(0, 1)
  edge       windows hanging over every border
  far        grid + 60 N(0, 1)
  guard      per-level queries whose windows straddle the floor guard [-32768, 70000] at either end
  nonfinite  NaN, +-inf and +-1e9 mixed into a grid
Floor indices are compared where the floor is a finite number: C leaves (int)floorf(x) undefined for NaN and +-inf
(the oracle's x86 conversion gives INT_MIN, the GPU's saturates), and the header defines no index there.

Tolerances (u = 2^-24):
  replay vs oracle                   floor indices and validity masks bit-exact
  adjoint identity (CPU, GPU)        |<lookup(P), G> - <P, lookup_backward(G)>| <= 1e-6 * <lookup(|P|), |G|>
  lookup backward                    |got - adj| <= 1e-6 * A per element, adj = float64 scatter of d_out * w_x * w_y,
                                     A = the same scatter of |d_out| * w_x * w_y (<= 16 fp32 roundings of terms
                                     bounded by A: 16 u A = 0.95e-6 A); A == 0: bit-unchanged.  Accumulated into a
                                     prefilled buffer: <= 1e-6 * (A1 + A2) + 2^-23 * |expected|
  forward lookup                     indices / masks bit-exact; values <= 1e-5 * max(1, |ref|_inf) against the oracle
                                     on the same (dtype-rounded) levels
  on-demand lookup                   |got - ref| <= 2e-6 * S per sample: ref samples the float64 level a_km . f2_l^T
                                     (rounded to fp32) of the kernel's own bf16 operands, S samples |a_km| . |f2_l|^T.
                                     The kernel sums C products in fp32 in at most CPL + 5 roundings (CPL <= 8 FMAs
                                     per lane, a 5-stage butterfly), each bounded by the level of S: 13 u S; the
                                     bilinear sample adds <= 5 u S on either side, the fp32 level 1 u S: 24 u S =
                                     1.4e-6 S.  Windows outside the image (S = 0) are exactly 0.
  on-demand operands                 a_km == bf16(fp32(f1) * fp32(1/sqrt(C))) bit for bit; f2_l within one bf16 ulp
                                     of the float64 mean of each complete 2^l x 2^l block, plus the fp32 summation
                                     bound 4^l u * mean|x|
"""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

import oracle

gpu = pytest.mark.gpu

OFB_OK, OFB_EINVAL, OFB_EUNSUPPORTED, OFB_EALIGN = 0, -1, -2, -3
KINDS = ("int", "half", "noise", "edge", "far", "guard", "nonfinite")
GUARD_ENDS = (-32768.0, 70000.0)          # ofb::LookupTap::in_guard
SPECIALS = np.array([np.nan, np.inf, -np.inf, 1e9, -1e9], np.float32)
BAND = 4096                               # guard band, elements on each side of every buffer


# =============================================================================== references (CPU)
def to_queries(coords):
    """(B, 2, h, w) -> (2, B*h*w), query q = b*h*w + p."""
    b, _, h, w = coords.shape
    return coords.transpose(1, 0, 2, 3).reshape(2, b * h * w)


def from_queries(cq, b, h, w):
    return np.ascontiguousarray(cq.reshape(2, b, h, w).transpose(1, 0, 2, 3))


def make_coords(kind, b, h, w, seed):
    """Coordinates (B, 2, h, w) float32 of one kind (module docstring)."""
    r = np.random.default_rng(seed)
    c = oracle.coords_grid(b, h, w)
    if kind == "half":
        c = c + np.float32(0.5)
    elif kind == "noise":
        c = c + 4 * r.standard_normal(c.shape)
    elif kind == "far":
        c = c + 60 * r.standard_normal(c.shape)
    elif kind == "edge":
        c[:, 0] = np.where(c[:, 0] < w / 2, c[:, 0] * 0.1 - 3.0, w - 1 + c[:, 0] * 0.05)
        c[:, 1] = np.where(c[:, 1] < h / 2, -2.0, h + 1.25)
    elif kind == "guard":
        # query k serves level k % 4: its centre, scaled by 2^l, puts that level's window across one end of the guard
        # (offsets -6 .. 6 in 1/8 steps: some taps on each side).  x, y or both axes; the other axis stays in the image
        cq = to_queries(c).copy()
        k = np.arange(cq.shape[1])
        lvl = k % 4
        for axis in (0, 1):
            end = np.array(GUARD_ENDS)[(k // 4 + axis) % 2]
            val = (end + r.integers(-48, 49, k.size) / 8.0) * 2.0 ** lvl
            on = ((k // 8) % 3 == axis) | ((k // 8) % 3 == 2)
            cq[axis] = np.where(on, val, cq[axis])
        c = from_queries(cq, b, h, w)
    elif kind == "nonfinite":
        cq = to_queries(c).copy()
        k = np.arange(cq.shape[1])
        cq[0] = np.where(k % 3 == 1, SPECIALS[(k // 3) % 5], cq[0])
        cq[1] = np.where(k % 4 == 2, SPECIALS[(k // 4 + 2) % 5], cq[1])
        c = from_queries(cq, b, h, w)
    else:
        assert kind == "int", kind
    return np.ascontiguousarray(c, dtype=np.float32)


def replay_taps(center, radius, size):
    """ofb::lookup_tap in numpy float32, one rounding per operation: center (...) -> floor, w0, w1, valid (..., 2r+1).
    `center` is the level-scaled coordinate coord * 2^-l (exact)."""
    f = np.float32
    c = np.asarray(center, np.float32)[..., None]
    off = (np.arange(2 * radius + 1) - radius).astype(np.float32)
    sm1 = f(size - 1)
    with np.errstate(invalid="ignore", over="ignore"):
        pos = c + off
        g = (f(2) * pos) / sm1 - f(1)
        ic = ((g + f(1)) * f(0.5)) * sm1
        fl = np.floor(ic)
        w1 = ic - fl
        w0 = (fl + f(1)) - ic
        valid = (g > f(-1)) & (g < f(1))
    return fl, w0, w1, valid


def level_taps(coords, level, radius, hl, wl):
    """The x and y taps of every query at one level: two (floor, w0, w1, valid) tuples of (Q, 2r+1) arrays."""
    cq = to_queries(coords)
    s = np.float32(2.0 ** -level)
    return replay_taps(cq[0] * s, radius, wl), replay_taps(cq[1] * s, radius, hl)


def in_guard(fl):
    with np.errstate(invalid="ignore"):
        return (fl >= -32768) & (fl <= 70000)


def replay_index(coords, level_shapes, radius):
    """idx (Q, L, 2, 2r+1) float32 floors (NaN / inf kept), valid (Q, L, (2r+1)^2) u8, in the kernels' layouts."""
    fls, valids = [], []
    for l, (hl, wl) in enumerate(level_shapes):
        tx, ty = level_taps(coords, l, radius, hl, wl)
        fls.append(np.stack([tx[0], ty[0]], 1))
        valids.append((tx[3][:, :, None] & ty[3][:, None, :]).reshape(tx[3].shape[0], -1))
    return np.stack(fls, 1), np.stack(valids, 1).astype(np.uint8)


def same_index(idx, fl):
    """Integer floor indices equal wherever the floor is a finite number (module docstring)."""
    ok = np.isfinite(fl)
    return bool(np.array_equal(idx[ok], fl[ok].astype(np.int64)))


def lookup_adjoint_f64(level_shapes, coords, d_out, radius):
    """The lookup's adjoint in float64: d_out (B, L*(2r+1)^2, h, w) scattered with weight w_x * w_y into the four taps
    of every sample that lie inside the image.  Returns per level the (Q, h_l, w_l) gradient and A, the same scatter of
    |d_out|."""
    b, _, h, w = coords.shape
    q, d, lv = b * h * w, 2 * radius + 1, len(level_shapes)
    g = d_out.reshape(b, -1, d, d, h * w)[:, :lv].transpose(0, 4, 1, 2, 3).reshape(q, lv, d, d).astype(np.float64)
    grads, absg = [], []
    for l, (hl, wl) in enumerate(level_shapes):
        tx, ty = level_taps(coords, l, radius, hl, wl)
        n = q * hl * wl
        acc, aacc = np.zeros(n), np.zeros(n)
        qbase = (np.arange(q) * (hl * wl))[:, None, None]
        with np.errstate(invalid="ignore"):
            for dx, wx in ((0, tx[1]), (1, tx[2])):
                xi = tx[0] + np.float32(dx)
                inx = (xi >= 0) & (xi < wl)
                xi = np.where(inx, xi, 0).astype(np.int64)
                for dy, wy in ((0, ty[1]), (1, ty[2])):
                    yi = ty[0] + np.float32(dy)
                    iny = (yi >= 0) & (yi < hl)
                    yi = np.where(iny, yi, 0).astype(np.int64)
                    m = inx[:, :, None] & iny[:, None, :]
                    flat = (qbase + yi[:, None, :] * wl + xi[:, :, None])[m]
                    wgt = (wx.astype(np.float64)[:, :, None] * wy.astype(np.float64)[:, None, :])[m]
                    gl = g[:, l][m]
                    acc += np.bincount(flat, weights=gl * wgt, minlength=n)
                    aacc += np.bincount(flat, weights=np.abs(gl) * wgt, minlength=n)
        grads.append(acc.reshape(q, hl, wl))
        absg.append(aacc.reshape(q, hl, wl))
    return grads, absg


def level_shapes_of(h, w, levels):
    return [(h >> l, w >> l) for l in range(levels)]


def dead_queries(coords, level_shapes, radius):
    """Queries whose windows have no tap inside the image at any level (non-finite, out-of-guard or far coordinates)."""
    dead = np.ones(coords.shape[0] * coords.shape[2] * coords.shape[3], bool)
    for l, (hl, wl) in enumerate(level_shapes):
        tx, ty = level_taps(coords, l, radius, hl, wl)
        with np.errstate(invalid="ignore"):
            hit_x = ((tx[0] >= -1) & (tx[0] < wl)).any(1)
            hit_y = ((ty[0] >= -1) & (ty[0] < hl)).any(1)
        dead &= ~(hit_x & hit_y)
    return dead


def window_branches(coords, level, radius, hl, wl):
    """Per query at one level: the backward kernel's branch (regular: every tap in the guard and floors consecutive on
    both axes) and whether some tap is outside the guard."""
    tx, ty = level_taps(coords, level, radius, hl, wl)
    t = np.arange(2 * radius + 1, dtype=np.float32)
    with np.errstate(invalid="ignore"):
        regular = np.ones(tx[0].shape[0], bool)
        out_guard = np.zeros(tx[0].shape[0], bool)
        for fl in (tx[0], ty[0]):
            ing = in_guard(fl)
            regular &= ing.all(1) & (fl == fl[:, :1] + t).all(1)
            out_guard |= ~ing.all(1)
    return regular, out_guard


# geometries (h, w) of the CPU replay check: odd sizes, a 2-pixel-wide last level, a non-square one
REPLAY_GEOMS = [(19, 37), (24, 16), (23, 41)]


@pytest.mark.parametrize("geom", REPLAY_GEOMS)
@pytest.mark.parametrize("radius", range(5))
def test_replay_matches_oracle_indices_and_masks(geom, radius):
    """The float32 replay of ofb::lookup_tap reproduces the oracle's floor indices and validity masks bit for bit (idx
    where the coordinate is not NaN), for every coordinate kind and 1 to 4 levels."""
    h, w = geom
    b = 2
    for kind in KINDS:
        coords = make_coords(kind, b, h, w, 11 + radius)
        for levels in range(1, 5):
            shapes = level_shapes_of(h, w, levels)
            zeros = [np.zeros((1, 1, hl, wl), np.float32) for hl, wl in shapes]
            _, ridx, rvalid = oracle.corr_lookup(zeros, coords, radius=radius, return_index=True, shared_slice=True)
            fl, valid = replay_index(coords, shapes, radius)
            assert np.array_equal(valid, rvalid), (kind, levels)
            notnan = ~np.isnan(fl)
            with np.errstate(invalid="ignore"):
                assert np.array_equal(ridx[notnan], fl[notnan].astype(np.int32)), (kind, levels)


@pytest.mark.parametrize("radius", range(5))
def test_adjoint_identity_against_oracle_forward(radius):
    """<oracle.corr_lookup(P), G> == <P, lookup_adjoint_f64(G)> on an fp32 pyramid, every coordinate kind."""
    b, h, w, levels = 2, 19, 37, 4
    r = np.random.default_rng(20 + radius)
    d = 2 * radius + 1
    shapes = level_shapes_of(h, w, levels)
    pyr = [r.standard_normal((b * h * w, 1, hl, wl)).astype(np.float32) for hl, wl in shapes]
    for kind in KINDS:
        coords = make_coords(kind, b, h, w, 30 + radius)
        g = r.standard_normal((b, levels * d * d, h, w)).astype(np.float32)
        fwd = oracle.corr_lookup(pyr, coords, radius=radius)
        adj, amag = lookup_adjoint_f64(shapes, coords, g, radius)
        lhs = float(np.dot(fwd.ravel().astype(np.float64), g.ravel().astype(np.float64)))
        rhs = sum(float(np.dot(p.ravel().astype(np.float64), a.ravel())) for p, a in zip(pyr, adj))
        scale = sum(float(np.dot(np.abs(p.ravel()).astype(np.float64), a.ravel())) for p, a in zip(pyr, amag))
        assert abs(lhs - rhs) <= 1e-6 * scale, (kind, lhs, rhs, scale)


# the lookup backward's matrix: B = 2 with a query count that is not a multiple of 128; a 2-pixel-wide last level
BWD_SHAPES = [(2, 19, 37), (1, 24, 16)]


def bwd_coords(kind, shape, radius):
    """The coordinates the lookup backward tests run (and whose branch coverage is asserted below)."""
    b, h, w = shape
    return make_coords(kind, b, h, w, 210 + radius)


@pytest.mark.parametrize("shape", BWD_SHAPES)
def test_backward_matrix_reaches_both_branches(shape):
    """The coordinates of test_lookup_backward_matches_float64_adjoint drive both branches of lookup_bwd_kernel:
    integer coordinates put more than 20 % of the level-0 windows (radius >= 1) through the irregular scatter, noise at
    least half through the separable regular path, and guard / non-finite coordinates give windows with an out-of-guard
    tap; the guard windows straddle an end of the guard (taps on both sides) on both axes at every level."""
    b, h, w = shape
    for radius in range(1, 5):
        reg = {k: window_branches(bwd_coords(k, shape, radius), 0, radius, h, w) for k in KINDS}
        assert (~reg["int"][0]).mean() > 0.2, (radius, (~reg["int"][0]).mean())
        assert reg["noise"][0].mean() >= 0.5, radius
        for kind in ("guard", "nonfinite"):
            assert reg[kind][1].any(), (kind, radius)
        coords = bwd_coords("guard", shape, radius)
        for l, (hl, wl) in enumerate(level_shapes_of(h, w, 4)):
            tx, ty = level_taps(coords, l, radius, hl, wl)
            both = [(in_guard(fl).any(1) & ~in_guard(fl).all(1)).any() for fl in (tx[0], ty[0])]
            assert all(both), (radius, l)


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


def test_lookup_backward_validates_arguments_without_launch(lib):
    import ofb200

    fake = ctypes.c_void_p(1 << 20)                      # never dereferenced: every call below is rejected first

    def pyr(levels=4, dtype=ofb200.DTYPE_F32, mode=1):
        p = ofb200.Pyramid()
        elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
        assert lib.ofb_pyramid_layout(16, 24, 4, mode, ctypes.byref(p), ctypes.byref(elems)) == 0
        for l in range(4):
            p.base[l] = 1 << 20
        p.levels, p.dtype = levels, dtype
        return p

    def call(p, coords=fake, d_out=fake, radius=4):
        return lib.ofb_corr_lookup_backward_f32(ctypes.byref(p) if p is not None else None, coords, d_out, 1, 16, 24,
                                                radius, None)

    assert call(None) == OFB_EINVAL
    assert call(pyr(), coords=None) == OFB_EINVAL
    assert call(pyr(), d_out=None) == OFB_EINVAL
    assert call(pyr(dtype=ofb200.DTYPE_BF16)) == OFB_EUNSUPPORTED
    assert call(pyr(dtype=ofb200.DTYPE_F16)) == OFB_EUNSUPPORTED
    assert call(pyr(mode=2)) == OFB_EUNSUPPORTED
    assert call(pyr(mode=3)) == OFB_EUNSUPPORTED
    assert call(pyr(), radius=5) == OFB_EUNSUPPORTED
    assert call(pyr(), radius=-1) == OFB_EUNSUPPORTED
    assert call(pyr(levels=0)) == OFB_EINVAL
    assert call(pyr(levels=5)) == OFB_EINVAL
    p = pyr()
    p.row_pitch[2] = p.lvl_w[2] - 1
    assert call(p) == OFB_EINVAL
    p = pyr()
    p.base[3] = None
    assert call(p) == OFB_EINVAL


def test_pyramid_descriptor_checks_agree_without_launch(lib):
    """A descriptor that breaks a rule every user relies on is OFB_EINVAL at all five pyramid entry points; and the
    forward lookup and its coordinate backward give the same code for every layout, dtype, radius 0-4 and descriptor
    variant.  B * h * w = 2^36 queries is too many for either launch, so a descriptor both readers accept is refused
    only there (OFB_EUNSUPPORTED) and nothing is launched."""
    import ofb200

    fake = ctypes.c_void_p(1 << 20)                      # never dereferenced: every call below returns before a launch

    def pyr(mode, dtype, base=1 << 20):
        p = ofb200.Pyramid()
        elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
        assert lib.ofb_pyramid_layout(16, 24, 4, mode, ctypes.byref(p), ctypes.byref(elems)) == 0
        for l in range(4):
            p.base[l] = base
        p.dtype = dtype
        return p

    def entry_points(p):
        r = ctypes.byref(p)
        return [lib.ofb_corr_lookup(r, fake, fake, None, None, 1, 16, 24, 4, None),
                lib.ofb_corr_lookup_coords_backward(r, fake, fake, fake, 1, 16, 24, 4, None),
                lib.ofb_corr_lookup_backward_f32(r, fake, fake, 1, 16, 24, 4, None),
                lib.ofb_corr_pyramid_bf16(fake, fake, fake, r, 1, 64, 16, 24, 1.0, 0, None),
                lib.ofb_corr_pyramid_simt_f32(fake, fake, r, 1, 64, 16, 24, 1.0, None)]

    def edit(**kw):
        def apply(p):
            for k, v in kw.items():
                if isinstance(v, tuple):
                    getattr(p, k)[v[0]] = v[1]
                else:
                    setattr(p, k, v)
            return p
        return apply

    before = lib.ofb_launch_count()
    broken = [edit(levels=0), edit(levels=5), edit(dtype=3), edit(dtype=-1), edit(layout=3), edit(layout=-1),
              edit(base=(2, None)), edit(lvl_h=(1, 0)), edit(lvl_w=(3, 0)), edit(row_pitch=(2, 5)),
              edit(q_stride=(1, 64))]
    for dtype in (ofb200.DTYPE_F32, ofb200.DTYPE_BF16):
        for k, fault in enumerate(broken):
            p = fault(pyr(3, dtype))                         # query-minor 8x4 blocks: q_stride = 32 until broken
            assert entry_points(p) == [OFB_EINVAL] * 5, (dtype, k)

    variants = [edit(), edit(base=(1, (1 << 20) + 2)), edit(base=(2, (1 << 20) + 4)), edit(row_pitch=(1, 13)),
                edit(row_pitch=(1, 14)), edit(lvl_w=(0, 70000), row_pitch=(0, 70000)), edit(q_stride=(3, 64))]
    seen = set()
    for mode in range(4):
        for dtype in (ofb200.DTYPE_F32, ofb200.DTYPE_BF16, ofb200.DTYPE_F16):
            for radius in range(5):
                for k, variant in enumerate(variants):
                    r = ctypes.byref(variant(pyr(mode, dtype)))
                    fwd = lib.ofb_corr_lookup(r, fake, fake, None, None, 65536, 1024, 1024, radius, None)
                    bwd = lib.ofb_corr_lookup_coords_backward(r, fake, fake, fake, 65536, 1024, 1024, radius, None)
                    assert fwd == bwd, (mode, dtype, radius, k, fwd, bwd)
                    seen.add(fwd)
    assert seen == {OFB_EINVAL, OFB_EUNSUPPORTED, OFB_EALIGN}
    assert lib.ofb_launch_count() == before


def test_ondemand_lookup_validates_arguments_without_launch(lib):
    fake = 1 << 20

    def call(c=64, levels=4, radius=4, f1=fake, lvl=(fake,) * 4, h=16, w=24):
        ptrs = (ctypes.c_void_p * 4)(*lvl)
        return lib.ofb_corr_lookup_ondemand(ctypes.c_void_p(f1), ptrs, ctypes.c_void_p(fake), ctypes.c_void_p(fake), 1, c,
                                            h, w, levels, radius, None)

    assert call(c=96) == OFB_EUNSUPPORTED
    assert call(c=192) == OFB_EUNSUPPORTED
    assert call(radius=5) == OFB_EUNSUPPORTED
    assert call(levels=0) == OFB_EINVAL
    assert call(levels=5) == OFB_EINVAL
    assert call(f1=fake + 8) == OFB_EALIGN
    assert call(lvl=(fake, fake, fake + 4, fake)) == OFB_EALIGN
    assert call(lvl=(fake, None, fake, fake)) == OFB_EINVAL
    assert call(h=4) == OFB_EINVAL                       # h >> 3 == 0
    assert call(w=7, levels=4) == OFB_EINVAL             # w >> 3 == 0
    assert lib.ofb_corr_lookup_ondemand(ctypes.c_void_p(fake), None, ctypes.c_void_p(fake), ctypes.c_void_p(fake), 1, 64,
                                        16, 24, 4, 4, None) == OFB_EINVAL


# =============================================================================== GPU helpers
def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().cpu().numpy()


def banded(n, dtype, sentinel):
    """A sentinel-filled allocation of n + 2 * BAND elements and its middle n-element view."""
    whole = torch.full((n + 2 * BAND,), sentinel, dtype=dtype, device="cuda")
    return whole, whole[BAND:BAND + n]


def bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}[t.dtype])


def bands_intact(whole, sentinel):
    ref = bits(torch.full((BAND,), sentinel, dtype=whole.dtype, device="cuda"))
    return bool(torch.equal(bits(whole[:BAND]), ref)) and bool(torch.equal(bits(whole[-BAND:]), ref))


# =============================================================================== lookup backward (GPU)
GRAD_PAD = -0.0   # padding / band sentinel of the gradient pyramid: adding anything but -0.0 to it changes its bits


def grad_pyramid(q, h, w, levels, mode, fill):
    """fp32 gradient pyramid in ofb_pyramid_layout mode 0 (tight rows, CorrBlock's) or 1 (padded rows), each level
    inside a GRAD_PAD-filled guard band; the image elements hold `fill` ((Q, h_l, w_l) arrays or a scalar)."""
    import ofb200

    lib = ofb200.load()
    pyr = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    ofb200.check(lib.ofb_pyramid_layout(h, w, levels, mode, ctypes.byref(pyr), ctypes.byref(elems)), "ofb_pyramid_layout")
    pyr.dtype = ofb200.DTYPE_F32
    keep = []
    for l in range(levels):
        whole, view = banded(q * int(elems[l]), torch.float32, GRAD_PAD)
        img = view.view(q, pyr.lvl_h[l], pyr.row_pitch[l])
        img[:, :, :pyr.lvl_w[l]] = T(fill[l]) if isinstance(fill, list) else fill
        pyr.base[l] = view.data_ptr()
        keep.append((whole, img))
    return pyr, keep


def run_backward(pyr, coords_d, d_out_d, radius):
    import ofb200

    b, _, h, w = coords_d.shape
    rc = ofb200.load().ofb_corr_lookup_backward_f32(ctypes.byref(pyr), ofb200.ptr(coords_d), ofb200.ptr(d_out_d), b, h,
                                                    w, radius, ofb200.stream_ptr())
    ofb200.check(rc, "ofb_corr_lookup_backward_f32")


def check_padding(keep, pyr, what):
    """Guard bands and padding columns keep the GRAD_PAD sentinel bit for bit."""
    pad = bits(torch.tensor(GRAD_PAD, device="cuda"))
    for l, (whole, img) in enumerate(keep):
        assert bands_intact(whole, GRAD_PAD), (what, l)
        if pyr.row_pitch[l] > pyr.lvl_w[l]:
            assert bool((bits(img[:, :, pyr.lvl_w[l]:]) == pad).all()), (what, l)


@gpu
@pytest.mark.parametrize("radius", range(5))
@pytest.mark.parametrize("shape", BWD_SHAPES)
def test_lookup_backward_matches_float64_adjoint(cuda_lib, shape, radius):
    """ofb_corr_lookup_backward_f32 through the C ABI on a zero-filled gradient pyramid, 1-4 levels, row layout modes 0
    and 1, every coordinate kind: |got - adj| <= 1e-6 * A per element, elements with A == 0 bit-unchanged (+0.0),
    padding columns and 4096-element guard bands around every level untouched."""
    b, h, w = shape
    q, d = b * h * w, 2 * radius + 1
    shapes = level_shapes_of(h, w, 4)
    r = np.random.default_rng(200 + radius + h)
    for kind in KINDS:
        coords = bwd_coords(kind, shape, radius)
        d_out = r.standard_normal((b, 4 * d * d, h, w)).astype(np.float32)
        adj, amag = lookup_adjoint_f64(shapes, coords, d_out, radius)
        coords_d = T(coords)
        for levels in range(1, 5):
            d_sub = T(d_out[:, :levels * d * d])
            for mode in (0, 1):
                what = (kind, levels, mode)
                pyr, keep = grad_pyramid(q, h, w, levels, mode, 0.0)
                run_backward(pyr, coords_d, d_sub, radius)
                torch.cuda.synchronize()
                check_padding(keep, pyr, what)
                for l in range(levels):
                    got_t = keep[l][1][:, :, :shapes[l][1]]
                    got = N(got_t).astype(np.float64)
                    err = np.abs(got - adj[l])
                    bad = ~(err <= 1e-6 * amag[l])                  # NaN fails
                    assert not bad.any(), (what, l, int(bad.sum()), float(err.max()), np.argwhere(bad)[:4].tolist())
                    untouched = N(bits(got_t.contiguous()))[amag[l] == 0]
                    assert not untouched.any(), (what, l)


@gpu
@pytest.mark.parametrize("radius", [1, 4])
def test_lookup_backward_accumulates_into_the_pyramid(cuda_lib, radius):
    """Two backward calls into a prefilled gradient pyramid (padded rows) equal prefill + adj1 + adj2; the slices of
    queries whose windows miss the image at every level (non-finite, out-of-guard or far coordinates) stay bit-equal
    to the prefill."""
    b, h, w, levels = 2, 19, 37, 4
    q, d = b * h * w, 2 * radius + 1
    shapes = level_shapes_of(h, w, levels)
    r = np.random.default_rng(300 + radius)
    prefill = [r.standard_normal((q, hl, wl)).astype(np.float32) for hl, wl in shapes]
    pyr, keep = grad_pyramid(q, h, w, levels, 1, prefill)
    expected = [p.astype(np.float64) for p in prefill]
    amag = [np.zeros(p.shape) for p in prefill]
    dead = np.ones(q, bool)
    k = np.arange(q)
    sel = k % 7 == 3
    for call, kind in enumerate(("int", "noise")):
        cq = to_queries(make_coords(kind, b, h, w, 310 + call)).copy()
        # every 7th query: a non-finite, out-of-guard or in-guard-but-far coordinate on one axis
        bad = np.array([np.nan, np.inf, -np.inf, 1e9, 9e4 * 8, -4e4, 5000.0], np.float32)[(k // 7 + call) % 7]
        axis = (k // 7) % 2
        cq[0] = np.where(sel & (axis == 0), bad, cq[0])
        cq[1] = np.where(sel & (axis == 1), bad, cq[1])
        coords = from_queries(cq, b, h, w)
        dead &= dead_queries(coords, shapes, radius)
        d_out = r.standard_normal((b, levels * d * d, h, w)).astype(np.float32)
        adj, am = lookup_adjoint_f64(shapes, coords, d_out, radius)
        for l in range(levels):
            expected[l] += adj[l]
            amag[l] += am[l]
        run_backward(pyr, T(coords), T(d_out), radius)
    torch.cuda.synchronize()
    check_padding(keep, pyr, "accumulate")
    assert dead[sel].all()
    for l in range(levels):
        got_t = keep[l][1][:, :, :shapes[l][1]].contiguous()
        got = N(got_t).astype(np.float64)
        bound = 1e-6 * amag[l] + 2.0 ** -23 * np.abs(expected[l])
        assert bool((np.abs(got - expected[l]) <= bound).all()), (l, float(np.abs(got - expected[l]).max()))
        assert np.array_equal(N(bits(got_t))[dead], prefill[l].view(np.int32)[dead]), l


# =============================================================================== forward lookup (GPU)
FWD_LAYOUTS = ("rows16", "rows2mod8", "block8x4", "qminor8x4")
FWD_SHAPES = [(2, 19, 37), (1, 24, 16)]
TORCH_DT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def poison(dtype):
    """Padding value: NaN in fp32 (never read); the largest finite value in 16-bit (read, with weight zero)."""
    return float("nan") if dtype == torch.float32 else float(torch.finfo(dtype).max)


def lookup_pyramid(levels, dtype, layout, b, h, w):
    """Device pyramid of the (Q, 1, h_l, w_l) float32 levels (already rounded to dtype) in one of FWD_LAYOUTS, padding
    poisoned.  Returns the descriptor and the buffers that back it."""
    import ofb200
    from ofb200.ops.corr import level_buffer

    q = levels[0].shape[0]
    pyr = ofb200.Pyramid()
    pyr.levels = len(levels)
    pyr.dtype = {torch.float32: ofb200.DTYPE_F32, torch.bfloat16: ofb200.DTYPE_BF16, torch.float16: ofb200.DTYPE_F16}[dtype]
    pyr.layout = {"block8x4": ofb200.LAYOUT_BLOCK8X4, "qminor8x4": ofb200.LAYOUT_QMINOR8X4}.get(layout, ofb200.LAYOUT_ROWS)
    bufs = []
    for l, lv in enumerate(levels):
        hl, wl = lv.shape[-2:]
        if layout == "rows16":
            pitch, rows = (wl + 15) & ~15, hl
        elif layout == "rows2mod8":
            pitch, rows = wl + (2 - wl) % 8, hl
        else:
            pitch, rows = (wl + 7) & ~7, (hl + 3) & ~3
        img = torch.full((q, rows, pitch), poison(dtype), dtype=dtype, device="cuda")
        img[:, :hl, :wl] = T(lv[:, 0]).to(dtype)
        buf = level_buffer(img, pyr.layout)
        bufs.append(buf)
        pyr.base[l] = buf.data_ptr()
        pyr.q_stride[l] = 32 if layout == "qminor8x4" else rows * pitch
        pyr.row_pitch[l] = pitch
        pyr.lvl_h[l] = hl
        pyr.lvl_w[l] = wl
    return pyr, bufs


def run_lookup(pyr, coords_d, radius):
    """ofb_corr_lookup -> (rc, out, idx, valid); the outputs are None when the call is rejected."""
    import ofb200

    b, _, h, w = coords_d.shape
    d, lv = 2 * radius + 1, pyr.levels
    out = torch.empty((b, lv * d * d, h, w), device="cuda")
    idx = torch.empty((b * h * w, lv, 2, d), dtype=torch.int32, device="cuda")
    valid = torch.empty((b * h * w, lv, d * d), dtype=torch.uint8, device="cuda")
    rc = ofb200.load().ofb_corr_lookup(ctypes.byref(pyr), ofb200.ptr(coords_d), ofb200.ptr(out), ofb200.ptr(idx),
                                       ofb200.ptr(valid), b, h, w, radius, ofb200.stream_ptr())
    if rc != OFB_OK:
        return rc, None, None, None
    return rc, N(out), N(idx), N(valid)


@gpu
@pytest.mark.parametrize("shape", FWD_SHAPES)
@pytest.mark.parametrize("dtype", ["fp32", "bf16", "fp16"])
def test_lookup_forward_every_kernel_matches_oracle(cuda_lib, dtype, shape):
    """ofb_corr_lookup on pyramids the test lays out itself: rows with a pitch that is a multiple of 16 (the register-tile
    kernel at radius 3 and 4 for 16-bit), rows with pitch = 2 (mod 8) (the generic kernel at every radius), 8x4 blocks
    and query-minor 8x4 blocks (register-tile only: fp32 and radius <= 2 must return OFB_EUNSUPPORTED); radius 0-4,
    1-4 levels, every coordinate kind.  Indices and masks bit-exact, values <= 1e-5 * max(1, |ref|_inf)."""
    b, h, w = shape
    tdt = TORCH_DT[dtype]
    q = b * h * w
    r = np.random.default_rng(400 + h)
    shapes = level_shapes_of(h, w, 4)
    levels = [T(8 * r.standard_normal((q, 1, hl, wl)).astype(np.float32)).to(tdt).float().cpu().numpy()
              for hl, wl in shapes]
    pyrs = {layout: lookup_pyramid(levels, tdt, layout, b, h, w) for layout in FWD_LAYOUTS}
    for radius in range(5):
        d = 2 * radius + 1
        for kind in KINDS:
            coords = make_coords(kind, b, h, w, 410 + radius)
            ref, _, rvalid = oracle.corr_lookup(levels, coords, radius=radius, return_index=True)
            fl, valid = replay_index(coords, shapes, radius)
            assert np.array_equal(valid, rvalid)
            coords_d = T(coords)
            for layout, (pyr, _) in pyrs.items():
                unsupported = layout.startswith(("block", "qminor")) and (dtype == "fp32" or radius <= 2)
                for nl in range(1, 5):
                    pyr.levels = nl
                    what = (kind, radius, layout, nl)
                    rc, out, idx, vmask = run_lookup(pyr, coords_d, radius)
                    if unsupported:
                        assert rc == OFB_EUNSUPPORTED, what
                        continue
                    assert rc == OFB_OK, what
                    assert same_index(idx, fl[:, :nl]), what
                    assert np.array_equal(vmask, rvalid[:, :nl]), what
                    want = ref[:, :nl * d * d]
                    err = float(np.abs(out.astype(np.float64) - want).max())
                    assert err <= 1e-5 * max(1.0, float(np.abs(want).max())), (what, err)
                pyr.levels = 4


@gpu
@pytest.mark.parametrize("radius", range(5))
def test_lookup_forward_and_backward_are_adjoint(cuda_lib, radius):
    """<lookup(P), G> == <P, lookup_backward(G)> between the two fp32 kernels, without the oracle: the forward's and
    the backward's tap sets and weights are the same."""
    import ofb200

    b, h, w, levels = 2, 19, 37, 4
    q, d = b * h * w, 2 * radius + 1
    gen = torch.Generator(device="cuda").manual_seed(500 + radius)
    lib = ofb200.load()
    p_pyr = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    ofb200.check(lib.ofb_pyramid_layout(h, w, levels, 0, ctypes.byref(p_pyr), ctypes.byref(elems)), "layout")
    p_pyr.dtype = ofb200.DTYPE_F32
    a_pyr = ofb200.Pyramid.from_buffer_copy(p_pyr)
    bufs = [torch.randn(q * int(elems[l]), device="cuda", generator=gen) for l in range(levels)]
    abs_bufs = [x.abs() for x in bufs]
    for l in range(levels):
        p_pyr.base[l] = bufs[l].data_ptr()
        a_pyr.base[l] = abs_bufs[l].data_ptr()
    for kind in KINDS:
        coords_d = T(make_coords(kind, b, h, w, 510 + radius))
        g = torch.randn((b, levels * d * d, h, w), device="cuda", generator=gen)
        rc, out, _, _ = run_lookup(p_pyr, coords_d, radius)
        assert rc == OFB_OK
        _, out_abs, _, _ = run_lookup(a_pyr, coords_d, radius)
        lhs = float((torch.from_numpy(out).double() * g.cpu().double()).sum())
        scale = float((torch.from_numpy(out_abs).double() * g.cpu().double().abs()).sum())
        dpyr, keep = grad_pyramid(q, h, w, levels, 0, 0.0)
        run_backward(dpyr, coords_d, g, radius)
        rhs = sum(float((keep[l][1].double().flatten() * bufs[l].double()).sum()) for l in range(levels))
        assert abs(lhs - rhs) <= 1e-6 * scale, (kind, lhs, rhs, scale)


# =============================================================================== on-demand lookup (GPU)
def ulp_bf16(x):
    """bf16 unit in the last place at the magnitude of x (float64 tensor), 2^(floor(log2|x|) - 7)."""
    _, e = torch.frexp(x.abs().float())
    return torch.ldexp(torch.ones_like(x), (e - 1).clamp(min=-126).to(torch.int32) - 7)


def ondemand_block(b, c, h, w, seed):
    from ofb200.ops.corr import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(seed)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2, num_levels=4, radius=4, on_demand=True)
    assert blk.builder == "on_demand"
    return f1, f2, blk._on_demand


@gpu
@pytest.mark.parametrize("c", [64, 128, 256])
def test_ondemand_operands(cuda_lib, c):
    """The on-demand lookup's operands: a_km == bf16(fp32(f1) * fp32(1/sqrt(C))) transposed, bit for bit; f2 pooled by
    1, 2, 4 and 8 within one bf16 ulp (+ the fp32 summation bound) of the float64 mean of each complete block."""
    b, h, w = 2, 19, 37
    f1, f2, (a_km, f2_levels) = ondemand_block(b, c, h, w, 600 + c)
    want = (f1 * torch.tensor(1.0 / math.sqrt(c), dtype=torch.float32)).bfloat16().reshape(b, c, h * w).transpose(1, 2)
    assert torch.equal(bits(a_km.contiguous()), bits(want.contiguous()))
    for l, got in enumerate(f2_levels):
        k = 1 << l
        ref = torch.nn.functional.avg_pool2d(f2.double(), k) if k > 1 else f2.double()
        mag = torch.nn.functional.avg_pool2d(f2.double().abs(), k) if k > 1 else f2.double().abs()
        ref = ref.reshape(b, c, -1).transpose(1, 2)
        mag = mag.reshape(b, c, -1).transpose(1, 2)
        assert got.shape == ref.shape
        bound = ulp_bf16(ref) + k * k * 2.0 ** -24 * mag
        err = (got.double() - ref).abs()
        assert bool((err <= bound).all()), (l, float((err / bound).max()))


def ondemand_queries(b, h, w, gen, count):
    """Every query for small shapes; else the corners of every 8 x 4 query tile, the image corners and `count` random."""
    n = h * w
    if b * n <= 4096:
        return np.arange(b * n)
    y, x = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    corner = ((x % 8 == 0) | (x % 8 == 7) | (x == w - 1)) & ((y % 4 == 0) | (y % 4 == 3) | (y == h - 1))
    tile = np.flatnonzero(corner.ravel())
    extra = gen.integers(0, b * n, count)
    return np.unique(np.concatenate([tile, (b - 1) * n + tile, extra]))


def ondemand_levels(a_km, f2_levels, sel, h, w):
    """For the selected queries: each level a_km . f2_l^T formed in float64 on the device and rounded to fp32, and
    |a_km| . |f2_l|^T, as (len(sel), 1, h_l, w_l) float32 arrays."""
    b, n, _ = a_km.shape
    qb, qp = sel // n, sel % n
    vals, mags = [], []
    for l, f2l in enumerate(f2_levels):
        hl, wl = h >> l, w >> l
        v = torch.empty((sel.size, hl * wl), dtype=torch.float64, device="cuda")
        m = torch.empty_like(v)
        for bi in range(b):
            rows = np.flatnonzero(qb == bi)
            if rows.size == 0:
                continue
            a = a_km[bi, torch.from_numpy(qp[rows]).cuda()].double()
            f = f2l[bi].double()
            ridx = torch.from_numpy(rows).cuda()
            v[ridx] = a @ f.t()
            m[ridx] = a.abs() @ f.abs().t()
        vals.append(N(v.float()).reshape(-1, 1, hl, wl))
        mags.append(N(m.float()).reshape(-1, 1, hl, wl))
    return vals, mags


# (C, (B, h, w)): w % 8 != 0 and h % 4 != 0 throughout; 47 x 156 has 960 work items (> 148 SMs x 4 resident CTAs), so
# the persistent loop wraps
OD_CASES = [(64, (2, 19, 37)), (128, (2, 19, 37)), (256, (2, 19, 37)), (128, (1, 47, 156))]


@gpu
@pytest.mark.parametrize("c,shape", OD_CASES)
def test_ondemand_lookup_matches_its_operands(cuda_lib, c, shape):
    """ofb_corr_lookup_ondemand against the oracle sampling the float64 product of the kernel's own bf16 operands:
    |got - ref| <= 2e-6 * S per sample (module docstring), radius 0-4, 1-4 levels, every coordinate kind; windows
    that miss the image (far, guard, non-finite) are exactly 0."""
    import ofb200

    b, h, w = shape
    n = h * w
    _, _, (a_km, f2_levels) = ondemand_block(b, c, h, w, 700 + c + h)
    r = np.random.default_rng(710 + c)
    sel = ondemand_queries(b, h, w, r, 2048)
    vals, mags = ondemand_levels(a_km, f2_levels, sel, h, w)
    lib = ofb200.load()
    ptrs = (ctypes.c_void_p * ofb200.MAX_LEVELS)(*[t.data_ptr() for t in f2_levels])
    for radius in range(5):
        dd = (2 * radius + 1) ** 2
        for kind in KINDS:
            coords = make_coords(kind, b, h, w, 720 + radius)
            csel = to_queries(coords)[:, sel].reshape(1, 2, 1, sel.size)
            ref = oracle.corr_lookup(vals, csel, radius=radius).reshape(4 * dd, sel.size).astype(np.float64)
            s = oracle.corr_lookup(mags, csel, radius=radius).reshape(4 * dd, sel.size).astype(np.float64)
            coords_d = T(coords)
            for levels in range(1, 5):
                out = torch.empty((b, levels * dd, h, w), device="cuda")
                rc = lib.ofb_corr_lookup_ondemand(ofb200.ptr(a_km), ptrs, ofb200.ptr(coords_d), ofb200.ptr(out), b, c, h,
                                                  w, levels, radius, ofb200.stream_ptr())
                assert rc == OFB_OK
                got = N(out).transpose(1, 0, 2, 3).reshape(levels * dd, b * n)[:, sel].astype(np.float64)
                err = np.abs(got - ref[:levels * dd])
                bad = ~(err <= 2e-6 * s[:levels * dd])                 # NaN fails
                what = (kind, radius, levels)
                assert not bad.any(), (what, int(bad.sum()), float(err.max()), np.argwhere(bad)[:4].tolist())
