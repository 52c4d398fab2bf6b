"""Element-by-element contract of the correlation block's tensor-core kernels and the passes that feed them.

The reference of every kernel is float64 arithmetic on the operands the kernel itself reads: its own 16-bit K-major
operands (prepare_operands), its own pooled operands, and bf16 of the gradient pyramid.  Those operand kernels are
checked bit for bit against torch replicas of their fp32 arithmetic, so the float64 references start from exactly
the values the tensor cores see.

Error bounds (`eps`), derived per output element from T = sum |terms| and m = the number of nonzero terms:
  * a tensor-core fp32 accumulation (tcgen05.mma kind::f16): the products of two bf16 / fp16 values are exact in fp32
    (8 + 8 and 11 + 11 significand bits <= 24).  The order and rounding of the hardware's additions are unspecified;
    each step that adds a nonzero term loses less than one fp32 ulp of a partial sum, and every partial sum is at most
    T in magnitude, so |acc - sum| <= m * 2^-23 * T (U_ACC);
  * an fp32 operation on the CUDA cores rounds to nearest: <= 2^-24 (U_RN) of its result's magnitude.  The 2x2 means
    add four values in three such steps (the * 0.25 is exact), the scale and alpha multiplies are one step each;
  * a 16-bit stored value passes when it lies in the BRACKET [RNE(ref - w), RNE(ref + w)] of its dtype, with
    w = eps + 2^-23 * (|ref| + eps): torch rounds float64 to bf16 / fp16 through fp32, and the extra fp32 ulp keeps
    that double rounding from narrowing the bracket (rounding is monotone).  fp32 outputs pass when |got - ref| <= eps.
The CPU test below shows the bracket rejects truncated, doubly rounded and one-ulp-off values.

K2 padding (DESIGN.md section 3): the builder computes whole 8x4 blocks / 32-column pieces from TMA-zero-filled
targets, so every element up to the row pitch is written, and holds the same formula evaluated on the zero-extended
level: +0.0 where the block is all padding, and at levels 1 and 3 of an odd-width (odd-height) level above, the first
padding column (row) holds the mean of the half block the floor crop drops.  Padding ROWS of the 8x4-blocked layouts
(between h_l and the next multiple of 4) may be left unwritten: no reader loads a row >= h_l.
"""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

U_ACC = 2.0 ** -23
U_RN = 2.0 ** -24
TINY = 2.0 ** -149
SIXTEEN = {"bf16": torch.bfloat16, "fp16": torch.float16}
IN_DT = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


# =============================================================================== the checker
def bracket(ref, eps, dtype):
    """[lo, hi] (float64) of the values of `dtype` a correct rounding of ref +- eps can give."""
    wid = eps + (ref.abs() + eps) * 2.0 ** -23 + TINY
    return (ref - wid).to(dtype).double(), (ref + wid).to(dtype).double()


def in_bracket(got, ref, eps):
    lo, hi = bracket(ref, eps, got.dtype)
    g = got.double()
    return (g >= lo) & (g <= hi)


def within(got, ref, eps):
    return (got.double() - ref).abs() <= eps


RATIOS = {}


def note(kind, got, ref, eps):
    """Largest |got - ref| / eps seen per kernel (fp32 outputs), printed at the end of the module."""
    r = float(((got.double() - ref).abs() / (eps + TINY)).max())
    RATIOS[kind] = max(RATIOS.get(kind, 0.0), r)


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    if RATIOS:
        print("\nlargest |got - ref| / eps: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(RATIOS.items())))


# ------------------------------------------------------------------------------- CPU self-test of the checker
def round_bits(x, p, trunc=False):
    """float64 -> nearest (ties to even) or truncated value with p significand bits (normal range)."""
    m, e = np.frexp(x)
    s = np.ldexp(m, p)
    return np.ldexp(np.trunc(s) if trunc else np.rint(s), e - p)


@pytest.mark.parametrize("name,p", [("bf16", 8), ("fp16", 11)])
def test_bracket_checker_has_teeth(name, p):
    dt = SIXTEEN[name]
    r = np.random.default_rng(5 + p)
    x = r.choice([-1.0, 1.0], 20000) * r.uniform(1.0, 2.0, 20000) * np.exp2(r.integers(-8, 8, 20000))   # normal range
    ref = torch.from_numpy(x)
    eps = ref.abs() * 2.0 ** -20                     # an accumulation bound far below half a 16-bit ulp
    good = torch.from_numpy(round_bits(x, p))
    assert torch.equal(good.to(dt).double(), good)   # representable
    assert bool(in_bracket(good.to(dt), ref, eps).all())

    def rejects(bad):
        bad = torch.from_numpy(bad).to(dt)
        differ = bad.double() != good
        ok = in_bracket(bad, ref, eps)
        assert int(differ.sum()) > 1000
        assert float((~ok[differ]).double().mean()) > 0.97
        assert not bool(ok.all())

    rejects(round_bits(x, p, trunc=True))                                  # round toward zero
    s = 1.0 / math.sqrt(192.0)
    ref_s, eps_s = ref * s, eps * s
    good_s = torch.from_numpy(round_bits(x * s, p))
    assert bool(in_bracket(good_s.to(dt), ref_s, eps_s).all())
    twice = torch.from_numpy(round_bits(round_bits(x, p) * s, p)).to(dt)    # rounded before the scale, then again
    differ = twice.double() != good_s
    ok = in_bracket(twice, ref_s, eps_s)
    assert int(differ.sum()) > 1000 and float((~ok[differ]).double().mean()) > 0.97
    rejects(round_bits(round_bits(x, p + 2), p))                           # rounded twice through a wider format
    up = good.to(dt).view(torch.int16) + 1                                 # one ulp away from the correct rounding
    rejects(up.view(dt).double().numpy())
    # double rounding through fp32 cannot narrow the bracket: refs just above a 16-bit midpoint, within half an fp32
    # ulp, round to the midpoint in fp32 and then (ties to even) to the wrong side; with eps = 0 the correct value stays in
    mid = torch.from_numpy(round_bits(np.abs(x), p)) + torch.from_numpy(np.ldexp(np.ones_like(x), np.frexp(np.abs(x))[1] - p - 1))
    near = mid + mid * 2.0 ** -27
    want = torch.from_numpy(round_bits(near.numpy(), p))
    assert bool(in_bracket(want.to(dt), near, torch.zeros_like(near)).all())
    # fp32 outputs
    g32 = ref.float()
    assert bool(within(g32, ref, ref.abs() * 2.0 ** -24).all())
    assert not bool(within(torch.nextafter(g32, torch.full_like(g32, math.inf)), ref, ref.abs() * 2.0 ** -26).any())


# =============================================================================== K2 configuration mirror
def k2_plan(b, h, w, layout_mode, cg, sms, pooled=False):
    """Mirror of run_gemm's tile-shape and chunk-split choice (csrc/corr_gemm.cu) for one GEMM run."""
    th, tw = (h >> 2, w >> 2) if pooled else (h, w)
    blk = layout_mode != 1
    cw, cr = (16, 4) if blk else (32, 2)
    best = None
    for x in (1, 2, 4):
        tiles = -(-tw // (cw * x)) * -(-th // (cr * (4 // x)))
        cost = tiles * 100 + ((0 if x == 2 else 2 * tiles) if blk else 4 - x)
        if best is None or cost < best[0]:
            best = (cost, x)
    xb = best[1]
    ntiles = -(-tw // (cw * xb)) * -(-th // (cr * (4 // xb)))
    if cg == 0:
        cg = 3 if layout_mode == 3 and h * w > 128 else 1
    cl = 2 if cg in (2, 3) else 1
    mblk, workers = -(-(h * w) // (128 * cl)), sms // cl
    best_c, best_cost = 1, None
    for nc in range(1, min(8, ntiles) + 1):
        tpi = -(-ntiles // nc)
        real = -(-ntiles // tpi)
        cost = -(-(b * mblk * real) // workers) * (tpi + 1)
        if best_cost is None or cost < best_cost:
            best_cost, best_c = cost, real
    tpi = -(-ntiles // best_c)
    n_chunks = -(-ntiles // tpi)
    return dict(xb=xb, cg=cg, rows=128 * cl, nq=h * w, tw=tw, ntiles=ntiles, tpi=tpi, n_chunks=n_chunks,
                items=b * mblk * n_chunks, workers=workers)


# =============================================================================== GPU plumbing
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


def randn(shape, seed, dtype=torch.float32):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, device="cuda", generator=g).to(dtype)


def bits16(t):
    return t.view(torch.int16)


def pool_sum(x, pool):
    """Sequential fp32 sum over complete pool x pool blocks in (dy, dx) order, starting from 0.0f, times 1/pool^2."""
    b, c, h, w = x.shape
    ho, wo = h // pool, w // pool
    xf = x.float()[:, :, : ho * pool, : wo * pool]
    acc = torch.zeros((b, c, ho, wo), dtype=torch.float32, device=x.device)
    for dy in range(pool):
        for dx in range(pool):
            acc = acc + xf[:, :, dy::pool, dx::pool]
    return acc * (1.0 / (pool * pool))


def prep_replica(x, pool, scale, out_dtype):
    """ofb_corr_prep_to: RNE(fp32(v * scale)), v = the input (pool 1) or its pooled mean; (B, n, C) K-major."""
    b, c = x.shape[:2]
    v = x.float() if pool == 1 else pool_sum(x, pool)
    v = v * float(np.float32(scale))
    return v.reshape(b, c, -1).transpose(1, 2).to(out_dtype)


def pool_cast_replica(x, pool):
    """ofb_pool_cast_bf16 without its K padding: (B, C, nk) bf16."""
    b, c = x.shape[:2]
    return pool_sum(x, pool).reshape(b, c, -1).to(torch.bfloat16)


# =============================================================================== operand preparation
@gpu
@pytest.mark.parametrize("in_dt", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("out_dt", [torch.bfloat16, torch.float16])
def test_prep_matches_its_fp32_replica_bit_for_bit(cuda_lib, in_dt, out_dt):
    import ofb200

    for c in (64, 128, 192, 256):
        x = randn((2, c, 37, 53), c, in_dt) * 3
        for pool in (1, 2, 4, 8):
            for scale in (1.0, 1.0 / math.sqrt(c)):
                ho, wo = 37 // pool, 53 // pool
                out = torch.full((2, ho * wo, c), float("nan"), dtype=out_dt, device="cuda")
                ofb200.check(cuda_lib.ofb_corr_prep_to(ofb200.ptr(x), IN_DT[in_dt], ofb200.ptr(out), IN_DT[out_dt], 2, c, 37,
                                                       53, pool, scale, ofb200.stream_ptr()), "ofb_corr_prep_to")
                want = prep_replica(x, pool, scale, out_dt)
                assert torch.equal(bits16(out), bits16(want)), (c, pool, scale)


@gpu
@pytest.mark.parametrize("in_dt", [torch.float32, torch.bfloat16, torch.float16])
def test_pool_cast_matches_its_fp32_replica_bit_for_bit(cuda_lib, in_dt):
    import ofb200

    for (b, c, h, w) in [(2, 48, 37, 53), (1, 256, 47, 156)]:
        x = randn((b, c, h, w), h + c, in_dt) * 3
        for pool in (1, 2, 4, 8):
            nk = (h // pool) * (w // pool)
            pk = (nk + 7) // 8 * 8 + 8
            out = torch.full((b, c, pk), float("nan"), dtype=torch.bfloat16, device="cuda")
            ofb200.check(cuda_lib.ofb_pool_cast_bf16(ofb200.ptr(x), IN_DT[in_dt], ofb200.ptr(out), b, c, h, w, pool, pk,
                                                     ofb200.stream_ptr()), "ofb_pool_cast_bf16")
            assert torch.equal(bits16(out[:, :, :nk]), bits16(pool_cast_replica(x, pool))), (b, c, h, w, pool)
            assert bool((bits16(out[:, :, nk:]) == 0).all()), "K padding must be +0.0"


# =============================================================================== K2
def nan_pyramid(lib, h, w, levels, mode, dtype, q):
    import ofb200

    pyr = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    ofb200.check(lib.ofb_pyramid_layout(h, w, levels, mode, ctypes.byref(pyr), ctypes.byref(elems)), "ofb_pyramid_layout")
    pyr.dtype = ofb200.DTYPE_F16 if dtype == torch.float16 else ofb200.DTYPE_BF16
    bufs = []
    for lvl in range(levels):
        buf = torch.full((q * int(elems[lvl]),), float("nan"), dtype=dtype, device="cuda")
        bufs.append(buf)
        pyr.base[lvl] = buf.data_ptr()
    return pyr, bufs


def level_refs(a_km, t_km, qsel, th, tw, shapes, s):
    """float64 reference and eps of a level and its 2x2 mean, over the zero-extended (rows, pitch) regions `shapes`
    [(rows0, pitch0), (rows1, pitch1)] of the queries qsel."""
    bsz, n, _ = a_km.shape
    (r0, p0), (r1, p1) = shapes
    he, we = max(r0, 2 * r1, th), max(p0, 2 * p1, tw)
    qs = qsel.numel()
    ref = torch.zeros((qs, he, we), dtype=torch.float64, device="cuda")
    eps = torch.zeros_like(ref)
    qb, qp = qsel // n, qsel % n
    for bi in range(bsz):
        sel = (qb == bi).nonzero().flatten()
        if not sel.numel():
            continue
        a = a_km[bi, qp[sel]].double()
        t = t_km[bi].double()
        acc = (a @ t.T).view(-1, th, tw)
        tot = (a.abs() @ t.abs().T).view(-1, th, tw)
        m = ((a != 0).double() @ (t != 0).double().T).view(-1, th, tw)
        e = m * U_ACC * tot
        if s != 1.0:                                    # the fp16 builder scales its fp32 accumulators: one more rounding
            e = s * e + U_RN * (s * acc.abs() + s * e)
        ref[sel, :th, :tw] = s * acc
        eps[sel, :th, :tw] = e
    # 2x2 means of the fp32 values: three fp32 additions (each <= U_RN of the partial, partials <= sum |v_i|), * 0.25 exact
    v = ref[:, : 2 * r1, : 2 * p1].reshape(qs, r1, 2, p1, 2)
    ev = eps[:, : 2 * r1, : 2 * p1].reshape(qs, r1, 2, p1, 2)
    ref1 = v.sum(dim=(2, 4)) * 0.25
    e_sum = ev.sum(dim=(2, 4))
    eps1 = 0.25 * (e_sum + 3 * U_RN * (v.abs().sum(dim=(2, 4)) + e_sum))
    return (ref[:, :r0, :p0], eps[:, :r0, :p0]), (ref1, eps1)


def check_level(got, ref, eps, h, w, blocked, what):
    """got (Qs, rows, pitch) 16-bit.  Rows < h: every column in the bracket (padding columns included); padding
    that is exactly zero in the reference is +0.0.  Rows >= h (8x4-blocked layouts): in the bracket or unwritten."""
    ok = in_bracket(got, ref, eps)
    top = ok[:, :h]
    if not bool(top.all()):
        bad = (~top).nonzero()[:5].tolist()
        pytest.fail(f"{what}: {int((~top).sum())} elements outside the bracket, e.g. (query, y, x) {bad}: "
                    f"got {[float(got[i, j, k]) for i, j, k in bad]} ref {[float(ref[i, j, k]) for i, j, k in bad]}")
    pad = torch.zeros_like(ok)
    pad[:, :, w:] = True
    pad[:, h:] = True
    zero_ref = pad & (ref == 0) & (eps == 0)
    signed = (bits16(got) == bits16(torch.full((), -0.0, dtype=got.dtype, device="cuda"))) & zero_ref
    assert not bool(signed.any()), f"{what}: padding holds -0.0"
    if got.shape[1] > h:
        assert blocked, what
        assert bool((ok[:, h:] | torch.isnan(got[:, h:])).all()), f"{what}: padding rows hold a value other than the bracket or the prefill"


def k2_queries(b, h, w, full, seed):
    n = h * w
    if full:
        return torch.arange(b * n, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    edges = [0, w - 1, n - w, n - 1]
    for k in range(1, n // 128 + 1):                         # both sides of every 128- and 256-query block boundary
        if k % 8 == 0 or k * 128 + 1 >= n - 256:
            edges += [k * 128 - 1, k * 128]
    fixed = torch.tensor([bi * n + e for bi in (0, b - 1) for e in edges if 0 <= e < n], device="cuda")
    return torch.cat([fixed, torch.randint(0, b * n, (384,), device="cuda", generator=g)]).unique()


def run_k2_case(lib, monkeypatch, shape, levels, dtype, mode, cg, epi=None, xb=None, full=True, seed=0):
    import ofb200
    from ofb200.ops.corr import build_pyramid, level_images, prepare_operands

    b, c, h, w = shape
    for name, val in (("OFB_K2_EPI", epi), ("OFB_K2_XB", xb)):
        if val is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(val))
    f1 = randn(shape, 100 + seed + c)
    f2 = randn(shape, 200 + seed + h)
    q = b * h * w
    ops = prepare_operands(f1, f2, levels, dtype)
    pyr, bufs = nan_pyramid(lib, h, w, levels, mode, dtype, q)
    ofb200.check(build_pyramid(ops, pyr, b, c, h, w, dtype, cg), "K2 build")
    torch.cuda.synchronize()
    # what the operands do not carry: the fp16 builder applies 1/sqrt(C) to its fp32 accumulators
    s = float(np.float32(1.0 / math.sqrt(c))) if dtype == torch.float16 else 1.0
    qsel = k2_queries(b, h, w, full, seed)
    blocked = mode != 1
    dims = []
    for lvl in range(levels):
        rows = bufs[lvl].numel() // (q * int(pyr.row_pitch[lvl]))
        assert rows == (((h >> lvl) + 3) // 4 * 4 if blocked else h >> lvl)
        dims.append((rows, int(pyr.row_pitch[lvl])))
    for run in range(0, levels, 2):
        t_km = ops[1] if run == 0 else ops[2]
        th, tw = (h, w) if run == 0 else (h >> 2, w >> 2)
        pair = dims[run:run + 2] + ([(1, 8)] if run + 1 >= levels else [])
        (r0, e0), (r1, e1) = level_refs(ops[0], t_km, qsel, th, tw, pair, s)
        for lvl, ref, eps in ((run, r0, e0), (run + 1, r1, e1)):
            if lvl >= levels:
                continue
            img = level_images(bufs[lvl], pyr.layout, q, int(pyr.row_pitch[lvl]))[qsel]
            check_level(img, ref, eps, h >> lvl, w >> lvl, blocked,
                        f"{dtype} mode {mode} cg {cg} epi {epi} xb {xb} {shape} level {lvl}")


def k2_matrix():
    cases = []
    for dt in ("bf16", "fp16"):
        for xb in (1, 2, 4):
            for mode in (1, 2):
                for cg in (1, 2):
                    cases.append((dt, mode, cg, None, xb))
            for cg in (1, 2, 3):
                for epi in (("direct", "bulk", "pipe") if dt == "bf16" else (None,)):
                    cases.append((dt, 3, cg, epi, xb))
    return cases


MATRIX_SHAPES = [((2, 64, 19, 37), 4), ((1, 192, 15, 31), 4)]


@gpu
@pytest.mark.parametrize("dt,mode,cg,epi,xb", k2_matrix())
def test_k2_every_launch_configuration_element_by_element(cuda_lib, monkeypatch, dt, mode, cg, epi, xb):
    for shape, levels in MATRIX_SHAPES:
        run_k2_case(cuda_lib, monkeypatch, shape, levels, SIXTEEN[dt], mode, cg, epi, xb)


# shape classes: (shape, levels, full volume?)
CLASS_SHAPES = [
    ((1, 64, 8, 12), 4, True),          # 96 queries: a CTA pair's second CTA has no rows; level 3 is 1 x 1
    ((2, 64, 19, 37), 4, True),         # ragged last query block (128 and 256), pooled run 9 wide
    ((2, 128, 47, 63), 4, True),        # odd at every level, no tile dimension divides h or w, pooled run 15 wide
    ((1, 192, 16, 129), 4, True),       # few query blocks: 9 target tiles split into chunks of 2, the last one ragged
    ((16, 256, 47, 156), 4, False),     # KITTI training shape: one chunk per item, far more items than workers
    ((2, 256, 136, 240), 4, False),     # the bench shape
]
CLASS_CONFIGS = [("bf16", 3, 0), ("bf16", 3, 1), ("bf16", 3, 2), ("bf16", 3, 3), ("bf16", 2, 2), ("fp16", 3, 0),
                 ("fp16", 3, 3)]


def class_flags(shape, sms):
    """Which coverage classes one case shape falls in, for every launch mode (runs 0 and 1)."""
    b, c, h, w = shape
    flags = set()
    for cg in (1, 2, 3):
        for pooled in (False, True):
            p = k2_plan(b, h, w, 3, cg, sms, pooled=pooled)
            if not pooled and h * w <= 128 and cg in (2, 3):
                flags.add(f"nq<=128 cg{cg}")
            if not pooled and b >= 2 and h * w % p["rows"]:
                flags.add(f"ragged query block {p['rows']}")
            if pooled and p["tw"] < 16:
                flags.add("pooled narrower than a chunk")
            if p["n_chunks"] > 1 and p["ntiles"] % p["tpi"]:
                flags.add("ragged last chunk")
            if p["n_chunks"] == 1 and p["items"] > p["workers"]:
                flags.add("one chunk, items > workers")
    if all((h >> l) % 2 and (w >> l) % 2 for l in range(4)) and h % 4 and w % 16:
        flags.add("odd at every level")
    flags.add(f"C={c}")
    return flags


@gpu
def test_k2_case_list_covers_every_shape_class(cuda_lib):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    got = set().union(*(class_flags(s, sms) for s, _, _ in CLASS_SHAPES))
    want = {"nq<=128 cg2", "nq<=128 cg3", "ragged query block 128", "ragged query block 256",
            "pooled narrower than a chunk", "ragged last chunk", "one chunk, items > workers", "odd at every level",
            "C=64", "C=128", "C=192", "C=256"}
    assert want <= got, sorted(want - got)


@gpu
@pytest.mark.parametrize("dt,mode,cg", CLASS_CONFIGS)
@pytest.mark.parametrize("shape,levels,full", CLASS_SHAPES, ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else str(v))
def test_k2_shape_classes_element_by_element(cuda_lib, monkeypatch, shape, levels, full, dt, mode, cg):
    run_k2_case(cuda_lib, monkeypatch, shape, levels, SIXTEEN[dt], mode, cg, full=full, seed=7)


# =============================================================================== CUDA-core builder, 16-bit pyramid
def pool2_replica(img):
    """pool2_kernel on one stored 16-bit level (Q, h, w) -> (Q, h/2, w/2): ((s0 + s1) + s2) + s3 in fp32, / 4, RNE."""
    q, h, w = img.shape
    x = img[:, : h // 2 * 2, : w // 2 * 2].float()
    v = x[:, 0::2, 0::2] + x[:, 0::2, 1::2]
    v = v + x[:, 1::2, 0::2]
    v = v + x[:, 1::2, 1::2]
    return (v / 4.0).to(img.dtype)


@gpu
@pytest.mark.parametrize("dt", ["bf16", "fp16"])
@pytest.mark.parametrize("c", [48, 96, 160])
def test_simt_builder_16bit_pyramid(cuda_lib, dt, c):
    import ofb200
    from ofb200.ops.corr import level_images

    dtype = SIXTEEN[dt]
    b, h, w, levels = 2, 19, 37, 4
    f1, f2 = randn((b, c, h, w), 11 + c), randn((b, c, h, w), 12 + c)
    if dtype == torch.float16:                 # CorrBlock rounds the maps to fp16 first (autocast's matmul operands)
        f1, f2 = f1.half().float(), f2.half().float()
    q = b * h * w
    pyr, bufs = nan_pyramid(cuda_lib, h, w, levels, 1, dtype, q)
    s = float(np.float32(1.0 / math.sqrt(c)))
    ofb200.check(cuda_lib.ofb_corr_pyramid_simt_f32(ofb200.ptr(f1), ofb200.ptr(f2), ctypes.byref(pyr), b, c, h, w, s,
                                                    ofb200.stream_ptr()), "ofb_corr_pyramid_simt_f32")
    imgs = [level_images(bufs[l], pyr.layout, q, int(pyr.row_pitch[l]))[:, : h >> l, : w >> l] for l in range(levels)]
    a = f1.double().reshape(b, c, -1)
    t = f2.double().reshape(b, c, -1)
    acc = torch.bmm(a.transpose(1, 2), t).reshape(q, h, w)
    tot = torch.bmm(a.abs().transpose(1, 2), t.abs()).reshape(q, h, w)
    e = s * c * U_RN * tot                      # C fused multiply-adds in fp32, each one rounding <= U_RN * T
    eps = e + U_RN * (s * acc.abs() + e)        # the scale
    ok = in_bracket(imgs[0], s * acc, eps)
    assert bool(ok.all()), (int((~ok).sum()), float((imgs[0].double() - s * acc).abs().max()))
    for lvl in range(1, levels):
        assert torch.equal(bits16(imgs[lvl].contiguous()), bits16(pool2_replica(imgs[lvl - 1]))), lvl


# =============================================================================== backward GEMM
def gemm_case(lib, batch, m, n, k, accumulate=False, alpha=1.0, seed=0):
    """ofb_gemm_nt_bf16 with NaN between K and the row pitch of A and B, batch strides beyond M * lda, and a sentinel D
    with ldd > N; checks every element of D."""
    import ofb200

    lda = ldb = (k + 7) // 8 * 8 + 8
    sa, sb = m * lda + 64, n * ldb + 64
    ldd, sd = n + 4, m * (n + 4) + 8
    a_buf = torch.full((batch * sa,), float("nan"), dtype=torch.bfloat16, device="cuda")
    b_buf = torch.full((batch * sb,), float("nan"), dtype=torch.bfloat16, device="cuda")
    a = a_buf.as_strided((batch, m, k), (sa, lda, 1))
    bm = b_buf.as_strided((batch, n, k), (sb, ldb, 1))
    a.copy_(randn((batch, m, k), seed + 1, torch.bfloat16))
    bm.copy_(randn((batch, n, k), seed + 2, torch.bfloat16))
    sentinel = -12345.0
    d_buf = torch.full((batch * sd,), sentinel, dtype=torch.float32, device="cuda")
    d = d_buf.as_strided((batch, m, n), (sd, ldd, 1))
    prior = randn((batch, m, n), seed + 3) * 4 if accumulate else None
    if accumulate:
        d.copy_(prior)
    keep = d_buf.clone()
    ofb200.check(lib.ofb_gemm_nt_bf16(ofb200.ptr(a_buf), ofb200.ptr(b_buf), ofb200.ptr(d_buf), batch, m, n, k, lda, ldb, ldd,
                                      sa, sb, sd, alpha, int(accumulate), ofb200.stream_ptr()), "ofb_gemm_nt_bf16")
    inside = torch.zeros_like(d_buf, dtype=torch.bool)
    inside.as_strided((batch, m, n), (sd, ldd, 1)).fill_(True)
    assert torch.equal(d_buf[~inside], keep[~inside]), "elements outside [M) x [N) changed"
    al = float(np.float32(alpha))
    for bi in range(batch):
        a64, b64 = a[bi].double(), bm[bi].double()
        acc = a64 @ b64.T
        tot = a64.abs() @ b64.abs().T
        cnt = (a64 != 0).double() @ (b64 != 0).double().T
        e = abs(al) * cnt * U_ACC * tot
        e = e + U_RN * (abs(al) * acc.abs() + e)                       # alpha
        ref = al * acc
        if accumulate:
            e = e + U_RN * (ref.abs() + e + prior[bi].double().abs())  # + D
            ref = ref + prior[bi].double()
        got = d[bi]
        note("gemm_nt_bf16", got, ref, e)
        ok = within(got, ref, e)
        assert bool(ok.all()), (batch, m, n, k, bi, int((~ok).sum()), float((got.double() - ref).abs().max()))


@gpu
@pytest.mark.parametrize("n", [32, 64, 96, 128, 160, 192, 224, 256])
def test_gemm_nt_every_n(cuda_lib, n):
    gemm_case(cuda_lib, 2, 300, n, 1000, seed=n)                               # items below the SM count
    gemm_case(cuda_lib, 1, 129, n, 63, accumulate=True, alpha=1.0 / math.sqrt(96.0), seed=n + 1)


@gpu
@pytest.mark.parametrize("batch,m,n,k,acc", [
    (2, 12801, 96, 8, True),        # 202 items: between 1x and 2x the SM count; M % 128 = 1; K < 64
    (1, 25727, 192, 65, False),     # 201 items, M % 128 = 127, K % 64 = 1
    (16, 7332, 256, 63, False),     # 928 items (KITTI B = 16): one k-block per item
    (16, 7332, 256, 136, True),     # three k-blocks, K % 64 = 8
    (16, 7423, 128, 257, False),    # five k-blocks, K % 64 = 1, M % 128 = 127
    (3, 1000, 224, 191, True),      # K % 64 = 63
])
def test_gemm_nt_persistent_loop(cuda_lib, batch, m, n, k, acc):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    gemm_case(cuda_lib, batch, m, n, k, accumulate=acc, alpha=1.0 / math.sqrt(96.0) if acc else 1.0, seed=m + k)
    items = batch * -(-m // 128)
    if batch == 16:
        assert items > 4 * sms
    elif batch < 3:
        assert sms < items < 2 * sms


# =============================================================================== CorrBlock gradients end to end
def dense_grad_pyramid(lib, coords, weight, b, h, w, levels, radius):
    """The gradient pyramid the block's backward consumes, rebuilt through the lookup backward (fp32, tight rows)."""
    import ofb200

    desc = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    ofb200.check(lib.ofb_pyramid_layout(h, w, levels, 0, ctypes.byref(desc), ctypes.byref(elems)), "ofb_pyramid_layout")
    desc.dtype = ofb200.DTYPE_F32
    bufs = []
    for lvl in range(levels):
        buf = torch.zeros(b * h * w * int(elems[lvl]), dtype=torch.float32, device="cuda")
        bufs.append(buf)
        desc.base[lvl] = buf.data_ptr()
    ofb200.check(lib.ofb_corr_lookup_backward(ctypes.byref(desc), ofb200.ptr(coords), ofb200.ptr(weight), ofb200.DTYPE_F32,
                                              b, h, w, radius, ofb200.stream_ptr()), "ofb_corr_lookup_backward")
    return [buf.view(b, h * w, (h >> l) * (w >> l)) for l, buf in enumerate(bufs)]


E2E_CASES = [  # (b, c, h, w, levels, radius, pyramid dtype, feature-map dtype)
    (1, 64, 9, 13, 2, 3, "bf16", torch.float32),
    (2, 96, 10, 11, 3, 4, "bf16", torch.bfloat16),      # C = 96: CUDA-core forward, tensor-core backward
    (1, 192, 12, 20, 4, 4, "fp16", torch.float16),
    (2, 256, 16, 24, 1, 3, "bf16", torch.float16),
    (1, 64, 19, 37, 4, 4, "fp16", torch.float32),
    (1, 96, 15, 17, 2, 3, "fp16", torch.bfloat16),
    (2, 192, 21, 29, 3, 4, "bf16", torch.float32),
    (16, 256, 47, 156, 4, 4, "bf16", torch.float32),    # KITTI training shape, sampled
]


@gpu
@pytest.mark.parametrize("case", E2E_CASES, ids=lambda c: f"{c[0]}x{c[1]}x{c[2]}x{c[3]}-L{c[4]}r{c[5]}-{c[6]}-{str(c[7])[6:]}")
def test_corr_block_tensor_core_gradients_element_by_element(cuda_lib, case):
    from ofb200.ops.corr import CorrBlock

    b, c, h, w, levels, radius, pdt, fdt = case
    n = h * w
    f1 = randn((b, c, h, w), 31 + c, fdt).requires_grad_(True)
    f2 = randn((b, c, h, w), 32 + h, fdt).requires_grad_(True)
    base = torch.stack(torch.meshgrid(torch.arange(w, device="cuda"), torch.arange(h, device="cuda"), indexing="xy"))
    coords = (base[None].float() + 3 * randn((b, 2, h, w), 33)).contiguous()
    d = 2 * radius + 1
    weight = randn((b, levels * d * d, h, w), 34)
    blk = CorrBlock(f1, f2, num_levels=levels, radius=radius, pyramid_dtype=SIXTEEN[pdt])
    assert blk.builder == ("tcgen05" if c % 64 == 0 else "simt")
    (blk(coords) * weight).sum().backward()
    dps = dense_grad_pyramid(cuda_lib, coords, weight, b, h, w, levels, radius)
    s = float(np.float32(1.0 / math.sqrt(c)))
    f1_16 = pool_cast_replica(f1.detach(), 1)                          # (B, C, n) bf16: the B operand of d fmap2
    full = b * n <= 4096
    g = torch.Generator(device="cuda").manual_seed(35)
    pix = torch.arange(n, device="cuda") if full else torch.cat([torch.tensor([0, w - 1, n - w, n - 1], device="cuda"),
                                                                  torch.randint(0, n, (96,), device="cuda", generator=g)]).unique()
    bsel = range(b) if full else (0, b - 1)
    ys, xs = pix // w, pix % w
    for bi in bsel:
        ref1 = torch.zeros((pix.numel(), c), dtype=torch.float64, device="cuda")
        e1 = torch.zeros_like(ref1)
        s1 = torch.zeros_like(ref1)
        ref2, e2, s2 = torch.zeros_like(ref1), torch.zeros_like(ref1), torch.zeros_like(ref1)
        for lvl in range(levels):
            hl, wl = h >> lvl, w >> lvl
            dp16 = dps[lvl][bi].to(torch.bfloat16)                        # (n, n_l) = ofb_cast_bf16's output
            p_l = pool_cast_replica(f2.detach()[bi:bi + 1], 1 << lvl)[0].double()   # (C, n_l)
            # d fmap1^T rows: s * bf16(dP_l) . P_l^T, accumulated level after level into one fp32 buffer
            rows = dp16[pix].double()
            acc = rows @ p_l.T
            tot = rows.abs() @ p_l.abs().T
            cnt = (rows != 0).double() @ (p_l != 0).double().T
            e = s * cnt * U_ACC * tot
            e1 += e + U_RN * (s * acc.abs() + e)                          # tensor cores, alpha
            ref1 += s * acc
            s1 += s * tot + e
            # d pool_l(fmap2) at the pixels' level-l targets, pooled back with weight 1/4^l (complete blocks only)
            yl, xl = ys >> lvl, xs >> lvl
            inl = (yl < hl) & (xl < wl)
            tl = (yl * wl + xl).clamp(max=hl * wl - 1)
            cols = dp16[:, tl].double()                                   # (n, P)
            f1b = f1_16[bi].double()                                      # (C, n)
            acc2 = (cols.T @ f1b.T)                                       # (P, C)
            tot2 = cols.abs().T @ f1b.abs().T
            cnt2 = (cols != 0).double().T @ (f1b != 0).double().T
            wgt = inl.double()[:, None] * 0.25 ** lvl
            e = s * cnt2 * U_ACC * tot2
            e2 += wgt * (e + U_RN * (s * acc2.abs() + e))
            ref2 += wgt * s * acc2
            s2 += wgt * (s * tot2 + e)
        e1 += levels * U_RN * s1                                          # the fp32 additions across levels
        e2 += levels * U_RN * s2                                          # ofb_pool_adjoint_f32's additions
        for got_all, ref, eps, what in ((f1.grad, ref1, e1, "d fmap1"), (f2.grad, ref2, e2, "d fmap2")):
            got = got_all[bi].reshape(c, n)[:, pix].T
            if got.dtype == torch.float32:
                note("corr_block_grad", got, ref, eps)
                ok = within(got, ref, eps)
            else:
                ok = in_bracket(got, ref, eps)
            assert bool(ok.all()), (what, bi, int((~ok).sum()), float((got.double() - ref).abs().max()))
