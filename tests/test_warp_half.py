"""The warp with half-precision frames and flows: `ofb_warp`, `ofb_warp_backward` and `optical_flow.warp`.

Under CUDA autocast the reference's grid_sample runs in fp32 on the exactly widened frame and grid, so its warp of an
fp16 / bf16 frame and flow returns fp32, and the gradients it hands the inputs are the fp32 gradients rounded once to
their dtypes.  The kernels widen each 16-bit element on load and run the fp32 arithmetic, so:
  forward    warp(frame, flow, ...) == warp(frame.float(), flow.float(), ...) bit for bit (NaN at the same positions),
             mask included, for every (frame, flow) dtype pair, mode, padding x align_corners, layout, variant 0 / 1 / 3
             and pixel_flow, on the coordinate kinds of test_warp_contract.py plus fp16 inf / NaN and the fp16 range edge
  backward   d_flow == the fp32 d_flow cast to the flow's dtype, bit for bit (one store per pixel); d_frame == the fp32
             d_frame cast to the frame's dtype, bit for bit where each source element receives one non-zero
             contribution (exact integer shifts), within one ulp of the dtype elsewhere (its atomics add in a varying
             order, in fp32 too)
  surface    no fp32 copy of a half frame or flow is made or kept; the forward is one library kernel
"""
import os

import pytest
import torch

gpu = pytest.mark.gpu
F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
DTYPES = {"fp32": F32, "fp16": F16, "bf16": BF16}
PAIRS = [(a, b) for a in DTYPES for b in DTYPES if (a, b) != ("fp32", "fp32")]
PADS = ("zeros", "border", "reflection")
KINDS = ("int", "half", "edge", "straddle", "far", "huge", "nonfinite", "fp16edge")
OFB_OK, OFB_EINVAL, OFB_EUNSUPPORTED, OFB_EALIGN = 0, -1, -2, -3
BAD_DTYPES = (-1, 3, 4, 99)          # 3 = OFB_DTYPE_F64
ALLOC_GRANULE = 512                  # the CUDA caching allocator rounds every block to 512 bytes


def bits(t):
    return t.view({F32: torch.int32, BF16: torch.int16, F16: torch.int16}[t.dtype])


def assert_same(got, want, what=None):
    """Bit-identical, NaN at the same positions (NaN payloads are not compared)."""
    assert got.dtype == want.dtype and got.shape == want.shape, what
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), what
    assert torch.equal(bits(got)[~nan], bits(want)[~nan]), (what, int((bits(got) != bits(want))[~nan].sum()))


def ulp(ref, dt):
    """The spacing of dt at |ref| (subnormal spacing below the smallest normal)."""
    mant, emin = {F16: (10, -14), BF16: (7, -126)}[dt]
    r = ref.float().abs()
    _, e = torch.frexp(torch.where(r > 0, r, torch.ones_like(r)))
    e = torch.where(r > 0, e, torch.full_like(e, emin + 1))
    return torch.exp2((torch.clamp(e - 1, min=emin) - mant).double()).float()


def assert_within_ulp(got, ref32, what=None):
    """got (16-bit) within one ulp of its dtype of the fp32 reference, infinities and NaN at the same positions.  The
    reference is itself a sum of atomics in another order: its own error, a few fp32 ulps of the largest terms
    (1e-6 * max(1, |ref|_inf)), is added, which matters only where the sum cancels to far below its terms."""
    assert got.dtype != F32
    g = got.float()
    fin = torch.isfinite(ref32) & torch.isfinite(g)
    assert torch.equal(torch.isnan(g), torch.isnan(ref32)), what
    assert torch.equal(g[~fin & ~torch.isnan(g)], ref32.to(got.dtype).float()[~fin & ~torch.isnan(g)]), what
    err = (g[fin] - ref32[fin]).abs()
    slack = 1e-6 * max(1.0, float(ref32[fin].abs().max())) if bool(fin.any()) else 0.0
    assert bool((err <= ulp(ref32[fin], got.dtype) + slack).all()), (what, float(err.max()))


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


def test_entry_points_validate_arguments_without_launch(lib):
    """ofb_warp / ofb_warp_backward: OFB_EINVAL for an unknown frame or flow dtype before anything else (empty sizes and
    null pointers included); OFB_EALIGN for a 16-bit frame, flow or d_flow not 2-byte aligned; OFB_EUNSUPPORTED for
    variants 2 and 4 with a 16-bit frame or flow; with fp32 for both, the code of the _f32 form in every case.
    Nothing launches."""
    import ofb200

    fake = 1 << 20                       # 16-byte aligned, never dereferenced: every call below returns before a launch
    f32, f16, bf16 = ofb200.DTYPE_F32, ofb200.DTYPE_F16, ofb200.DTYPE_BF16
    good = (f32, f16, bf16)

    def fwd(dt_i, dt_v, frame=fake, flow=fake, out=fake, b=2, c=3, h=4, w=8, mode=0, pad=1, variant=0):
        return lib.ofb_warp(frame, dt_i, flow, dt_v, out, None, b, c, h, w, mode, pad, 0, 0, variant, 1.0, 1.0, None)

    def fwd_f32(frame=fake, flow=fake, out=fake, b=2, c=3, h=4, w=8, mode=0, pad=1, variant=0):
        return lib.ofb_warp_f32(frame, flow, out, None, b, c, h, w, mode, pad, 0, 0, variant, 1.0, 1.0, None)

    def bwd(dt_i, dt_v, frame=fake, flow=fake, d_out=fake, d_frame=fake, d_flow=fake, b=2, c=3, h=4, w=8, pad=1):
        return lib.ofb_warp_backward(frame, dt_i, flow, dt_v, d_out, d_frame, d_flow, b, c, h, w, pad, 0, 1.0, 1.0, None)

    def bwd_f32(frame=fake, flow=fake, d_out=fake, d_frame=fake, d_flow=fake, b=2, c=3, h=4, w=8, pad=1):
        return lib.ofb_warp_backward_f32(frame, flow, d_out, d_frame, d_flow, b, c, h, w, pad, 0, 1.0, 1.0, None)

    before = lib.ofb_launch_count()
    empty = ({"b": 0}, {"h": 0}, {"w": 0})
    for bad in BAD_DTYPES:
        for dts in ((bad, f32), (f32, bad), (bad, f16), (bf16, bad), (bad, bad)):
            for kw in ({},) + empty:
                assert fwd(*dts, **kw) == OFB_EINVAL, (dts, kw)
                assert fwd(*dts, frame=None, flow=None, out=None, **kw) == OFB_EINVAL, (dts, kw)
                assert bwd(*dts, **kw) == OFB_EINVAL, (dts, kw)
                assert bwd(*dts, frame=None, flow=None, d_out=None, d_frame=None, d_flow=None, **kw) == OFB_EINVAL
    fwd_cases = [({"frame": None}, OFB_EINVAL), ({"flow": None}, OFB_EINVAL), ({"out": None}, OFB_EINVAL),
                 ({"mode": 2}, OFB_EINVAL), ({"pad": 3}, OFB_EINVAL), ({"variant": 5}, OFB_EINVAL),
                 ({"b": 65536}, OFB_EUNSUPPORTED), ({"mode": 1, "variant": 3}, OFB_EUNSUPPORTED),
                 ({"frame": None, "flow": None, "out": None, "b": 0}, OFB_OK)]
    bwd_cases = [({"frame": None}, OFB_EINVAL), ({"flow": None}, OFB_EINVAL), ({"d_out": None}, OFB_EINVAL),
                 ({"pad": 3}, OFB_EINVAL), ({"d_frame": None, "d_flow": None}, OFB_OK), ({"b": 65536}, OFB_EUNSUPPORTED),
                 ({"h": 65536}, OFB_EUNSUPPORTED), ({"frame": None, "flow": None, "d_out": None, "h": 0}, OFB_OK)]
    for dt_i in good:
        for dt_v in good:
            half_i, half_v = dt_i != f32, dt_v != f32
            cases = list(fwd_cases)
            cases += [({"frame": fake + 1}, OFB_EALIGN if half_i else None),
                      ({"flow": fake + 1}, OFB_EALIGN if half_v else None)]
            for variant in (2, 4):
                cases.append(({"variant": variant}, OFB_EUNSUPPORTED if (half_i or half_v) else None))
            for kw, want in cases:
                if want is None:
                    continue
                got = fwd(dt_i, dt_v, **kw)
                assert got == want, (dt_i, dt_v, kw, got)
                if not (half_i or half_v):
                    assert fwd_f32(**kw) == got, kw
            cases = list(bwd_cases)
            if half_i:
                cases.append(({"frame": fake + 1}, OFB_EALIGN))
            if half_v:
                cases += [({"flow": fake + 1}, OFB_EALIGN), ({"d_flow": fake + 1}, OFB_EALIGN),
                          ({"flow": fake + 1, "d_flow": None}, OFB_EALIGN)]
            for kw, want in cases:
                got = bwd(dt_i, dt_v, **kw)
                assert got == want, (dt_i, dt_v, kw, got)
                if not (half_i or half_v):
                    assert bwd_f32(**kw) == got, kw
    assert lib.ofb_launch_count() == before


def test_other_dtypes_still_raise():
    """fp64 and integer frames or flows raise NotImplementedError before touching a device; so does a half frame with
    mode='bicubic'."""
    from optical_flow import warp

    x = torch.zeros(1, 3, 4, 4)
    f = torch.zeros(1, 2, 4, 4)
    for frame, flow in ((x.double(), f), (x, f.double()), (x.half(), f.double()), (x.int(), f.half())):
        with pytest.raises(NotImplementedError, match="fp32, fp16 or bf16 only"):
            warp(frame, flow)
    with pytest.raises(NotImplementedError):
        warp(x.half(), f.half(), mode="bicubic")


# =============================================================================== forward (GPU)
B, H, W = 2, 12, 16


def source_to_grid(ix, size, ac):
    ix = torch.as_tensor(ix, dtype=torch.float64)
    return 2.0 * ix / (size - 1) - 1.0 if ac else (2.0 * ix + 1.0) / size - 1.0


def make_flow(kind, ac, b=B, h=H, w=W, seed=0):
    """Normalised flow (b, 2, h, w) fp32 of one kind: those of test_warp_contract.py, plus fp16edge (components at
    +-65504, +-65520, which rounds to fp16 inf, and fp16's smallest subnormal).  Cast to a 16-bit dtype, huge and
    fp16edge hold fp16 infinities and nonfinite holds NaN and +-inf."""
    g = torch.Generator().manual_seed(seed)
    shape = (b, 2, h, w)
    mx, my = 2.0 / max(w - 1, 1), 2.0 / max(h - 1, 1)
    mul = torch.tensor([mx, my], dtype=torch.float64).view(1, 2, 1, 1)
    pick = lambda vals: torch.tensor(vals, dtype=torch.float64)[torch.randint(len(vals), shape, generator=g)]
    if kind == "int":
        px = torch.randint(-3, 4, shape, generator=g).double()
    elif kind == "half":
        px = torch.randint(-3, 3, shape, generator=g).double() + 0.5
    elif kind == "far":
        px = torch.where(torch.rand(shape, generator=g) < 0.5, -1e3, 1e3) + torch.randn(shape, generator=g).double()
    elif kind == "huge":
        return pick([1e9, -1e9, 3e9, -3e9, 0.0]).float()
    elif kind == "fp16edge":
        return pick([65504.0, -65504.0, 65520.0, -65520.0, 2.0 ** -24, -(2.0 ** -24), 0.0]).float()
    elif kind in ("edge", "straddle"):
        out = torch.empty(shape, dtype=torch.float64)
        for axis, n in ((0, w), (1, h)):
            if kind == "edge":
                targets = torch.cat([torch.tensor([-1.0, 1.0]), source_to_grid([0.0, n - 1.0], n, ac)])
            else:
                targets = source_to_grid([-0.5, -0.25, n - 0.75, n - 0.5], n, ac)
            gg = targets[torch.randint(len(targets), (b, h, w), generator=g)]
            lin = torch.linspace(-1, 1, n).double()
            lin = lin.view(1, 1, n) if axis == 0 else lin.view(1, n, 1)
            out[:, axis] = gg - lin
        return out.float()
    else:
        assert kind == "nonfinite", kind
        flow = torch.randn(shape, generator=g)
        k = torch.arange(b * h * w).view(b, h, w)
        special = torch.tensor([float("nan"), float("inf"), float("-inf")])
        flow[:, 0] = torch.where((k % 4 == 0) | (k % 4 == 2), special[(k // 4) % 3], flow[:, 0])
        flow[:, 1] = torch.where((k % 4 == 1) | (k % 4 == 2), special[(k // 12) % 3], flow[:, 1])
        return flow
    return (px * mul).float()


def make_frame(dt, c=8, b=B, h=H, w=W, seed=1):
    """(b, c, h, w) in dt with +-inf at a few pixels and, for fp16, subnormals (fp32 / bf16 get the same values, which
    are normal there)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((b, c, h, w), generator=g) - 0.5
    flat = x.view(-1)
    flat[7::97] = float("inf")
    flat[11::89] = float("-inf")
    flat[3::13] = 2.0 ** -24 * torch.randint(1, 1023, flat[3::13].shape, generator=g)
    return x.to(dt)


def run_pair(frame, flow, **kw):
    """(warp of the inputs, warp of their fp32 widening) with the same arguments."""
    from optical_flow import warp

    return warp(frame, flow, **kw), warp(frame.float(), flow.float(), **kw)


@gpu
@pytest.mark.parametrize("ac", [False, True])
@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("pair", PAIRS, ids=lambda p: f"{p[0]}-{p[1]}")
def test_forward_is_the_widened_fp32_warp(cuda_lib, pair, pad, ac):
    """Every kind, bilinear and nearest, NCHW (variants 0, 1, 3) and channels_last (C = 3 and C = 8), with and without
    the mask and pixel_flow: bit-identical to the fp32 warp of the widened inputs, mask included."""
    dt_i, dt_v = DTYPES[pair[0]], DTYPES[pair[1]]
    frame = make_frame(dt_i).cuda()
    for kind in KINDS:
        flow32 = make_flow(kind, ac, seed=KINDS.index(kind)).cuda()
        for pixel_flow in (False, True):
            flow = (flow32 * torch.tensor([(W - 1) / 2, (H - 1) / 2], device="cuda").view(1, 2, 1, 1)
                    if pixel_flow else flow32).to(dt_v)
            common = dict(padding_mode=pad, align_corners=ac, pixel_flow=pixel_flow)
            for mode in ("bilinear", "nearest"):
                variants = (0, 1, 3) if mode == "bilinear" else (0, 1)
                for variant in variants:
                    what = (kind, pixel_flow, mode, variant)
                    (got, mask), (want, want_mask) = run_pair(frame, flow, mode=mode, variant=variant,
                                                              return_mask=True, **common)
                    assert got.dtype == F32
                    assert_same(got, want, what)
                    assert torch.equal(mask, want_mask), what
                    if variant == 0:
                        got, want = run_pair(frame, flow, mode=mode, **common)
                        assert_same(got, want, what)
                for c in (3, 8):
                    cl = frame[:, :c].contiguous(memory_format=torch.channels_last)
                    assert not cl.is_contiguous()
                    got, want = run_pair(cl, flow, mode=mode, **common)
                    assert_same(got, want, what + ("channels_last", c))


@gpu
@pytest.mark.parametrize("shape", [(2, 3, 436, 1024), (8, 128, 136, 240)], ids=["C2", "feature"])
def test_forward_full_size(cuda_lib, shape):
    """A full-size C2 frame and the 8 x 128 x 136 x 240 feature shape, smooth flows: fp16 / bf16 frames with flows of
    every dtype, bit-identical to the fp32 warp of the widened inputs (the default border padding, and zeros with
    align_corners)."""
    b, c, h, w = shape
    g = torch.Generator(device="cuda").manual_seed(40)
    frame32 = torch.rand(shape, device="cuda", generator=g)
    flow32 = torch.nn.functional.interpolate(torch.randn((b, 2, h // 16, w // 16), device="cuda", generator=g) * 0.05,
                                             size=(h, w), mode="bilinear")
    for dt_i in (F16, BF16):
        for dt_v in (F32, F16, BF16):
            for kw in ({}, {"padding_mode": "zeros", "align_corners": True}):
                got, want = run_pair(frame32.to(dt_i), flow32.to(dt_v), **kw)
                assert_same(got, want, (dt_i, dt_v, kw))


@gpu
@pytest.mark.parametrize("name", ["fp16", "bf16"])
def test_forward_against_reference_under_autocast(cuda_lib, name):
    """oracle/torch_port.warp on half inputs under torch.autocast returns fp32 within the forward tolerance of the
    contract tests (1e-5 * max(1, |ref|_inf): ATen's fp32 grid_sample does not share the kernel's FMA order), for
    half and fp32 frames with a half flow."""
    from oracle import torch_port as tp
    from optical_flow import warp

    dt = DTYPES[name]
    for kind in ("int", "half", "far", "straddle"):
        for ac in (False, True):
            for pad in PADS:
                frame = (torch.rand((B, 3, H, W)) - 0.5).cuda()
                flow = make_flow(kind, ac, seed=50).cuda().to(dt)
                for fr in (frame.to(dt), frame):
                    with torch.autocast("cuda", dtype=dt):
                        ref = tp.warp(fr, flow, padding_mode=pad, align_corners=ac)
                        got = warp(fr, flow, padding_mode=pad, align_corners=ac)
                    assert ref.dtype == F32 and got.dtype == F32
                    tol = 1e-5 * max(1.0, float(ref.abs().max()))
                    assert float((got - ref).abs().max()) <= tol, (kind, ac, pad, fr.dtype)


# =============================================================================== backward (GPU)
def grads(frame, flow, wgt, frame_grad=True, flow_grad=True, cast=False, **kw):
    """(out, d frame, d flow) of sum(warp(frame, flow) * wgt); cast: through frame.float(), flow.float() first."""
    from optical_flow import warp

    f = frame.clone().requires_grad_(frame_grad)
    v = flow.clone().requires_grad_(flow_grad)
    out = warp(f.float() if cast else f, v.float() if cast else v, **kw)
    (out * wgt).sum().backward()
    return out.detach(), f.grad, v.grad


@gpu
@pytest.mark.parametrize("pair", PAIRS, ids=lambda p: f"{p[0]}-{p[1]}")
def test_backward_is_the_cast_fp32_gradient(cuda_lib, pair):
    """d_flow in the flow's dtype is the fp32 d_flow cast to it, bit for bit; d_frame in the frame's dtype within one
    ulp of the fp32 d_frame; every padding x align_corners, finite kinds, pixel_flow on and off."""
    dt_i, dt_v = DTYPES[pair[0]], DTYPES[pair[1]]
    g = torch.Generator().manual_seed(60)
    frame = torch.rand((B, 3, H, W), generator=g).to(dt_i).cuda()
    wgt = torch.randn((B, 3, H, W), generator=g).cuda()
    for kind in ("int", "half", "edge", "straddle", "far"):
        for pad in PADS:
            for ac in (False, True):
                for pixel_flow in (False, True):
                    flow = make_flow(kind, ac, seed=61).cuda()
                    if pixel_flow:
                        flow = flow * torch.tensor([(W - 1) / 2, (H - 1) / 2], device="cuda").view(1, 2, 1, 1)
                    flow = flow.to(dt_v)
                    kw = dict(padding_mode=pad, align_corners=ac, pixel_flow=pixel_flow)
                    what = (kind, pad, ac, pixel_flow)
                    out, d_frame, d_flow = grads(frame, flow, wgt, **kw)
                    ref_out, ref_frame32, ref_flow32 = grads(frame.float(), flow.float(), wgt, **kw)
                    assert_same(out, ref_out, what)
                    assert d_frame.dtype == dt_i and d_flow.dtype == dt_v
                    assert_same(d_flow, ref_flow32.to(dt_v), what)
                    if dt_i == F32:
                        tol = 1e-5 * max(1.0, float(ref_frame32.abs().max()))
                        assert float((d_frame - ref_frame32).abs().max()) <= tol, what
                    else:
                        assert_within_ulp(d_frame, ref_frame32, what)


@gpu
@pytest.mark.parametrize("pair", PAIRS, ids=lambda p: f"{p[0]}-{p[1]}")
def test_backward_exact_on_integer_shifts(cuda_lib, pair):
    """Uniform integer shifts with align_corners on a 9 x 17 frame (W - 1, H - 1 powers of two: every coordinate is an
    exact integer) under zeros padding: each source element receives at most one non-zero contribution, so d_frame in
    the frame's dtype is the fp32 d_frame cast, bit for bit, as the explicit-cast path gives it."""
    dt_i, dt_v = DTYPES[pair[0]], DTYPES[pair[1]]
    b, c, h, w = 2, 4, 9, 17
    g = torch.Generator().manual_seed(70)
    frame = torch.randn((b, c, h, w), generator=g).to(dt_i).cuda()
    wgt = torch.randn((b, c, h, w), generator=g).cuda()
    shift = torch.tensor([[2.0, -1.0], [-3.0, 2.0]]).view(b, 2, 1, 1).expand(b, 2, h, w)
    for pixel_flow in (False, True):
        flow = (shift if pixel_flow else shift * torch.tensor([2 / (w - 1), 2 / (h - 1)]).view(1, 2, 1, 1))
        flow = flow.contiguous().to(dt_v).cuda()
        kw = dict(padding_mode="zeros", align_corners=True, pixel_flow=pixel_flow)
        _, d_frame, d_flow = grads(frame, flow, wgt, **kw)
        _, ref_frame, ref_flow = grads(frame, flow, wgt, cast=True, **kw)
        assert d_frame.dtype == dt_i and ref_frame.dtype == dt_i
        assert_same(d_frame, ref_frame, pixel_flow)
        assert_same(d_flow, ref_flow, pixel_flow)


@gpu
@pytest.mark.parametrize("name", ["fp16", "bf16"])
def test_backward_gradient_selection_and_host_tensors(cuda_lib, name):
    """Only the inputs that require grad get one (frame only, flow only), with the bits of the both-inputs run;
    host inputs get host gradients in their dtypes, with the device run's d_flow bits and d_frame within one ulp."""
    dt = DTYPES[name]
    g = torch.Generator().manual_seed(80)
    frame = torch.rand((B, 3, H, W), generator=g).to(dt)
    flow = make_flow("half", False, seed=81).to(dt)
    wgt = torch.randn((B, 3, H, W), generator=g)
    out, d_frame, d_flow = grads(frame.cuda(), flow.cuda(), wgt.cuda())
    _, only_frame, none = grads(frame.cuda(), flow.cuda(), wgt.cuda(), flow_grad=False)
    assert none is None and only_frame.dtype == dt
    assert_within_ulp(only_frame, d_frame.float())
    _, none, only_flow = grads(frame.cuda(), flow.cuda(), wgt.cuda(), frame_grad=False)
    assert none is None
    assert_same(only_flow, d_flow)
    h_out, h_frame, h_flow = grads(frame, flow, wgt)
    assert h_out.device.type == "cpu" and h_frame.device.type == "cpu" and h_flow.device.type == "cpu"
    assert h_frame.dtype == dt and h_flow.dtype == dt
    assert_same(h_out, out.cpu())
    assert_same(h_flow, d_flow.cpu())
    assert_within_ulp(h_frame, d_frame.float().cpu())


@gpu
@pytest.mark.parametrize("name", ["fp16", "bf16"])
def test_integrate_with_half_flows(cuda_lib, name):
    """integrate(f0, f1, f2) with half flows promotes as the reference does (flows[k] + warp(...) is fp32) and equals
    integrate of the fp32 flows bit for bit; its backward reaches every flow in its dtype."""
    from optical_flow import integrate

    dt = DTYPES[name]
    flows = [make_flow("half", False, seed=90 + k).cuda().to(dt) for k in range(3)]
    got = integrate(*flows)
    want = integrate(*[f.float() for f in flows])
    assert got.dtype == F32
    assert_same(got, want)
    leaves = [f.clone().requires_grad_(True) for f in flows]
    integrate(*leaves).square().sum().backward()
    for f in leaves:
        assert f.grad is not None and f.grad.dtype == dt and bool(torch.isfinite(f.grad.float()).all())


# =============================================================================== memory, launches (GPU)
@gpu
@pytest.mark.parametrize("name", ["fp16", "bf16"])
def test_forward_keeps_no_fp32_copy(cuda_lib, name):
    """A forward with a half frame and flow that require grad allocates only its fp32 output and the mask: the graph
    keeps the caller's tensors, and no fp32 frame-sized buffer lives until the backward."""
    from optical_flow import warp

    dt = DTYPES[name]
    b, c, h, w = 2, 32, 136, 240
    frame = torch.rand((b, c, h, w), device="cuda").to(dt).requires_grad_(True)
    flow = (0.01 * torch.randn((b, 2, h, w), device="cuda")).to(dt).requires_grad_(True)
    warp(frame, flow, return_mask=True)                  # warm-up: module load, allocator pools
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    out, mask = warp(frame, flow, return_mask=True)
    torch.cuda.synchronize()
    new = out.numel() * out.element_size() + mask.numel() * mask.element_size()
    assert 0 <= torch.cuda.memory_allocated() - before - new < 2 * ALLOC_GRANULE
    d_frame, d_flow = torch.autograd.grad(out, (frame, flow), grad_outputs=torch.ones_like(out))
    assert d_frame.dtype == dt and d_flow.dtype == dt


@gpu
@pytest.mark.parametrize("name", ["fp16", "bf16"])
def test_forward_is_one_kernel(cuda_lib, name):
    """The forward of a half frame and flow that require grad is one library kernel, the row kernel, with no ATen cast
    or copy."""
    from optical_flow import warp
    from torch.profiler import ProfilerActivity, profile

    dt = DTYPES[name]
    frame = torch.rand((2, 3, 64, 128), device="cuda").to(dt).requires_grad_(True)
    flow = (0.01 * torch.randn((2, 2, 64, 128), device="cuda")).to(dt).requires_grad_(True)
    warp(frame, flow)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        warp(frame, flow)
        torch.cuda.synchronize()
    events = prof.events()
    kernels = [e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA]
    ops = {e.name for e in events if e.device_type == torch.autograd.DeviceType.CPU}
    assert not ops & {"aten::copy_", "aten::_to_copy"}, sorted(ops)
    assert len(kernels) == 1 and "warp_rows_kernel" in kernels[0], kernels


# =============================================================================== autocast training stand-in (GPU)
@gpu
@pytest.mark.parametrize("name", ["fp16", "bf16"])
def test_autocast_feature_warp_gradients(cuda_lib, name):
    """A conv producing features under torch.autocast, warped by a half flow, then a weighted sum and backward: the
    conv's parameter gradients and the flow gradient equal those of the explicit-cast path (warp(feat.float(),
    flow.float())) bit for bit on exact integer shifts (as test_backward_exact_on_integer_shifts).  On a general flow
    the loss and the flow gradient are still bit-identical, and the parameter gradients differ only by what one-ulp
    differences of the half d_frame (whose fp32 atomics add in a varying order) give through the conv's backward:
    within 2^-8 of their norm."""
    from optical_flow import warp

    dt = DTYPES[name]
    n, h, w = 2, 33, 65
    torch.manual_seed(100)
    conv = torch.nn.Conv2d(3, 16, 3, padding=1).cuda()
    gen = torch.Generator(device="cuda").manual_seed(101)
    img = torch.randn((n, 3, h, w), device="cuda", generator=gen)
    wgt = torch.randn((n, 16, h, w), device="cuda", generator=gen)
    shift = torch.tensor([[2.0, -1.0], [-3.0, 4.0]], device="cuda").view(n, 2, 1, 1).expand(n, 2, h, w)
    smooth = torch.randn((n, 2, h, w), device="cuda", generator=gen) * 1.5

    def step(flow_px, cast):
        conv.zero_grad(set_to_none=True)
        f = flow_px.to(dt).requires_grad_(True)
        with torch.autocast("cuda", dtype=dt):
            feat = conv(img)
            assert feat.dtype == dt
            out = warp(feat.float() if cast else feat, f.float() if cast else f, padding_mode="zeros",
                       align_corners=True, pixel_flow=True)
            loss = (out * wgt).sum()
        loss.backward()
        return loss.detach(), [p.grad.clone() for p in conv.parameters()], f.grad

    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        step(shift, False)                                                       # warm-up: cuDNN plans
        got, ref = step(shift.contiguous(), False), step(shift.contiguous(), True)
        assert torch.equal(got[0], ref[0])
        for k, (a, b) in enumerate(zip(got[1], ref[1])):
            assert a.dtype == b.dtype and torch.equal(a, b), k
        assert_same(got[2], ref[2])
        got, ref = step(smooth, False), step(smooth, True)
    finally:
        torch.backends.cudnn.deterministic = det
    assert torch.equal(got[0], ref[0])
    assert_same(got[2], ref[2])
    for k, (a, b) in enumerate(zip(got[1], ref[1])):
        assert a.dtype == b.dtype and float((a - b).norm()) <= 2.0 ** -8 * float(b.norm()), k
