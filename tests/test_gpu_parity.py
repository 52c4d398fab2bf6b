"""GPU parity tests: the CUDA path (through the Python shims -> C ABI -> sm_100a kernels) against
the CPU oracle on the same seeded inputs, against the committed golden vectors produced by the
reference itself, and -- at full BASELINE sizes -- through size-independent properties.

Tolerances (BASELINE.md section 5 / north_star):
  warp, resize, upflow8, convex upsample : max-abs <= 1e-5 * max(1, |ref|_inf)   (fp32)
  lookup floor indices / validity masks   : bit-exact
  lookup values (same pyramid)            : max-abs <= 1e-5 * max(1, |ref|_inf)
  correlation pyramid (bf16 in, fp32 acc, bf16 stored) : rel-Frobenius <= 4e-3 per level and
                                            max-abs <= 4e-2 * rms vs the fp32 reference
  EPE sum / count                         : rel <= 1e-6 / exact
  gradients (warp, upsample, sequence_loss, CorrBlock) : max-abs <= 1e-5 .. 5e-5 * |ref|_inf vs autograd through the
                                            reference (golden) / oracle/torch_port.py
"""
import os

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ofb200

    ofb200.load()     # fail loudly if the extension is missing


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().cpu().numpy()


def maxabs(a, b):
    return float(np.max(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)))) if np.size(a) else 0.0


def tol(ref, eps=1e-5):
    return eps * max(1.0, float(np.abs(ref).max()))


def rng(seed):
    return np.random.default_rng(seed)


# =============================================================================== K1 warp
def test_warp_reference_known_answers():
    """reference tests/operator/test_operator.py:6-38, CPU tensors in, exact equality."""
    from optical_flow import normalize, warp

    img = torch.tensor([[[1.0, 2.0]]]).unsqueeze(0)
    flow = torch.tensor([[[1.0, 0.0]], [[0.0, 0.0]]]).unsqueeze(0)
    assert torch.equal(warp(img, normalize(flow)), torch.tensor([[[2.0, 2.0]]]).unsqueeze(0))
    img = torch.tensor([[[1.0], [2.0]]]).unsqueeze(0)
    flow = torch.tensor([[[0.0], [0.0]], [[1.0], [0.0]]]).unsqueeze(0)
    assert torch.equal(warp(img, normalize(flow)), torch.tensor([[[2.0], [2.0]]]).unsqueeze(0))


def warp_variants(w):
    """Every bilinear NCHW kernel variant that supports this width (4 = TMA window: 16-byte row strides)."""
    return (1, 2, 3, 4) if w % 4 == 0 else (1, 2, 3)


@pytest.mark.parametrize("variant", [1, 2, 3, 4])
def test_warp_golden(golden, variant):
    from optical_flow import normalize, warp

    g = golden("warp")
    for i in range(int(g["n"])):
        frame, flow_px = T(g[f"frame{i}"]), T(g[f"flow_px{i}"])
        if variant not in warp_variants(frame.shape[-1]):
            continue
        flow = normalize(flow_px)
        assert maxabs(N(flow), g[f"flow{i}"]) == 0.0
        out = warp(frame, flow, variant=variant)
        assert out.shape == frame.shape and out.is_contiguous()
        assert maxabs(N(out), g[f"out{i}"]) <= 1e-5, (i, variant)


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
@pytest.mark.parametrize("pad", ["zeros", "border", "reflection"])
@pytest.mark.parametrize("ac", [False, True])
def test_warp_options_golden(golden, mode, pad, ac):
    from optical_flow import warp

    g = golden("warp")
    ref = g[f"opt_{mode}_{pad}_{int(ac)}"]
    for variant in ([1] if mode == "nearest" else warp_variants(g["opt_frame"].shape[-1])):
        out = N(warp(T(g["opt_frame"]), T(g["opt_flow"]), mode=mode, padding_mode=pad, align_corners=ac, variant=variant))
        if mode == "nearest":
            assert np.array_equal(out, ref)                               # index work: exact
        else:
            assert maxabs(out, ref) <= 1e-5, variant


@pytest.mark.parametrize("shape,sigma", [((2, 3, 70, 130), 5.0), ((1, 3, 368, 496), 5.0), ((3, 5, 33, 257), 20.0), ((1, 1, 16, 64), 0.3),
                                         ((1, 2, 1, 7), 0.6), ((1, 3, 5, 1), 0.6), ((2, 1, 1, 1), 0.4)])
@pytest.mark.parametrize("pad,ac", [("border", False), ("zeros", False), ("reflection", True)])
def test_warp_vs_oracle(shape, sigma, pad, ac):
    from optical_flow import normalize, warp

    r = rng(1)
    b, c, h, w = shape
    frame = r.random(shape, dtype=np.float32)
    flow_px = (sigma * r.standard_normal((b, 2, h, w))).astype(np.float32)
    flow = oracle.normalize(flow_px).astype(np.float32)
    ref, ref_mask = oracle.warp(frame, flow, padding_mode=pad, align_corners=ac, return_mask=True)
    outs = []
    for variant in warp_variants(w):
        out, mask = warp(T(frame), T(flow), padding_mode=pad, align_corners=ac, return_mask=True, variant=variant)
        assert maxabs(N(out), ref) <= 1e-5, variant
        assert np.array_equal(N(mask).astype(np.uint8), ref_mask), variant      # validity mask bit-exact
        outs.append(N(out))
    assert all(np.array_equal(outs[0], o) for o in outs[1:])                      # all kernels agree bit for bit
    # fused normalize: pixel-unit flow in, same bits out
    fused, fmask = warp(T(frame), T(flow_px), padding_mode=pad, align_corners=ac, return_mask=True, pixel_flow=True)
    assert np.array_equal(N(fused), outs[2]) and np.array_equal(N(fmask).astype(np.uint8), ref_mask)
    assert maxabs(N(normalize(T(flow_px))), flow) == 0.0


@pytest.mark.parametrize("pad", ["zeros", "border", "reflection"])
@pytest.mark.parametrize("ac", [False, True])
def test_warp_backward_golden(golden, pad, ac):
    """Backward kernel against the gradients autograd produced through the unmodified reference warp."""
    from optical_flow import warp

    g = golden("warp_grad")
    frame, flow = T(g["frame"]).requires_grad_(True), T(g["flow"]).requires_grad_(True)
    out = warp(frame, flow, padding_mode=pad, align_corners=ac)
    (out * T(g["weight"])).sum().backward()
    want_f, want_w = g[f"dframe_{pad}_{int(ac)}"], g[f"dflow_{pad}_{int(ac)}"]
    assert maxabs(N(frame.grad), want_f) <= 1e-5 * max(1.0, np.abs(want_f).max())
    assert maxabs(N(flow.grad), want_w) <= 1e-5 * max(1.0, np.abs(want_w).max())


@pytest.mark.parametrize("shape,sigma", [((2, 3, 70, 130), 5.0), ((1, 2, 368, 496), 30.0), ((3, 5, 33, 257), 2.0),
                                         ((1, 2, 1, 7), 2.0), ((1, 3, 5, 1), 2.0), ((2, 1, 2, 2), 0.5)])
@pytest.mark.parametrize("pad,ac", [("border", False), ("zeros", False), ("reflection", True), ("border", True),
                                    ("reflection", False), ("zeros", True)])
def test_warp_backward_vs_oracle(shape, sigma, pad, ac):
    """Backward kernel against autograd through oracle/torch_port.py (pinned to the reference's gradients on CPU):
    both gradients, each alone, the fused pixel-flow variant, host tensors and the forward-with-mask form."""
    from oracle import torch_port as tp
    from optical_flow import warp

    r = rng(31)
    b, c, h, w = shape
    frame = r.random(shape, dtype=np.float32)
    flow_px = (sigma * r.standard_normal((b, 2, h, w))).astype(np.float32)
    flow = oracle.normalize(flow_px).astype(np.float32)
    weight = r.standard_normal(shape).astype(np.float32)
    cf, cw = torch.from_numpy(frame).requires_grad_(True), torch.from_numpy(flow).requires_grad_(True)
    (tp.warp(cf, cw, padding_mode=pad, align_corners=ac) * torch.from_numpy(weight)).sum().backward()
    want_f, want_w = cf.grad.numpy(), cw.grad.numpy()
    tol_f, tol_w = 1e-5 * max(1.0, np.abs(want_f).max()), 2e-5 * max(1.0, np.abs(want_w).max())

    gf, gw = T(frame).requires_grad_(True), T(flow).requires_grad_(True)
    out, mask = warp(gf, gw, padding_mode=pad, align_corners=ac, return_mask=True)
    assert not mask.requires_grad
    (out * T(weight)).sum().backward()
    assert maxabs(N(gf.grad), want_f) <= tol_f and maxabs(N(gw.grad), want_w) <= tol_w
    # one gradient at a time
    only_f = T(frame).requires_grad_(True)
    (warp(only_f, T(flow), padding_mode=pad, align_corners=ac) * T(weight)).sum().backward()
    assert maxabs(N(only_f.grad), want_f) <= tol_f
    only_w = T(flow).requires_grad_(True)
    (warp(T(frame), only_w, padding_mode=pad, align_corners=ac) * T(weight)).sum().backward()
    assert torch.equal(only_w.grad, gw.grad)
    # pixel-unit flow with the fused normalize: chain rule through the 2/(W-1), 2/(H-1) factors
    px = T(flow_px).requires_grad_(True)
    (warp(T(frame), px, padding_mode=pad, align_corners=ac, pixel_flow=True) * T(weight)).sum().backward()
    fac = np.array([2.0 / max(w - 1, 1), 2.0 / max(h - 1, 1)], np.float32).reshape(1, 2, 1, 1)
    assert maxabs(N(px.grad), want_w * fac) <= tol_w * float(fac.max())
    # host tensors: staged through the GPU, gradients come back on the host
    hf = torch.from_numpy(frame).requires_grad_(True)
    (warp(hf, torch.from_numpy(flow), padding_mode=pad, align_corners=ac) * torch.from_numpy(weight)).sum().backward()
    assert not hf.grad.is_cuda and maxabs(hf.grad.numpy(), want_f) <= tol_f


@pytest.mark.parametrize("shape,size", [((2, 2, 9, 14), (20, 31)), ((1, 2, 40, 64), (17, 23)), ((3, 2, 5, 7), (5, 7)), ((1, 2, 1, 6), (3, 1))])
def test_resize_and_upflow8_backward(shape, size):
    """resize / upflow8 gradients against autograd through the ATen ops the reference calls."""
    from model import upflow8
    from optical_flow import resize
    from oracle import torch_port as tp

    r = rng(61)
    flow = r.standard_normal(shape).astype(np.float32)
    wr = r.standard_normal((shape[0], 2) + size).astype(np.float32)
    cf = torch.from_numpy(flow).requires_grad_(True)
    (tp.resize(cf, size) * torch.from_numpy(wr)).sum().backward()
    gf = T(flow).requires_grad_(True)
    (resize(gf, size=size) * T(wr)).sum().backward()
    assert maxabs(N(gf.grad), cf.grad.numpy()) <= 1e-5 * max(1.0, np.abs(cf.grad.numpy()).max())
    wu = r.standard_normal((shape[0], 2, 8 * shape[2], 8 * shape[3])).astype(np.float32)
    cf = torch.from_numpy(flow).requires_grad_(True)
    (tp.upflow8(cf) * torch.from_numpy(wu)).sum().backward()
    gf = T(flow).requires_grad_(True)
    (upflow8(gf) * T(wu)).sum().backward()
    assert maxabs(N(gf.grad), cf.grad.numpy()) <= 2e-5 * max(1.0, np.abs(cf.grad.numpy()).max())


def test_scale_normalize_backward():
    """scale / normalize / denormalize are differentiable: the gradient is the same per-channel multiply."""
    from optical_flow import denormalize, normalize, scale

    flow = torch.randn(2, 2, 9, 14, device="cuda", requires_grad=True)
    wgt = torch.randn(2, 2, 9, 14, device="cuda")
    (normalize(flow) * wgt).sum().backward()
    fac = torch.tensor([2.0 / 13, 2.0 / 8], device="cuda").view(1, 2, 1, 1)
    assert torch.allclose(flow.grad, wgt * fac, rtol=1e-6, atol=0)
    flow.grad = None
    (denormalize(scale(flow, (3.0, -0.5))) * wgt).sum().backward()
    assert torch.allclose(flow.grad, wgt * torch.tensor([3.0 * 6.5, -0.5 * 4.0], device="cuda").view(1, 2, 1, 1), rtol=1e-6, atol=0)


def test_scale_is_dtype_preserving_and_epe_takes_any_dim():
    """The reference's `scale` keeps the flow's dtype (operator.py:79-82: factor filled into a tensor of that dtype, one
    multiply) and `end_point_error` / `AverageEndPointError` take any `dim` (epe.py:41-61)."""
    from optical_flow import denormalize, normalize, scale
    from optical_flow.metrics import AverageEndPointError, end_point_error

    gen = torch.Generator(device="cuda").manual_seed(81)
    for dt in (torch.float64, torch.float16, torch.bfloat16, torch.float32):
        flow = (5 * torch.randn((2, 2, 9, 14), device="cuda", generator=gen)).to(dt)
        for fac in ((3.0, -0.5), (2.0 / 13, 2.0 / 8), (1.0 / 3.0, 7.1)):
            got = scale(flow, fac)
            ref_fac = torch.stack([torch.empty_like(flow[:, 0]).fill_(fac[0]), torch.empty_like(flow[:, 1]).fill_(fac[1])], dim=1)
            assert got.dtype == dt and torch.equal(got, flow * ref_fac), (dt, fac)
        assert normalize(flow).dtype == dt and denormalize(flow).dtype == dt
    with pytest.raises(NotImplementedError):
        scale(torch.zeros((1, 2, 3, 3), dtype=torch.int32, device="cuda"), 2)
    # EPE along other dims: (B, H, W, 2) with dim=-1 and (2, B, H, W) with dim=0 equal the (B, 2, H, W) result
    pred = torch.randn((3, 2, 11, 17), device="cuda", generator=gen)
    tgt = torch.randn((3, 2, 11, 17), device="cuda", generator=gen)
    want_map = end_point_error(pred, tgt, reduce=False)
    want = end_point_error(pred, tgt)
    assert maxabs(N(want_map), oracle.end_point_error(N(pred), N(tgt), reduce=False)) <= 1e-6
    for dim, perm in ((-1, (0, 2, 3, 1)), (0, (1, 0, 2, 3)), (2, (0, 2, 1, 3))):
        p2, t2 = pred.permute(perm).contiguous(), tgt.permute(perm).contiguous()
        got_map = end_point_error(p2, t2, dim=dim, reduce=False)
        inv = [x for x in perm if x != 1]                         # the map keeps the remaining dims in permuted order
        assert torch.equal(got_map, want_map.permute([sorted(inv).index(x) for x in inv]))
        assert abs(float(end_point_error(p2, t2, dim=dim)) - float(want)) <= 1e-6 * float(want)
        m = AverageEndPointError(dim=dim)
        m.update(p2, t2)
        assert abs(float(m.compute()) - float(want)) <= 1e-6 * float(want)
    with pytest.raises(NotImplementedError):
        end_point_error(torch.zeros(2, 3, 4, 4, device="cuda"), torch.zeros(2, 3, 4, 4, device="cuda"))


def test_warp_channels_last_and_host_tensors():
    from optical_flow import warp

    r = rng(2)
    frame = r.random((2, 8, 40, 72), dtype=np.float32)
    flow = oracle.normalize((4 * r.standard_normal((2, 2, 40, 72))).astype(np.float32)).astype(np.float32)
    ref = oracle.warp(frame, flow)
    cl = T(frame).contiguous(memory_format=torch.channels_last)
    out = warp(cl, T(flow))
    assert out.is_contiguous() and maxabs(N(out), ref) <= 1e-5
    cl3 = T(frame[:, :3].copy()).contiguous(memory_format=torch.channels_last)
    assert maxabs(N(warp(cl3, T(flow))), oracle.warp(frame[:, :3].copy(), flow)) <= 1e-5
    host = warp(torch.from_numpy(frame), torch.from_numpy(flow))       # staged through the GPU, returned on host
    assert not host.is_cuda and maxabs(host.numpy(), ref) <= 1e-5


def test_warp_full_size_properties():
    """C2 32x3x436x1024: zero flow is the reference's non-identity resample; an integer pixel shift
    (in the reference's W/(W-1) units) reproduces shifted pixels exactly; linear in the frame."""
    from optical_flow import warp

    b, c, h, w = 32, 3, 436, 1024
    gen = torch.Generator(device="cuda").manual_seed(7)
    frame = torch.rand((b, c, h, w), device="cuda", generator=gen)
    flow = torch.randn((b, 2, h, w), device="cuda", generator=gen) * 0.01
    o1 = warp(frame, flow, variant=1)
    o2 = warp(frame, flow, variant=2)
    o3 = warp(frame, flow, variant=3)
    o4 = warp(frame, flow, variant=4)
    assert torch.equal(o1, o2) and torch.equal(o1, o3) and torch.equal(o1, o4)
    big = torch.randn((b, 2, h, w), device="cuda", generator=gen) * 0.05   # +-25 px: most taps leave the TMA window
    assert torch.equal(warp(frame, big, variant=3), warp(frame, big, variant=4))
    frame2 = torch.rand((b, c, h, w), device="cuda", generator=gen)
    lin = warp(frame + frame2, flow)
    assert float((lin - (o1 + warp(frame2, flow))).abs().max()) <= 4e-6
    # align_corners=True + zero flow is the identity
    ident = warp(frame, torch.zeros_like(flow), align_corners=True)
    assert float((ident - frame).abs().max()) <= 2e-4       # ulp(1023) = 6e-5 on the source coordinate
    out, mask = warp(frame, torch.zeros_like(flow), return_mask=True)
    assert int(mask.sum()) == b * (h - 2) * (w - 2)          # border pixels sit exactly on -1 / +1


@pytest.mark.parametrize("shape", [(2, 3, 436, 1024), (1, 3, 1088, 1920)])
@pytest.mark.parametrize("pad", ["border", "zeros"])
def test_warp_full_size_vs_oracle(shape, pad):
    """BASELINE shapes against the CPU oracle: the Sintel frame of C2 (two of its 32 images) and the 1088x1920
    frame of C5 -- W = 1920 is where a non-fused coordinate un-normalisation is 5.8e-5 off (SURVEY.md "five things"
    #3; reference operator.py:30).  Every kernel variant, pixel-unit flow both ways (normalize() then warp, and the
    fused pixel_flow path), validity mask bit-exact, values <= 1e-5."""
    from optical_flow import normalize, warp

    r = rng(31)
    b, c, h, w = shape
    frame = r.random(shape, dtype=np.float32)
    flow_px = (5.0 * r.standard_normal((b, 2, h, w))).astype(np.float32)
    flow_px[:, :, : h // 8] *= 12.0                      # a band of +-60 px flows: taps far outside any staged window
    flow = oracle.normalize(flow_px).astype(np.float32)
    ref, ref_mask = oracle.warp(frame, flow, padding_mode=pad, return_mask=True)
    frame_d, flow_d = T(frame), T(flow)
    assert maxabs(N(normalize(T(flow_px))), flow) == 0.0
    first = None
    for variant in warp_variants(w):
        out, mask = warp(frame_d, flow_d, padding_mode=pad, return_mask=True, variant=variant)
        out = N(out)
        assert maxabs(out, ref) <= 1e-5, variant
        assert np.array_equal(N(mask).astype(np.uint8), ref_mask), variant
        if first is None:
            first = out
        else:
            assert np.array_equal(first, out), variant
    fused, fmask = warp(frame_d, T(flow_px), padding_mode=pad, return_mask=True, pixel_flow=True)
    assert np.array_equal(N(fused), first) and np.array_equal(N(fmask).astype(np.uint8), ref_mask)


def test_warp_errors():
    from optical_flow import resize, scale, warp

    x = torch.zeros(1, 3, 4, 4, device="cuda")
    f = torch.zeros(1, 2, 4, 4, device="cuda")
    with pytest.raises(NotImplementedError):
        warp(x, f, mode="bicubic")
    with pytest.raises(NotImplementedError):
        warp(x.double(), f.double())
    with pytest.raises(RuntimeError):
        warp(x, torch.zeros(1, 2, 5, 4, device="cuda"))
    with pytest.raises(AssertionError):
        scale(torch.zeros(1, 3, 4, 4, device="cuda"), 2.0)
    with pytest.raises(AssertionError):
        scale(f, (1.0, 2.0, 3.0))
    with pytest.raises(NotImplementedError):                      # nearest has no backward kernel
        warp(x.requires_grad_(), f, mode="nearest").sum().backward()
    with pytest.raises(NotImplementedError):                      # forward-only ops say so instead of returning zeros
        from model import bilinear_sampler
        bilinear_sampler(x.detach().clone().requires_grad_(), torch.zeros(1, 2, 2, 2, device="cuda")).sum().backward()


def test_warp_grid_and_integrate_golden(golden):
    from optical_flow import integrate
    from optical_flow.operator.operator import warp_grid

    g = golden("warp")
    grid = warp_grid(T(g["flow0"]).permute(0, 2, 3, 1).contiguous())
    assert maxabs(N(grid), g["grid0"]) == 0.0
    r = golden("resize")
    out = integrate(T(r["int_f1"]), T(r["int_f2"]), T(r["int_f3"]))
    assert maxabs(N(out), r["integrate"]) <= 1e-5
    with pytest.raises(AssertionError):
        integrate(T(r["int_f1"]))


# =============================================================================== K4a resize / scale
FLOW22 = [[[1.0, 3.0], [2.0, 4.0]], [[-1.0, -2.0], [-3.0, -4.0]]]


def test_resize_reference_known_answers():
    """reference tests/operator/test_operator.py:41-132 (exact, CPU tensors)."""
    from optical_flow import resize, scale

    flow = torch.tensor(FLOW22).unsqueeze(0)
    s = scale(flow, 2)
    assert torch.equal(s[:, 0], 2 * flow[:, 0]) and torch.equal(s[:, 1], 2 * flow[:, 1])
    s = scale(flow, (3, -1))
    assert torch.equal(s[:, 0], 3 * flow[:, 0]) and torch.equal(s[:, 1], -1 * flow[:, 1])
    x = torch.tensor([[1.0, 1.5, 2.5, 3.0], [1.25, 1.75, 2.75, 3.25], [1.75, 2.25, 3.25, 3.75], [2.0, 2.5, 3.5, 4.0]])
    y = torch.tensor([[-1.0, -1.25, -1.75, -2.0], [-1.5, -1.75, -2.25, -2.5], [-2.5, -2.75, -3.25, -3.5], [-3.0, -3.25, -3.75, -4.0]])
    assert torch.equal(resize(flow, scale_factor=2), 2 * torch.stack([x, y]).unsqueeze(0))
    assert torch.equal(resize(flow, size=(4, 2)), torch.stack([x[:, [0, 3]], 2 * y[:, [0, 3]]]).unsqueeze(0))
    assert torch.equal(resize(flow, size=(2, 4)), torch.stack([2 * x[[0, 3]], y[[0, 3]]]).unsqueeze(0))


def test_resize_golden(golden):
    from model.utils import upflow8
    from optical_flow import denormalize, normalize, resize, scale

    g = golden("resize")
    flow = T(g["flow"])
    assert maxabs(N(scale(flow, 2)), g["scale_2"]) == 0.0
    assert maxabs(N(scale(flow, (3, -1))), g["scale_3_m1"]) == 0.0
    assert maxabs(N(normalize(flow)), g["normalize"]) == 0.0
    assert maxabs(N(denormalize(flow)), g["denormalize"]) == 0.0
    for key, kw in [("resize_20_31", dict(size=(20, 31))), ("resize_4_5", dict(size=(4, 5))),
                    ("resize_9_13", dict(size=(9, 13))), ("resize_sf2", dict(scale_factor=2)),
                    ("resize_sf2p5", dict(scale_factor=2.5)), ("resize_sf0p5", dict(scale_factor=0.5))]:
        out = N(resize(flow, **kw))
        assert out.shape == g[key].shape, key
        assert maxabs(out, g[key]) <= tol(g[key]), key
    assert maxabs(N(upflow8(T(g["small"]))), g["upflow8"]) <= tol(g["upflow8"])
    with pytest.raises(NotImplementedError):
        resize(flow, scale_factor=2, mode="bicubic")


def test_resize_vs_oracle_kitti():
    from model.utils import upflow8
    from optical_flow import resize

    r = rng(3)
    flow = (4 * r.standard_normal((4, 2, 47, 156))).astype(np.float32)
    ref = oracle.upflow8(flow)
    assert maxabs(N(upflow8(T(flow))), ref) <= tol(ref)
    ref = oracle.resize(flow, size=(375, 1242))
    assert maxabs(N(resize(T(flow), size=(375, 1242))), ref) <= tol(ref)


# =============================================================================== K4b convex upsample
def test_upsample_flow_golden(golden):
    from model.raft import RAFT

    g = golden("upsample_epe")
    out = N(RAFT.upsample_flow(T(g["flow"]), T(g["mask"])))
    assert out.shape == g["up"].shape
    assert maxabs(out, g["up"]) <= tol(g["up"])


def test_upsample_flow_vs_oracle_kitti_shape():
    from model.raft import upsample_flow

    r = rng(4)
    flow = (1.0 * r.standard_normal((2, 2, 47, 156))).astype(np.float32)
    mask = (2.0 * r.standard_normal((2, 576, 47, 156))).astype(np.float32)
    ref = oracle.upsample_flow(flow, mask)
    out = N(upsample_flow(T(flow), T(mask)))
    assert maxabs(out, ref) <= tol(ref)


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_upsample_flow_half_precision_mask(dt):
    """`precision: 16` callers hand the mask head's half-precision output to upsample_flow (reference raft.py:73-85; its
    softmax autocasts to fp32).  Same result as the fp32 kernel on the same (rounded) logits, <= 1e-5 against the oracle
    on them; differentiable with respect to the flow and -- through an fp32 cast -- the mask."""
    from model.raft import upsample_flow

    r = rng(95)
    n, h, w = 2, 19, 37
    flow = (2 * r.standard_normal((n, 2, h, w))).astype(np.float32)
    mask_h = T((2 * r.standard_normal((n, 576, h, w))).astype(np.float32)).to(dt)
    mask_f = mask_h.float()
    got = upsample_flow(T(flow), mask_h)
    assert got.dtype == torch.float32 and torch.equal(got, upsample_flow(T(flow), mask_f))
    ref = oracle.upsample_flow(flow, N(mask_f))
    assert maxabs(N(got), ref) <= tol(ref)
    # gradients: flow only (half mask stays half), and flow + mask (mask cast to fp32 inside)
    f1 = T(flow).requires_grad_(True)
    wgt = torch.randn((n, 2, 8 * h, 8 * w), device="cuda")
    (upsample_flow(f1, mask_h) * wgt).sum().backward()
    f2, m2 = T(flow).requires_grad_(True), mask_f.clone().requires_grad_(True)
    (upsample_flow(f2, m2) * wgt).sum().backward()
    close = lambda a, b: float((a - b).abs().max()) <= 1e-5 * float(b.abs().max())   # d flow is summed with atomics
    assert close(f1.grad, f2.grad)
    m3 = mask_h.clone().requires_grad_(True)
    f3 = T(flow).requires_grad_(True)
    (upsample_flow(f3, m3) * wgt).sum().backward()
    assert m3.grad.dtype == dt and close(f3.grad, f2.grad)
    assert float((m3.grad.float() - m2.grad).abs().max()) <= 1e-2 * float(m2.grad.abs().max())


def test_upsample_flow_properties_full_size():
    """C4 16x(2+576)x47x156: a constant flow stays constant (softmax weights sum to 1) away from the
    zero-padded border; a one-hot mask (logit +50 on the centre tap) gives nearest upsampling * 8."""
    from model.raft import upsample_flow

    n, h, w = 16, 47, 156
    gen = torch.Generator(device="cuda").manual_seed(5)
    mask = torch.randn((n, 576, h, w), device="cuda", generator=gen)
    flow = torch.full((n, 2, h, w), 0.75, device="cuda")
    out = upsample_flow(flow, mask)
    inner = out[:, :, 8:-8, 8:-8]
    assert float((inner - 6.0).abs().max()) <= 1e-5
    flow = torch.randn((n, 2, h, w), device="cuda", generator=gen)
    onehot = torch.zeros((n, 576, h, w), device="cuda")
    onehot.view(n, 9, 64, h, w)[:, 4] = 50.0
    out = upsample_flow(flow, onehot)
    ref = 8 * flow.repeat_interleave(8, dim=2).repeat_interleave(8, dim=3)
    assert float((out - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


# =============================================================================== K4c EPE
def test_epe_golden(golden):
    from optical_flow.metrics import AverageEndPointError, end_point_error

    g = golden("upsample_epe")
    pred, target, valid = T(g["pred"]), T(g["target"]), T(g["valid"])
    assert maxabs(N(end_point_error(pred, target, reduce=False)), g["epe_map"]) <= 1e-6
    assert abs(float(end_point_error(pred, target)) - float(g["epe_mean"])) <= 1e-6
    m = AverageEndPointError()
    m.update(pred, target, valid)
    assert int(m.total) == int(g["m1_total"])
    assert abs(float(m.sum_epe) - float(g["m1_sum"])) <= 1e-5 * float(g["m1_sum"])
    m.update(pred * 0.5, target)
    assert int(m.total) == int(g["m2_total"])
    assert abs(float(m.compute()) - float(g["m2_compute"])) <= 1e-5


def test_outlier_ratio_golden_and_oracle(golden):
    """OutlierRatio (reference optical_flow/metrics/f1.py): golden vectors from the reference, then a KITTI-size
    case against the oracle; counts are exact."""
    from optical_flow.metrics import OutlierRatio

    g = golden("upsample_epe")
    m = OutlierRatio(abs_threshold=3.0, rel_threshold=0.05)
    m.update(T(g["f1_pred"]), T(g["f1_target"]), T(g["valid"]))
    assert float(m.sum_outliers) == float(g["f1a_sum"]) and int(m.total) == int(g["f1a_total"])
    m.update(T(g["f1_pred"]), T(g["f1_target"]))
    assert float(m.sum_outliers) == float(g["f1b_sum"]) and int(m.total) == int(g["f1b_total"])
    assert abs(float(m.compute()) - float(g["f1b_compute"])) <= 1e-6
    r = rng(17)
    target = (6 * r.standard_normal((4, 2, 376, 1248))).astype(np.float32)
    pred = (target + 2.5 * r.standard_normal(target.shape)).astype(np.float32)
    valid = (r.random((4, 376, 1248)) > 0.2).astype(np.float32)
    m = OutlierRatio()
    m.update(T(pred), T(target), T(valid))
    s, n = oracle.outlier_sum_count(pred, target, valid)
    assert float(m._acc[0]) == s and int(m.total) == n


def _gemm_nt(a, b, accumulate_into=None, alpha=1.0):
    """ofb_gemm_nt_bf16 on (batch, M, lda) / (batch, N, ldb) bf16 tensors whose logical K is the last argument."""
    import ofb200
    (a_t, k), (b_t, _) = a, b
    batch, m, lda = a_t.shape
    n, ldb = b_t.shape[1], b_t.shape[2]
    d = accumulate_into if accumulate_into is not None else torch.empty((batch, m, n), device="cuda")
    ofb200.check(ofb200.load().ofb_gemm_nt_bf16(ofb200.ptr(a_t), ofb200.ptr(b_t), ofb200.ptr(d), batch, m, n, k, lda, ldb, n,
                                                m * lda, n * ldb, m * n, alpha, int(accumulate_into is not None),
                                                ofb200.stream_ptr()), "ofb_gemm_nt_bf16")
    return d


@pytest.mark.parametrize("batch,m,n,k", [(1, 128, 256, 64), (2, 300, 256, 1000), (1, 7332, 256, 7332), (3, 130, 64, 72),
                                         (1, 33, 128, 2040), (2, 1, 32, 8)])
def test_gemm_nt_bf16_and_cast(batch, m, n, k):
    """The backward GEMM kernel (tcgen05, long K) and the cast / transpose that feeds it, against torch: ragged M and
    K tails, every N the kernel accepts, accumulation, alpha."""
    import ofb200

    gen = torch.Generator(device="cuda").manual_seed(m * 7 + k)
    src = torch.randn((batch, m, k), device="cuda", generator=gen)           # fp32 "gradient level": rows x cols
    bop = torch.randn((batch, n, k), device="cuda", generator=gen)
    pk, pm = (k + 7) // 8 * 8, (m + 7) // 8 * 8
    a16 = torch.full((batch, m, pk), 7.0, dtype=torch.bfloat16, device="cuda")
    a16_t = torch.full((batch, k, pm), 7.0, dtype=torch.bfloat16, device="cuda")
    ofb200.check(ofb200.load().ofb_cast_bf16(ofb200.ptr(src), ofb200.ptr(a16), ofb200.ptr(a16_t), batch, m, k, pk, pm,
                                             ofb200.stream_ptr()), "ofb_cast_bf16")
    want16 = src.to(torch.bfloat16)
    assert torch.equal(a16[:, :, :k], want16) and bool((a16[:, :, k:] == 0).all())
    assert torch.equal(a16_t[:, :, :m], want16.transpose(1, 2)) and bool((a16_t[:, :, m:] == 0).all())
    b16 = torch.zeros((batch, n, pk), dtype=torch.bfloat16, device="cuda")
    b16[:, :, :k] = bop.to(torch.bfloat16)
    ref = torch.bmm(a16[:, :, :k].float(), b16[:, :, :k].float().transpose(1, 2))
    got = _gemm_nt((a16, k), (b16, k))
    tol = 2e-3 * float(ref.abs().max()) + 1e-4
    assert float((got - ref).abs().max()) <= tol
    got2 = _gemm_nt((a16, k), (b16, k), accumulate_into=got.clone(), alpha=0.5)
    assert float((got2 - 1.5 * ref).abs().max()) <= 1.5 * tol
    # the transposed operand: D2 = src^T . X^T with X (n x m)
    x16 = torch.zeros((batch, n, pm), dtype=torch.bfloat16, device="cuda")
    x16[:, :, :m] = torch.randn((batch, n, m), device="cuda", generator=gen).to(torch.bfloat16)
    ref2 = torch.bmm(a16_t[:, :, :m].float(), x16[:, :, :m].float().transpose(1, 2))
    got3 = _gemm_nt((a16_t, m), (x16, m))
    assert float((got3 - ref2).abs().max()) <= 2e-3 * float(ref2.abs().max()) + 1e-4


@pytest.mark.parametrize("shape", [(2, 64, 47, 156), (1, 32, 9, 13), (3, 40, 17, 30)])
def test_pool_cast_and_pool_adjoint_kernels(shape):
    """The two passes around CorrBlock's backward GEMMs against the ATen ops they replace: the pooled K-padded bf16
    operand = bf16(avg_pool2d chain of corr.py:52-54), and the pooling adjoint = autograd through that chain (with the
    (B, N_l, C) -> (B, C, h, w) layout change fused)."""
    import ctypes

    import ofb200

    b, c, h, w = shape
    gen = torch.Generator(device="cuda").manual_seed(97)
    f = torch.randn(shape, device="cuda", generator=gen)
    lib, st = ofb200.load(), ofb200.stream_ptr()
    levels = [f]
    for _ in range(3):
        if min(levels[-1].shape[-2:]) < 2:
            break
        levels.append(torch.nn.functional.avg_pool2d(levels[-1], 2, stride=2))
    for lvl, ref in enumerate(levels):
        nl = ref.shape[-2] * ref.shape[-1]
        pk = (nl + 7) // 8 * 8 + 8
        for src in (f, f.bfloat16(), f.half()):
            out = torch.full((b, c, pk), 7.0, dtype=torch.bfloat16, device="cuda")
            ofb200.check(lib.ofb_pool_cast_bf16(ofb200.ptr(src), {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}[src.dtype],
                                                ofb200.ptr(out), b, c, h, w, 1 << lvl, pk, st), "ofb_pool_cast_bf16")
            want = src.float()
            for _ in range(lvl):
                want = torch.nn.functional.avg_pool2d(want, 2, stride=2)
            assert float(out[:, :, nl:].abs().max()) == 0.0                           # padding is written, as zeros
            got = out[:, :, :nl].float().view(b, c, *ref.shape[-2:])
            assert float((got - want).abs().max()) <= 2 ** -8 * float(want.abs().max()) + 1e-6   # one bf16 rounding
    # adjoint
    leaf = f.clone().requires_grad_(True)
    chain, cur = [leaf], leaf
    for _ in range(len(levels) - 1):
        cur = torch.nn.functional.avg_pool2d(cur, 2, stride=2)
        chain.append(cur)
    grads = [torch.randn_like(t) for t in chain]
    want = torch.autograd.grad(chain, leaf, grads)[0]
    d_bnc = [g.reshape(b, c, -1).transpose(1, 2).contiguous() for g in grads]          # (B, N_l, C), the GEMMs' layout
    ptrs = (ctypes.c_void_p * ofb200.MAX_LEVELS)(*[t.data_ptr() for t in d_bnc])
    got = torch.empty_like(f)
    ofb200.check(lib.ofb_pool_adjoint_f32(ptrs, ofb200.ptr(got), b, c, h, w, len(d_bnc), st), "ofb_pool_adjoint_f32")
    assert float((got - want).abs().max()) <= 1e-5 * float(want.abs().max())
    one = (ctypes.c_void_p * ofb200.MAX_LEVELS)(d_bnc[0].data_ptr())
    ofb200.check(lib.ofb_pool_adjoint_f32(one, ofb200.ptr(got), b, c, h, w, 1, st), "ofb_pool_adjoint_f32")
    assert torch.equal(got, grads[0])                                                  # levels = 1: the transpose alone


def test_corr_block_backward(golden):
    """CorrBlock gradients with respect to the feature maps: the reference's autograd result (two lookups into one
    pyramid, tests/golden/corr_grad.npz), then other shapes / radii / level counts against autograd through
    oracle/torch_port.py.  The gradients do not depend on the stored (bf16) volume, only on the fp32 feature maps
    and the lookup weights, so the tolerance is fp32 summation noise."""
    from model import CorrBlock
    from oracle import torch_port as tp

    g = golden("corr_grad")
    relnorm = lambda got, want: float(np.linalg.norm(got - want) / np.linalg.norm(want))
    for dt in (torch.float32, torch.bfloat16):
        f1, f2 = T(g["fmap1"]).requires_grad_(True), T(g["fmap2"]).requires_grad_(True)
        blk = CorrBlock(f1, f2, num_levels=4, radius=4, pyramid_dtype=dt)
        total = sum((blk(T(g[f"coords{k}"])) * T(g[f"weight{k}"])).sum() for k in range(2))
        total.backward()
        for got, want in ((N(f1.grad), g["dfmap1"]), (N(f2.grad), g["dfmap2"])):
            if dt == torch.float32:                                   # fp32 pyramid -> fp32 GEMMs: fp32 summation noise
                assert maxabs(got, want) <= 2e-5 * np.abs(want).max()
            else:                                                     # default: bf16 operands on the tensor cores
                assert relnorm(got, want) <= 6e-3
        assert blk._grad.dpyr is None                                 # the gradient pyramid is freed once consumed

    r = rng(51)
    for (b, c, h, w, lv, rad, dt) in [(1, 64, 9, 13, 2, 3, torch.bfloat16), (2, 32, 8, 20, 3, 2, torch.float32),
                                      (1, 128, 24, 40, 4, 4, torch.bfloat16), (2, 48, 10, 11, 2, 4, torch.bfloat16)]:
        a1 = r.standard_normal((b, c, h, w)).astype(np.float32)
        a2 = r.standard_normal((b, c, h, w)).astype(np.float32)
        base = np.stack(np.meshgrid(np.arange(w), np.arange(h)), 0)[None].astype(np.float32)
        cs = [(base + 2.5 * r.standard_normal((b, 2, h, w))).astype(np.float32) for _ in range(3)]
        ws = [r.standard_normal((b, lv * (2 * rad + 1) ** 2, h, w)).astype(np.float32) for _ in range(3)]
        c1, c2 = torch.from_numpy(a1).requires_grad_(True), torch.from_numpy(a2).requires_grad_(True)
        pyr = tp.corr_pyramid(c1, c2, lv)
        sum((tp.corr_lookup(pyr, torch.from_numpy(x), rad) * torch.from_numpy(y)).sum() for x, y in zip(cs, ws)).backward()
        g1, g2 = T(a1).requires_grad_(True), T(a2).requires_grad_(True)
        blk = CorrBlock(g1, g2, num_levels=lv, radius=rad, pyramid_dtype=dt)
        sum((blk(T(x)) * T(y)).sum() for x, y in zip(cs, ws)).backward()
        for got, want in ((N(g1.grad), c1.grad.numpy()), (N(g2.grad), c2.grad.numpy())):
            if dt == torch.float32 or c % 32:                         # fp32 GEMMs (also the fallback when C % 32 != 0)
                assert maxabs(got, want) <= 5e-5 * np.abs(want).max(), (b, c, h, w, lv, rad)
            else:
                assert relnorm(got, want) <= 6e-3, (b, c, h, w, lv, rad)
    # bf16 GEMM operands (fp32 accumulation) for the feature-map gradients: mixed-precision tolerance
    os.environ["OFB200_BWD_GEMM"] = "bf16"
    try:
        h1, h2 = T(a1).requires_grad_(True), T(a2).requires_grad_(True)
        blk = CorrBlock(h1, h2, num_levels=lv, radius=rad)
        sum((blk(T(x)) * T(y)).sum() for x, y in zip(cs, ws)).backward()
    finally:
        del os.environ["OFB200_BWD_GEMM"]
    for got, want in ((h1.grad, g1.grad), (h2.grad, g2.grad)):
        assert float((got - want).norm() / want.norm()) <= 1e-2
    # only fmap2 requires grad; no_grad lookups stay forward-only
    g2 = T(a2).requires_grad_(True)
    blk = CorrBlock(T(a1), g2, num_levels=lv, radius=rad)
    with torch.no_grad():
        assert not blk(T(cs[0])).requires_grad
    (blk(T(cs[0])) * T(ws[0])).sum().backward()
    assert g2.grad is not None and bool(torch.isfinite(g2.grad).all())


def test_corr_block_autograd_holds_no_block_and_drops_stale_gradients():
    """ADVICE r1: (1) the autograd contexts keep a small state object, not the CorrBlock -- dropping the last user
    reference frees the block (and its multi-GB pyramid) at once, without the cyclic collector; (2) a gradient pyramid
    left behind by another backward pass (one that raised, or never reached the handle node) is not accumulated into."""
    import gc
    import weakref

    from model import CorrBlock
    from model.utils import coords_grid

    gen = torch.Generator(device="cuda").manual_seed(61)
    f1 = torch.randn((1, 64, 16, 24), device="cuda", generator=gen, requires_grad=True)
    f2 = torch.randn((1, 64, 16, 24), device="cuda", generator=gen, requires_grad=True)
    coords = coords_grid(1, 16, 24).cuda() + torch.randn((1, 2, 16, 24), device="cuda", generator=gen)
    wgt = torch.randn((1, 324, 16, 24), device="cuda", generator=gen)
    gc.collect()
    gc.disable()
    try:
        blk = CorrBlock(f1, f2)
        out = blk(coords)
        alive = weakref.ref(blk)
        del blk
        assert alive() is None, "CorrBlock is kept alive by its own autograd graph (reference cycle)"
        (out * wgt).sum().backward()                       # the graph still works without the block
    finally:
        gc.enable()
    clean1, clean2 = f1.grad.clone(), f2.grad.clone()
    f1.grad = f2.grad = None
    blk = CorrBlock(f1, f2)
    out = blk(coords)
    st = blk._grad
    st.alloc()
    for t in st.dpyr:
        t.fill_(7.0)                                       # what an aborted backward would have left behind
    st.task = -12345
    (out * wgt).sum().backward()
    assert torch.equal(f1.grad, clean1) and torch.equal(f2.grad, clean2)
    assert st.dpyr is None


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
def test_corr_block_half_precision_feature_maps(dt):
    """`precision: 16` callers (reference methods/raft/config/train/default.yaml:20): the prep kernel reads bf16 / fp16
    maps directly.  Same bits as handing over the same values in fp32 (1/sqrt(C) is a power of two for C = 64, 256)."""
    from model.corr import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(62)
    for (b, c, h, w) in [(2, 256, 24, 40), (1, 64, 19, 37)]:
        f1 = torch.randn((b, c, h, w), device="cuda", generator=gen).to(dt)
        f2 = torch.randn((b, c, h, w), device="cuda", generator=gen).to(dt)
        half = CorrBlock(f1, f2)
        full = CorrBlock(f1.float(), f2.float())
        assert half.builder == "tcgen05"
        for a, bb in zip(half.corr_pyramid, full.corr_pyramid):
            assert torch.equal(a, bb)
        ref = oracle.corr_pyramid(N(f1.float()), N(f2.float()), 4)
        for (rel, mx) in _pyr_errors(half.corr_pyramid, ref):
            assert rel <= 4e-3 and mx <= 4e-2


@pytest.mark.parametrize("shape", [(2, 256, 47, 156), (1, 128, 24, 40), (1, 64, 19, 37), (1, 256, 136, 240)])
def test_corr_block_on_demand_matches_materialised(shape):
    """SURVEY.md 8f row 4: lookups without a materialised volume.  Same floor indices by construction (same coordinate
    code path as the oracle-checked kernels); values against (1) the fp32 CUDA-core pyramid + lookup -- the reference's
    arithmetic -- within the bf16-operand tolerance (rel-Frobenius <= 4e-3: here only the OPERANDS are bf16, the
    correlation values themselves stay fp32), (2) the CPU oracle on the small shapes; zeros outside the image, finite
    output for non-finite coordinates."""
    from model.corr import CorrBlock
    from model.utils import coords_grid

    b, c, h, w = shape
    gen = torch.Generator(device="cuda").manual_seed(71)
    f1 = torch.randn(shape, device="cuda", generator=gen)
    f2 = torch.randn(shape, device="cuda", generator=gen)
    od = CorrBlock(f1, f2, on_demand=True)
    assert od.builder == "on_demand"
    base = coords_grid(b, h, w).cuda()
    kinds = {"int": base, "noise": base + 4 * torch.randn((b, 2, h, w), device="cuda", generator=gen),
             "far": base + 60 * torch.randn((b, 2, h, w), device="cuda", generator=gen)}
    nonf = base.clone()
    nonf[:, 0, ::3, ::5] = 1e9
    nonf[:, 1, 1::4, 2::7] = float("nan")
    kinds["nonfinite"] = nonf
    ref_blk = CorrBlock(f1, f2, pyramid_dtype=torch.float32, builder="simt") if h * w <= 8000 else CorrBlock(f1, f2)
    for kind, coords in kinds.items():
        got = od(coords)
        assert got.shape == (b, 324, h, w) and torch.isfinite(got).all(), kind
        want = ref_blk(coords)
        rel = float((got - want).norm() / want.norm().clamp_min(1e-6))
        assert rel <= (4e-3 if h * w <= 8000 else 6e-3), (kind, rel)
    if h * w <= 1000:
        f1r, f2r = oracle.round_bf16(N(f1) / np.float32(np.sqrt(c))) * np.float32(np.sqrt(c)), N(f2)
        pyr = oracle.corr_pyramid(N(f1), N(f2), 4)
        ref = oracle.corr_lookup(pyr, N(kinds["noise"]), 4)
        got = N(od(kinds["noise"]))
        assert np.linalg.norm(got - ref) / np.linalg.norm(ref) <= 4e-3
    with pytest.raises(NotImplementedError):
        od.corr_pyramid
    with pytest.raises(NotImplementedError):
        od(base, return_index=True)
    with pytest.raises(NotImplementedError):
        CorrBlock(f1.requires_grad_(), f2, on_demand=True)


def test_empty_batches():
    """Zero-size inputs: every op returns an empty tensor of the right shape (as the ATen ops behind the reference
    do) instead of tripping over the null data pointer of an empty tensor; metrics stay untouched."""
    from model import CorrBlock, bilinear_sampler, upflow8, upsample_flow
    from optical_flow import normalize, resize, warp
    from optical_flow.metrics import AverageEndPointError, OutlierRatio

    z = lambda *s: torch.zeros(s, device="cuda")
    out, mask = warp(z(0, 3, 8, 8), z(0, 2, 8, 8), return_mask=True)
    assert out.shape == (0, 3, 8, 8) and mask.shape == (0, 8, 8)
    assert warp(z(2, 0, 8, 8), z(2, 2, 8, 8)).shape == (2, 0, 8, 8)
    assert normalize(z(0, 2, 4, 4)).shape == (0, 2, 4, 4)
    assert resize(z(0, 2, 4, 4), size=(8, 6)).shape == (0, 2, 8, 6)
    assert upflow8(z(0, 2, 3, 3)).shape == (0, 2, 24, 24)
    assert upsample_flow(z(0, 2, 3, 3), z(0, 576, 3, 3)).shape == (0, 2, 24, 24)
    assert bilinear_sampler(z(0, 1, 5, 5), z(0, 3, 3, 2)).shape == (0, 1, 3, 3)
    blk = CorrBlock(z(0, 64, 8, 8), z(0, 64, 8, 8), num_levels=2, radius=4)
    assert blk(z(0, 2, 8, 8)).shape == (0, 2 * 81, 8, 8)
    for m in (AverageEndPointError(), OutlierRatio()):
        m.update(z(0, 2, 4, 4), z(0, 2, 4, 4))
        m.update(torch.ones(1, 2, 4, 4, device="cuda"), z(1, 2, 4, 4))
        assert int(m.total) == 16
    # gradients through an empty warp are empty too
    fr = z(0, 3, 8, 8).requires_grad_(True)
    warp(fr, z(0, 2, 8, 8)).sum().backward()
    assert fr.grad.shape == (0, 3, 8, 8)


def test_corr_block_4k_indexing():
    """2160 x 3840 frames (270 x 480 features): level 0 of ONE pair holds 1.68e10 elements (33.6 GB in bf16), past
    2^32 -- every offset in the builder and the lookup has to be 64-bit.  Sampled queries from the start, the
    middle and the very end of the volume are checked against direct dot products."""
    free, _ = torch.cuda.mem_get_info()
    if free < 70e9:
        pytest.skip("needs ~50 GB of free device memory")
    from model import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(11)
    c, h, w = 64, 270, 480
    n = h * w
    f1 = torch.randn((1, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((1, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2, num_levels=4, radius=4)
    ys, xs = torch.meshgrid(torch.arange(h, device="cuda"), torch.arange(w, device="cuda"), indexing="ij")
    coords = torch.stack((xs, ys), 0).float()[None].contiguous()            # integer coordinates: taps are exact samples
    out = blk(coords)                                                       # (1, 324, h, w)
    assert bool(torch.isfinite(out).all())
    a = (f1[0].reshape(c, n) / 8.0).to(torch.bfloat16).float()              # operands as the builder rounds them (1/sqrt(64))
    b2 = f2[0].reshape(c, n).to(torch.bfloat16).float()
    for q in (0, 1, n // 2 + 7, n - w - 3, n - 1):
        qy, qx = divmod(q, w)
        row = (a[:, q] @ b2).view(h, w)                                      # level-0 slice of query q, fp32
        for i, j in ((4, 4), (0, 0), (8, 8), (2, 7)):                        # channel i*9 + j samples (x + i - 4, y + j - 4)
            x, y = qx + i - 4, qy + j - 4
            want = float(row[y, x]) if 0 <= x < w and 0 <= y < h else 0.0
            got = float(out[0, i * 9 + j, qy, qx])
            assert abs(got - want) <= 2e-2 * max(1.0, abs(want)), (q, i, j, got, want)
    del blk, out
    torch.cuda.empty_cache()


def test_host_staged_runner_arena_matches_dict():
    """HostStagedRunner: a pinned pair-major arena (one DMA per micro-batch) gives the same EPE as the per-field
    staging of a dict of pinned tensors and as the device-resident pass, for micro-batches of 1 and 2 pairs."""
    from ofb200.runner import FIELDS, HostStagedRunner, PairArena, hot_path
    from optical_flow.metrics import AverageEndPointError

    gen = torch.Generator(device="cuda").manual_seed(3)
    pairs, c, h, w, iters = 3, 64, 16, 24, 2
    rn = lambda *s: torch.randn(s, device="cuda", generator=gen)
    base = torch.stack(torch.meshgrid(torch.arange(w, device="cuda"), torch.arange(h, device="cuda"), indexing="xy"), 0).float()
    batch = {"fmap1": rn(pairs, c, h, w), "fmap2": rn(pairs, c, h, w),
             "coords": (base[None, None] + 2 * rn(iters, pairs, 2, h, w)).contiguous(), "flow_lo": rn(pairs, 2, h, w),
             "up_mask": rn(pairs, 576, h, w), "frame": torch.rand((pairs, 3, 8 * h, 8 * w), device="cuda", generator=gen),
             "target": 5 * rn(pairs, 2, 8 * h, 8 * w), "valid": (torch.rand((pairs, 8 * h, 8 * w), device="cuda", generator=gen) > 0.2).float()}
    m0 = AverageEndPointError()
    hot_path(batch, m0)
    want = float(m0.compute())
    arena = PairArena(pairs, PairArena.shapes_of(batch), pin=True).fill(batch)
    for k in FIELDS:
        assert arena[k].shape == batch[k].shape and torch.equal(arena[k], batch[k].cpu())
    host = {k: batch[k].cpu().pin_memory() for k in FIELDS}
    for micro in (1, 2):
        for src in (arena, host):
            runner = HostStagedRunner(torch.device("cuda", 0), micro)
            got = runner.run(src, AverageEndPointError())
            assert abs(got - want) <= 1e-6 * abs(want), (micro, type(src).__name__)
            assert runner.h2d_bytes >= sum(batch[k].numel() * 4 for k in FIELDS) and runner.d2h_bytes == 16
        # cross-step prefetch: three steps, the next step's first micro-batch staged during the current one
        runner = HostStagedRunner(torch.device("cuda", 0), micro)
        other = PairArena(pairs, PairArena.shapes_of(batch), pin=True).fill(batch)
        for nxt in (arena, other, None):                       # same arena, a different arena, none
            got = runner.run(arena if nxt is not other else arena, AverageEndPointError(), prefetch=nxt)
            assert abs(got - want) <= 1e-6 * abs(want), (micro, "prefetch")
        assert abs(runner.run(other, AverageEndPointError()) - want) <= 1e-6 * abs(want)   # a stale prefetch is ignored
    # half-precision feature maps in the arena: fewer bytes over the link, same result (the EPE does not depend on them;
    # the lookup output must match a device-resident pass on the same rounded maps)
    half = PairArena(pairs, PairArena.shapes_of(batch), pin=True,
                     dtypes={"fmap1": torch.bfloat16, "fmap2": torch.bfloat16}).fill(batch)
    runner = HostStagedRunner(torch.device("cuda", 0), 1)
    got = runner.run(half, AverageEndPointError())
    assert abs(got - want) <= 1e-6 * abs(want)
    assert runner.h2d_bytes < sum(batch[k].numel() * 4 for k in FIELDS)
    ref_out = hot_path(dict(batch, fmap1=batch["fmap1"].bfloat16().float(), fmap2=batch["fmap2"].bfloat16().float()),
                       AverageEndPointError())["corr"]
    got_out = hot_path({k: half[k].cuda() for k in FIELDS}, AverageEndPointError())["corr"]
    assert torch.equal(ref_out, got_out)


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_training_step_composes(dt):
    """A miniature RAFT training step through every differentiable op of the package -- CorrBlock, three lookups
    feeding a small update head, convex upsampling, sequence_loss, and a photometric warp term -- against the same
    computation through oracle/torch_port.py on the CPU: loss value and the gradients of the feature maps, the
    head's weights and the image."""
    from model import CorrBlock, sequence_loss, upsample_flow
    from optical_flow import warp
    from oracle import torch_port as tp

    torch.manual_seed(5)
    b, c, h, w, iters = 1, 64, 16, 24, 3
    f1, f2 = torch.randn(b, c, h, w), torch.randn(b, c, h, w)
    img = torch.rand(b, 3, 8 * h, 8 * w)
    head_flow = 0.02 * torch.randn(2, 4 * 81, 1, 1)
    head_mask = 0.05 * torch.randn(576, 4 * 81, 1, 1)
    gt = 4.0 * torch.randn(b, 2, 8 * h, 8 * w)
    valid = (torch.rand(b, 8 * h, 8 * w) > 0.2).float()
    base = torch.stack(torch.meshgrid(torch.arange(w), torch.arange(h), indexing="xy"), 0)[None].float()

    def step(dev, corr_fn, lookup_fn, up_fn, loss_fn, warp_fn, norm_fn):
        leaves = [t.clone().to(dev).requires_grad_(True) for t in (f1, f2, head_flow, head_mask, img)]
        a1, a2, wf, wm, im = leaves
        state = corr_fn(a1, a2)
        coords = base.to(dev).clone()
        preds = []
        for _ in range(iters):
            corr = lookup_fn(state, coords.detach())
            delta = torch.nn.functional.conv2d(corr, wf)
            mask = torch.nn.functional.conv2d(corr, wm)
            coords = coords + delta
            preds.append(up_fn(coords - base.to(dev), mask))
        loss, _ = loss_fn(preds, gt.to(dev), valid.to(dev))
        photo = ((warp_fn(im, norm_fn(preds[-1])) - im) ** 2).mean()
        total = loss + 0.1 * photo
        total.backward()
        return float(total.detach()), [t.grad.cpu() for t in leaves]

    want_loss, want = step("cpu", lambda x, y: tp.corr_pyramid(x, y, 4), lambda p, cds: tp.corr_lookup(p, cds, 4),
                           tp.upsample_flow, lambda p, g_, v: tp.sequence_loss(p, g_, v), tp.warp, tp.normalize)
    from optical_flow import normalize
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                  # the head's convolutions are torch glue: keep them fp32
    try:
        got_loss, got = step("cuda", lambda x, y: CorrBlock(x, y, num_levels=4, radius=4, pyramid_dtype=dt),
                             lambda blk, cds: blk(cds), upsample_flow, lambda p, g_, v: sequence_loss(p, g_, v), warp, normalize)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    # fp32 volume: fp32 noise through three refinement iterations; bf16 volume (the product default): the loss agrees
    # to mixed-precision accuracy, the gradients to a few per cent (sign(pred - gt) flips where the two runs' flows
    # straddle the ground truth)
    tol_loss, tol_grad = (1e-6, 2e-5) if dt == torch.float32 else (2e-3, 5e-2)   # measured: 7e-8 / 1.5e-6 and 3e-6 / 1.6e-2
    assert abs(got_loss - want_loss) <= tol_loss * abs(want_loss)
    for name, gg, ww in zip(("fmap1", "fmap2", "head_flow", "head_mask", "image"), got, want):
        rel = float((gg - ww).norm() / ww.norm())
        print(f"training step [{dt}] {name}: rel grad diff {rel:.2e}; loss diff {abs(got_loss - want_loss) / abs(want_loss):.2e}")
        assert rel <= tol_grad, (name, rel)


def test_upsample_and_sequence_loss_backward(golden):
    """Backward kernels of the convex upsampling and of sequence_loss: the reference's own autograd gradients
    (tests/golden/raft_grad.npz), then larger cases against autograd through oracle/torch_port.py."""
    from model import sequence_loss, upsample_flow
    from oracle import torch_port as tp

    g = golden("raft_grad")
    flow, mask = T(g["up_flow"]).requires_grad_(True), T(g["up_mask"]).requires_grad_(True)
    (upsample_flow(flow, mask) * T(g["up_weight"])).sum().backward()
    assert maxabs(N(flow.grad), g["up_dflow"]) <= 1e-5 * np.abs(g["up_dflow"]).max()
    assert maxabs(N(mask.grad), g["up_dmask"]) <= 1e-5 * max(1.0, np.abs(g["up_dmask"]).max())
    preds = [T(g["sl_preds"][i]).requires_grad_(True) for i in range(g["sl_preds"].shape[0])]
    loss, _ = sequence_loss(preds, T(g["sl_gt"]), T(g["sl_valid"]), gamma=0.8)
    (3.0 * loss).backward()
    for i, p in enumerate(preds):
        assert maxabs(N(p.grad), g["sl_dpreds"][i]) <= 1e-6 * np.abs(g["sl_dpreds"]).max(), i

    r = rng(41)
    for (n, h, w) in [(2, 47, 156), (1, 3, 5), (3, 17, 33)]:
        fl = r.standard_normal((n, 2, h, w)).astype(np.float32)
        mk = (2 * r.standard_normal((n, 576, h, w))).astype(np.float32)
        wt = r.standard_normal((n, 2, 8 * h, 8 * w)).astype(np.float32)
        cf, cm = torch.from_numpy(fl).requires_grad_(True), torch.from_numpy(mk).requires_grad_(True)
        (tp.upsample_flow(cf, cm) * torch.from_numpy(wt)).sum().backward()
        gf, gm = T(fl).requires_grad_(True), T(mk).requires_grad_(True)
        (upsample_flow(gf, gm) * T(wt)).sum().backward()
        assert maxabs(N(gf.grad), cf.grad.numpy()) <= 2e-5 * np.abs(cf.grad.numpy()).max(), (n, h, w)
        assert maxabs(N(gm.grad), cm.grad.numpy()) <= 2e-5 * max(1.0, np.abs(cm.grad.numpy()).max()), (n, h, w)
        only = T(mk).requires_grad_(True)                       # mask gradient alone
        (upsample_flow(T(fl), only) * T(wt)).sum().backward()
        assert torch.equal(only.grad, gm.grad)
    for (b, h, w, n) in [(2, 376, 1248, 12), (3, 11, 17, 3)]:
        gt = (8 * r.standard_normal((b, 2, h, w))).astype(np.float32)
        valid = (r.random((b, h, w)) > 0.3).astype(np.float32)
        ps = [(gt + (4.0 / (i + 1)) * r.standard_normal(gt.shape)).astype(np.float32) for i in range(n)]
        cp = [torch.from_numpy(p).requires_grad_(True) for p in ps]
        tp.sequence_loss(cp, torch.from_numpy(gt), torch.from_numpy(valid), gamma=0.85)[0].backward()
        gp = [T(p).requires_grad_(i != 1) for i, p in enumerate(ps)]   # one prediction without grad
        sequence_loss(gp, T(gt), T(valid), gamma=0.85)[0].backward()
        for i in range(n):
            if i == 1:
                assert gp[i].grad is None
            else:
                assert maxabs(N(gp[i].grad), cp[i].grad.numpy()) <= 1e-6 * np.abs(cp[i].grad.numpy()).max(), (b, h, w, i)


def test_sequence_loss_golden_and_oracle(golden):
    """sequence_loss (reference methods/raft/model/raft.py:231-260) as one fused reduction: the reference's own
    outputs, then a 12-prediction KITTI-size case against the oracle (counts exact, loss to 1e-6 relative), a
    non-vectorisable size, host tensors and the error paths."""
    from model import sequence_loss

    g = golden("sequence_loss")
    preds = [T(g["preds"][i]) for i in range(g["preds"].shape[0])]
    loss, m = sequence_loss(preds, T(g["gt"]), T(g["valid"]))
    assert loss.is_cuda and loss.dtype == torch.float32 and loss.dim() == 0
    assert abs(float(loss) - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    assert [m["1px"], m["3px"], m["5px"]] == pytest.approx(list(g["m"]), abs=1e-7)
    loss2, m2 = sequence_loss(preds[:1], T(g["gt"]), T(g["valid"]), gamma=0.5, max_flow=10.0)
    assert abs(float(loss2) - float(g["loss2"])) <= 1e-5 * abs(float(g["loss2"]))
    assert [m2["1px"], m2["3px"], m2["5px"]] == pytest.approx(list(g["m2"]), abs=1e-7)
    host_loss, host_m = sequence_loss([p.cpu() for p in preds], T(g["gt"]).cpu(), T(g["valid"]).cpu())
    assert not host_loss.is_cuda and float(host_loss) == float(loss) and host_m == m

    r = rng(23)
    for (b, h, w, n) in [(2, 376, 1248, 12), (3, 11, 17, 3), (1, 5, 7, 24)]:
        gt = (8 * r.standard_normal((b, 2, h, w))).astype(np.float32)
        gt[0, :, 0, 0] = 1000.0
        valid = (r.random((b, h, w)) > 0.3).astype(np.float32)
        ps = [(gt + (4.0 / (i + 1)) * r.standard_normal(gt.shape)).astype(np.float32) for i in range(n)]
        want, wm, extra = oracle.sequence_loss(ps, gt, valid, gamma=0.85, max_flow=400.0)
        got, gm = sequence_loss([T(p) for p in ps], T(gt), T(valid), gamma=0.85, max_flow=400.0)
        assert abs(float(got) - want) <= 1e-6 * abs(want), (b, h, w, n)
        assert gm == pytest.approx(wm, abs=1e-12), (b, h, w, n)                     # ratios of exact counts
    # nothing kept: the reference's mean() of an empty selection is NaN
    _, em = sequence_loss([T(ps[0])], T(gt), T(np.zeros_like(valid)))
    assert all(np.isnan(v) for v in em.values())
    with pytest.raises(NotImplementedError):
        sequence_loss([T(ps[0])] * 25, T(gt), T(valid))
    with pytest.raises(RuntimeError):
        sequence_loss([T(ps[0])[:, :, :-1]], T(gt), T(valid))


@pytest.mark.parametrize("shape", [(16, 376, 1248), (3, 11, 17), (2, 1088, 1920)])
def test_epe_vs_oracle(shape):
    from optical_flow.metrics import AverageEndPointError

    b, h, w = shape
    r = rng(6)
    pred = (3 * r.standard_normal((b, 2, h, w))).astype(np.float32)
    target = (pred + r.standard_normal((b, 2, h, w))).astype(np.float32)
    valid = (r.random((b, h, w)) > 0.1).astype(np.float32)
    s, c = oracle.epe_sum_count(pred, target, valid)
    m = AverageEndPointError()
    m.update(T(pred), T(target), T(valid))
    assert int(m.total) == c                                        # exact count
    assert abs(float(m._acc[0]) - s) <= 1e-6 * s                    # rel <= 1e-6 on the sum
    s2, c2 = oracle.epe_sum_count(pred, target)
    m2 = AverageEndPointError()
    m2.update(T(pred), T(target))
    assert int(m2.total) == c2 == b * h * w and abs(float(m2._acc[0]) - s2) <= 1e-6 * s2


# =============================================================================== K3 lookup
def _pyramid_from_numpy(levels, dtype, blocked=False):
    """Wrap oracle-built fp32 levels into a CorrBlock-like object that owns padded device buffers
    (padded rows, or the 8x4-blocked layout of include/ofb200.h)."""
    import ofb200
    from ofb200.ops.corr import level_buffer

    q = levels[0].shape[0]
    pyr = ofb200.Pyramid()
    pyr.levels = len(levels)
    pyr.dtype = ofb200.DTYPE_BF16 if dtype == torch.bfloat16 else ofb200.DTYPE_F32
    pyr.layout = (ofb200.LAYOUT_QMINOR8X4 if blocked == "qminor" else ofb200.LAYOUT_BLOCK8X4) if blocked else ofb200.LAYOUT_ROWS
    # fp32 rows kernel: pads must never be read (NaN).  bf16 register-tile kernel: pads may be read but must
    # not reach the output -- the contract is "finite", so poison them with a huge finite value
    poison = float("nan") if dtype == torch.float32 and not blocked else 3.0e38
    bufs = []
    for l, lv in enumerate(levels):
        hl, wl = lv.shape[-2:]
        pitch, rows = ((wl + 7) & ~7, (hl + 3) & ~3) if blocked else ((wl + 15) & ~15, hl)
        img = torch.full((q, rows, pitch), poison, dtype=dtype, device="cuda")
        img[:, :hl, :wl] = T(lv[:, 0]).to(dtype)
        buf = level_buffer(img, pyr.layout)
        bufs.append(buf)
        pyr.base[l] = buf.data_ptr()
        pyr.q_stride[l] = 32 if blocked == "qminor" else rows * pitch
        pyr.row_pitch[l] = pitch
        pyr.lvl_h[l] = hl
        pyr.lvl_w[l] = wl
    return pyr, bufs


def _lookup(pyr, coords, radius, levels):
    import ctypes

    import ofb200

    b, _, h, w = coords.shape
    d = 2 * radius + 1
    out = torch.empty((b, levels * d * d, h, w), device="cuda")
    idx = torch.empty((b * h * w, levels, 2, d), dtype=torch.int32, device="cuda")
    valid = torch.empty((b * h * w, levels, d * d), dtype=torch.uint8, device="cuda")
    rc = ofb200.load().ofb_corr_lookup(ctypes.byref(pyr), ofb200.ptr(coords), ofb200.ptr(out), ofb200.ptr(idx),
                                       ofb200.ptr(valid), b, h, w, radius, ofb200.stream_ptr())
    ofb200.check(rc, "ofb_corr_lookup")
    return N(out), N(idx), N(valid)


@pytest.mark.parametrize("name", ["int", "noise", "far", "half"])
def test_lookup_golden_fp32_pyramid(golden, name):
    g = golden("corr")
    if name in ("int", "noise"):
        levels = [g[f"pyr{i}"] for i in range(4)]
    else:
        levels = [g[f"b2_pyr{i}"] for i in range(3)]
    pyr, bufs = _pyramid_from_numpy(levels, torch.float32)
    out, idx, valid = _lookup(pyr, T(g[f"coords_{name}"]), 4, len(levels))
    ref = g[f"lookup_{name}"]
    assert maxabs(out, ref) <= tol(ref)
    assert np.array_equal(idx, g[f"idx_{name}"])                  # bit-exact
    assert np.array_equal(valid, g[f"valid_{name}"])              # bit-exact


def test_lookup_golden_odd_radius3(golden):
    g = golden("corr")
    levels = [g[f"odd_pyr{i}"] for i in range(3)]
    pyr, bufs = _pyramid_from_numpy(levels, torch.float32)
    out, idx, valid = _lookup(pyr, T(g["odd_coords"]), 3, 3)
    assert maxabs(out, g["odd_lookup"]) <= tol(g["odd_lookup"])
    assert np.array_equal(idx, g["odd_idx"]) and np.array_equal(valid, g["odd_valid"])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, "bf16_blocked", "bf16_qminor"])
@pytest.mark.parametrize("hw", [(47, 156), (55, 128), (24, 40)])
def test_lookup_vs_oracle(dtype, hw):
    """Seeded pyramid + coords (integer coords, sub-pixel noise, far out of range) vs the oracle."""
    blocked = {"bf16_blocked": True, "bf16_qminor": "qminor"}.get(dtype, False)
    if blocked:
        dtype = torch.bfloat16
    h, w = hw
    b = 1
    r = rng(8)
    q = b * h * w
    levels = [r.standard_normal((q, 1, h >> l, w >> l)).astype(np.float32) for l in range(4)]
    if dtype == torch.bfloat16:
        levels = [oracle.round_bf16(lv) for lv in levels]          # same stored values on both sides
    pyr, bufs = _pyramid_from_numpy(levels, dtype, blocked)
    grid = oracle.coords_grid(b, h, w)
    for kind in ("int", "noise", "far", "half", "edge", "nonfinite"):
        coords = grid.copy()
        if kind == "noise":
            coords = (coords + 4 * r.standard_normal(coords.shape)).astype(np.float32)
        if kind == "far":
            coords = (coords + 60 * r.standard_normal(coords.shape)).astype(np.float32)
        if kind == "half":
            coords = (coords + 0.5).astype(np.float32)
        if kind == "edge":          # windows hanging over every border, plus exact integers at the corners
            coords[:, 0] = np.where(coords[:, 0] < w / 2, coords[:, 0] * 0.1 - 3.0, w - 1 + coords[:, 0] * 0.05)
            coords[:, 1] = np.where(coords[:, 1] < h / 2, -2.0, h + 1.25)
            coords = coords.astype(np.float32)
        if kind == "nonfinite":
            coords = coords.astype(np.float32)
            coords[:, 0, ::3, ::5] = np.float32(1e9)
            coords[:, 1, 1::4, 2::7] = np.float32(-3e7)
        ref, ridx, rvalid = oracle.corr_lookup(levels, coords, radius=4, return_index=True)
        out, idx, valid = _lookup(pyr, T(coords), 4, 4)
        assert np.array_equal(idx, ridx), kind
        assert np.array_equal(valid, rvalid), kind
        assert maxabs(out, ref) <= tol(ref), kind


def test_bilinear_sampler_golden(golden):
    from model.utils import bilinear_sampler, coords_grid

    g = golden("corr")
    out, m = bilinear_sampler(T(g["bs_img"]), T(g["bs_pts"]), mask=True)
    assert maxabs(N(out), g["bs_out"]) <= 1e-5
    assert np.array_equal(N(m), g["bs_mask"])
    assert np.array_equal(coords_grid(1, 16, 16).numpy(), g["coords_grid"])


# =============================================================================== K2 pyramid
def _pyr_errors(levels_gpu, levels_ref):
    errs = []
    for got, ref in zip(levels_gpu, levels_ref):
        got = N(got.float())
        assert got.shape == ref.shape
        rel = float(np.linalg.norm(got - ref) / np.linalg.norm(ref))
        mx = float(np.abs(got - ref).max() / np.sqrt(np.mean(ref.astype(np.float64) ** 2)))
        errs.append((rel, mx))
    return errs


@pytest.mark.parametrize("builder,dtype", [("simt", torch.float32), ("simt", torch.bfloat16)])
def test_corr_pyramid_simt_golden(golden, builder, dtype):
    from model.corr import CorrBlock

    g = golden("corr")
    blk = CorrBlock(T(g["fmap1"]), T(g["fmap2"]), num_levels=4, radius=4, pyramid_dtype=dtype, builder=builder)
    refs = [g[f"pyr{i}"] for i in range(4)]
    for (rel, mx) in _pyr_errors(blk.corr_pyramid, refs):
        if dtype == torch.float32:
            assert rel <= 1e-5 and mx <= 1e-4
        else:
            assert rel <= 4e-3 and mx <= 4e-2
    blk = CorrBlock(T(g["odd_fmap1"]), T(g["odd_fmap2"]), num_levels=3, radius=3, pyramid_dtype=torch.float32)
    assert [tuple(p.shape) for p in blk.corr_pyramid] == [(273, 1, 13, 21), (273, 1, 6, 10), (273, 1, 3, 5)]
    for (rel, mx) in _pyr_errors(blk.corr_pyramid, [g[f"odd_pyr{i}"] for i in range(3)]):
        assert rel <= 1e-5
    out = blk(T(g["odd_coords"]))
    assert maxabs(N(out), g["odd_lookup"]) <= 1e-4


@pytest.mark.parametrize("cta_group", [1, 2, 3])
def test_corr_pyramid_tcgen05_golden(golden, cta_group):
    """tcgen05 builder on the golden 16x16 / C=64 case (single partial tile, pooled levels clipped)."""
    from model.corr import CorrBlock

    g = golden("corr")
    blk = CorrBlock(T(g["fmap1"]), T(g["fmap2"]), num_levels=4, radius=4, cta_group=cta_group)
    assert blk.builder == "tcgen05"
    torch.cuda.synchronize()
    for (rel, mx) in _pyr_errors(blk.corr_pyramid, [g[f"pyr{i}"] for i in range(4)]):
        assert rel <= 4e-3 and mx <= 4e-2, (rel, mx)
    # end to end: lookup on the bf16 pyramid vs the reference's fp32 result
    out = N(blk(T(g["coords_noise"])))
    ref = g["lookup_noise"]
    assert np.linalg.norm(out - ref) / np.linalg.norm(ref) <= 6e-3


@pytest.mark.parametrize("cta_group", [1, 2, 3])
@pytest.mark.parametrize("shape", [(2, 256, 47, 156), (1, 128, 55, 128), (1, 256, 40, 72), (3, 64, 9, 35), (2, 256, 33, 50)])
def test_corr_pyramid_tcgen05_vs_fp32(cta_group, shape):
    """Against the fp32 CUDA-core builder (reference op order) and, for the small case, the CPU oracle."""
    from model.corr import CorrBlock

    b, c, h, w = shape
    gen = torch.Generator(device="cuda").manual_seed(11)
    f1 = torch.randn(shape, device="cuda", generator=gen)
    f2 = torch.randn(shape, device="cuda", generator=gen)
    levels = 4 if min(h, w) >= 8 else 3
    ref_blk = CorrBlock(f1, f2, num_levels=levels, pyramid_dtype=torch.float32, builder="simt")
    blk = CorrBlock(f1, f2, num_levels=levels, cta_group=cta_group)
    torch.cuda.synchronize()
    refs = [N(p) for p in ref_blk.corr_pyramid]
    if h * w <= 3000:
        orc = oracle.corr_pyramid(N(f1), N(f2), levels)
        for a, o in zip(refs, orc):
            assert maxabs(a, o) <= 2e-4
    for lvl, (rel, mx) in enumerate(_pyr_errors(blk.corr_pyramid, refs)):
        assert rel <= 4e-3 and mx <= 4e-2, (lvl, rel, mx)


@pytest.mark.parametrize("shape", [(2, 256, 47, 156), (1, 256, 40, 72), (3, 64, 9, 35)])
def test_corr_pyramid_store_and_launch_modes_agree(shape, monkeypatch):
    """The measured K2 alternatives stay correct: every epilogue store mode (direct 32-byte register stores, TMA bulk
    stores, software-pipelined 32-column pieces) under every launch mode (one CTA per tile, cta_group::2 pair, multicast
    clusters) writes the same bits inside the images of all four levels."""
    from model.corr import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(91)
    f1 = torch.randn(shape, device="cuda", generator=gen)
    f2 = torch.randn(shape, device="cuda", generator=gen)
    levels = 4 if min(shape[2:]) >= 8 else 3
    ref = None
    for epi in ("direct", "bulk", "pipe"):
        monkeypatch.setenv("OFB_K2_EPI", epi)
        for cg in (1, 2, 3):
            blk = CorrBlock(f1, f2, num_levels=levels, cta_group=cg)
            torch.cuda.synchronize()
            got = [p.clone() for p in blk.corr_pyramid]
            if ref is None:
                ref = got
            else:
                for lvl, (a, b) in enumerate(zip(ref, got)):
                    assert torch.equal(a, b), (epi, cg, lvl)


def test_corr_block_is_immune_to_poisoned_allocator_memory():
    """The lookup kernel may read the padding of the pyramid buffers (with zero weights): whatever the
    caching allocator hands back, the builder must have left finite values there."""
    from model.corr import CorrBlock
    from model.utils import coords_grid

    gen = torch.Generator(device="cuda").manual_seed(21)
    b, c, h, w = 1, 64, 19, 37                                  # odd sizes: every level has padding
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    ref = CorrBlock(f1, f2, pyramid_dtype=torch.float32, builder="simt")
    coords = coords_grid(b, h, w).cuda() + 3 * torch.randn((b, 2, h, w), device="cuda", generator=gen)
    want = ref(coords)
    for _ in range(3):
        poison = torch.full((64 << 20,), float("nan"), dtype=torch.bfloat16, device="cuda")
        del poison                                               # back to the caching allocator, NaN-filled
        blk = CorrBlock(f1, f2)
        got = blk(coords)
        assert torch.isfinite(got).all()
        assert float((got - want).norm() / want.norm()) <= 6e-3
        del blk


def test_corr_volume_static_and_errors():
    from model.corr import CorrBlock

    gen = torch.Generator(device="cuda").manual_seed(12)
    f1 = torch.randn((1, 64, 8, 24), device="cuda", generator=gen)
    f2 = torch.randn((1, 64, 8, 24), device="cuda", generator=gen)
    vol = CorrBlock.corr(f1, f2, pyramid_dtype=torch.float32)
    assert vol.shape == (1, 8, 24, 1, 8, 24) and vol.dtype == torch.float32
    ref = oracle.corr_volume(N(f1), N(f2))
    assert maxabs(N(vol), ref) <= 2e-5
    with pytest.raises(RuntimeError):
        CorrBlock(f1[:, :, :4, :4], f2[:, :, :4, :4], num_levels=4)      # too small: reference raises too
    with pytest.raises(RuntimeError):
        CorrBlock(f1, f2)(torch.zeros(1, 2, 8, 23, device="cuda"))


def test_corr_pyramid_full_size_properties():
    """C3 B=16, 256 ch, 55x128: every pooled level equals the mean of complete 2^l x 2^l blocks of
    level 0 (pyramid identity), checked on a random subset of queries; swapping fmap1 and fmap2
    transposes level 0."""
    from model.corr import CorrBlock

    b, c, h, w = 16, 256, 55, 128
    gen = torch.Generator(device="cuda").manual_seed(13)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2)
    torch.cuda.synchronize()
    q = torch.randint(0, b * h * w, (512,), device="cuda", generator=gen)
    l0 = blk.corr_pyramid[0][q, 0].float()
    # direct fp32 recomputation of those rows
    qb, qp = q // (h * w), q % (h * w)
    a = f1.view(b, c, h * w)[qb, :, qp]                                   # (512, c)
    ref0 = torch.einsum("qc,qcn->qn", a, f2.view(b, c, h * w)[qb]) / 16.0
    ref0 = ref0.view(-1, h, w)
    assert float((l0 - ref0).norm() / ref0.norm()) <= 4e-3
    for lvl in range(1, 4):
        k = 2 ** lvl
        hl, wl = h // k, w // k
        pooled = ref0[:, : hl * k, : wl * k].reshape(-1, hl, k, wl, k).mean(dim=(2, 4))
        got = blk.corr_pyramid[lvl][q, 0].float()
        assert got.shape == pooled.shape
        assert float((got - pooled).norm() / pooled.norm()) <= 4e-3, lvl
    blk_t = CorrBlock(f2, f1, num_levels=1)
    torch.cuda.synchronize()
    bsel = 3
    v = blk.corr_pyramid[0].view(b, h * w, h, w)[bsel].reshape(h * w, h * w).float()
    vt = blk_t.corr_pyramid[0].view(b, h * w, h, w)[bsel].reshape(h * w, h * w).float()
    assert float((v - vt.t()).abs().max()) <= 0.05


def _sampled_rows_fp32(f1, f2, q):
    """fp32 rows q of corr = fmap1^T . fmap2 / sqrt(C) (reference corr.py:82-87), one matmul per batch element."""
    b, c, h, w = f1.shape
    n = h * w
    out = torch.empty((q.numel(), n), dtype=torch.float32, device=f1.device)
    qb, qp = q // n, q % n
    for bi in range(b):
        sel = (qb == bi).nonzero().flatten()
        if sel.numel():
            a = f1.view(b, c, n)[bi][:, qp[sel]].t().contiguous()          # (k, C)
            out[sel] = (a @ f2.view(b, c, n)[bi]) / float(c) ** 0.5
    return out.view(-1, h, w)


def test_corr_pyramid_c5_bench_shape_vs_fp32():
    """The bench shape (C5 micro-batch: 256 ch, 136x240, two pairs): sampled query rows of every level against an fp32
    recomputation (level 0) and the means of complete 2^l x 2^l blocks of it (levels 1-3; 136 = 8 * 17 exercises the
    floor of reference corr.py:52-54 on the last level: 17 x 30), plus a CPU-oracle cross-check of a few rows."""
    from model.corr import CorrBlock

    b, c, h, w = 2, 256, 136, 240
    gen = torch.Generator(device="cuda").manual_seed(41)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2)
    assert blk.builder == "tcgen05"
    torch.cuda.synchronize()
    n = h * w
    corners = torch.tensor([0, w - 1, n - w, n - 1, n, 2 * n - 1, n + 127, n + 128, 32639, 32640 - 241], device="cuda")
    q = torch.cat([corners, torch.randint(0, b * n, (758,), device="cuda", generator=gen)])
    ref0 = _sampled_rows_fp32(f1, f2, q)
    assert [tuple(p.shape[-2:]) for p in blk.corr_pyramid] == [(136, 240), (68, 120), (34, 60), (17, 30)]
    for lvl in range(4):
        k = 2 ** lvl
        hl, wl = h // k, w // k
        want = ref0[:, : hl * k, : wl * k].reshape(-1, hl, k, wl, k).mean(dim=(2, 4))
        got = blk.corr_pyramid[lvl][q, 0].float()
        assert got.shape == want.shape
        rel = float((got - want).norm() / want.norm())
        mx = float((got - want).abs().max() / want.pow(2).mean().sqrt())
        assert rel <= 4e-3 and mx <= 4e-2, (lvl, rel, mx)
    # the fp32 recomputation itself against the CPU oracle's sgemm (reference op order) on 6 rows
    f1n, f2n = N(f1), N(f2)
    for qi in (0, 9, 100):
        qq = int(q[qi]); bi, p = divmod(qq, n)
        row = (f1n[bi].reshape(c, n)[:, p] @ f2n[bi].reshape(c, n)) / np.float32(16.0)
        assert maxabs(N(ref0[qi]).ravel(), row) <= 2e-4


@pytest.mark.parametrize("kind", ["int", "noise", "edge"])
def test_lookup_c5_bench_shape_on_stored_pyramid(kind):
    """K3 at 136x240 on the pyramid the tcgen05 builder stored (query-minor 8x4 blocks): floor indices and validity
    masks bit-exact for EVERY query, values <= 1e-5 against the CPU oracle run on the GPU's own stored levels for
    2048 sampled queries (the oracle needs fp32 slices: 131 KB per query and level 0)."""
    from model.corr import CorrBlock

    b, c, h, w = 1, 256, 136, 240
    gen = torch.Generator(device="cuda").manual_seed(43)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    blk = CorrBlock(f1, f2)
    r = rng(44)
    coords = oracle.coords_grid(b, h, w)
    if kind == "noise":
        coords = (coords + 4 * r.standard_normal(coords.shape)).astype(np.float32)
    if kind == "edge":
        coords[:, 0] = np.where(coords[:, 0] < w / 2, coords[:, 0] * 0.1 - 3.0, w - 1 + coords[:, 0] * 0.05)
        coords[:, 1] = np.where(coords[:, 1] < h / 2, -2.0, h + 1.25)
        coords = coords.astype(np.float32)
    out, idx, valid = blk(T(coords), return_index=True)
    out, idx, valid = N(out), N(idx), N(valid)
    n = h * w
    sel = np.unique(np.concatenate([[0, w - 1, n - w, n - 1, n // 2], r.integers(0, n, 2043)]))
    sel_d = torch.from_numpy(sel).cuda()
    levels = [N(blk.corr_pyramid[l][sel_d].float()) for l in range(4)]
    csel = coords.reshape(1, 2, n)[:, :, sel].reshape(1, 2, 1, sel.size)
    ref, ridx, rvalid = oracle.corr_lookup(levels, csel, radius=4, return_index=True)
    assert np.array_equal(idx[sel], ridx) and np.array_equal(valid[sel], rvalid)
    got = out.reshape(324, n)[:, sel]
    assert maxabs(got, ref.reshape(324, sel.size)) <= tol(ref)
    # indices / masks of all queries: a pyramid of the same level sizes carries no values into them
    zeros = [np.zeros((1, 1, h >> l, w >> l), np.float32) for l in range(4)]
    _, ridx, rvalid = oracle.corr_lookup(zeros, coords, radius=4, return_index=True, shared_slice=True)
    assert np.array_equal(idx, ridx) and np.array_equal(valid, rvalid)


# =============================================================================== RAFT.forward trace
@pytest.mark.parametrize("mode", ["fp32_simt", "bf16_tcgen05"])
def test_raft_forward_trace(golden, mode):
    """SURVEY 8f row 1: the accelerated block inside the unmodified model.  The reference's RAFT.forward was
    run on CPU with hooks on the hot-path boundary (tests/golden/make_golden.py:make_raft_trace); here the
    recorded CorrBlock / corr_fn / upsample_flow calls are replayed on the B200 kernels."""
    from model.corr import CorrBlock
    from model.raft import RAFT

    g = golden("raft_trace")
    f1, f2 = T(g["fmap1"]), T(g["fmap2"])
    if mode == "fp32_simt":
        blk, rtol = CorrBlock(f1, f2, radius=4, pyramid_dtype=torch.float32), 2e-4
    else:
        blk, rtol = CorrBlock(f1, f2, radius=4), 6e-3        # bf16 operands and bf16 stored volume
        assert blk.builder == "tcgen05"
    for it in range(g["coords"].shape[0]):
        out = N(blk(T(g["coords"][it])))
        ref = g["corr"][it]
        assert out.shape == ref.shape
        if mode == "fp32_simt":
            assert maxabs(out, ref) <= rtol * max(1.0, float(np.abs(ref).max())), it
        else:
            assert np.linalg.norm(out - ref) / np.linalg.norm(ref) <= rtol, it
        up = N(RAFT.upsample_flow(T(g["up_flow"][it]), T(g["up_mask"][it])))
        assert maxabs(up, g["up_out"][it]) <= tol(g["up_out"][it]), it


# =============================================================================== memory safety
def test_kernels_do_not_write_outside_their_buffers():
    """compute-sanitizer is closed on this GPU pool, so out-of-bounds WRITES are caught with guard bands:
    every output buffer is carved out of a larger sentinel-filled allocation and the bands must survive.
    Odd sizes exercise every edge path (partial tiles, partial blocks, padded rows)."""
    import ctypes

    import ofb200
    from model.corr import prepare_operands

    lib = ofb200.load()
    guard = 4096                                                     # elements on each side
    gen = torch.Generator(device="cuda").manual_seed(31)

    def banded(n, dtype, sentinel):
        whole = torch.full((n + 2 * guard,), sentinel, dtype=dtype, device="cuda")
        return whole, whole[guard:guard + n]

    def intact(whole, n, sentinel):
        ref = torch.full((guard,), sentinel, dtype=whole.dtype, device="cuda")
        return bool(torch.equal(whole[:guard], ref)) and bool(torch.equal(whole[guard + n:], ref))

    for (b, c, h, w) in [(2, 64, 19, 37), (1, 128, 47, 156), (1, 256, 9, 35)]:
        f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
        f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
        a_km, b_km, q_km = prepare_operands(f1, f2, 4)
        for mode in (1, 2, 3):                                       # padded rows, 8x4 blocks, query-minor blocks
            for cg in (1, 2):
                pyr = ofb200.Pyramid()
                elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
                ofb200.check(lib.ofb_pyramid_layout(h, w, 4, mode, ctypes.byref(pyr), ctypes.byref(elems)), "layout")
                pyr.dtype = ofb200.DTYPE_BF16
                keep = []
                for lvl in range(4):
                    n = b * h * w * int(elems[lvl])
                    whole, view = banded(n, torch.bfloat16, -7.0)
                    keep.append((whole, n))
                    pyr.base[lvl] = view.data_ptr()
                ofb200.check(lib.ofb_corr_pyramid_bf16(ofb200.ptr(a_km), ofb200.ptr(b_km), ofb200.ptr(q_km), ctypes.byref(pyr),
                                                       b, c, h, w, 1.0, cg, ofb200.stream_ptr()), "pyramid")
                n_out = b * 324 * h * w
                whole_o, out = banded(n_out, torch.float32, -7.0)
                coords = torch.randn((b, 2, h, w), device="cuda", generator=gen) * 30 + 10
                ofb200.check(lib.ofb_corr_lookup(ctypes.byref(pyr), ofb200.ptr(coords), ofb200.ptr(out), None, None,
                                                 b, h, w, 4, ofb200.stream_ptr()), "lookup")
                torch.cuda.synchronize()
                for whole, n in keep:
                    assert intact(whole, n, -7.0), (b, c, h, w, mode, cg)
                assert intact(whole_o, n_out, -7.0) and bool(torch.isfinite(out).all())
    # streaming kernels at odd sizes
    for (b, c, h, w) in [(2, 3, 37, 53), (1, 5, 16, 130), (2, 6, 19, 132)]:
        frame = torch.rand((b, c, h, w), device="cuda", generator=gen)
        flow = torch.randn((b, 2, h, w), device="cuda", generator=gen) * 0.3
        for variant in warp_variants(w):
            whole, out = banded(b * c * h * w, torch.float32, -7.0)
            wm, mask = banded(b * h * w, torch.uint8, 200)
            ofb200.check(lib.ofb_warp_f32(ofb200.ptr(frame), ofb200.ptr(flow), ofb200.ptr(out), ofb200.ptr(mask), b, c, h, w,
                                          0, 1, 0, 0, variant, 1.0, 1.0, ofb200.stream_ptr()), "warp")
            torch.cuda.synchronize()
            assert intact(whole, b * c * h * w, -7.0) and intact(wm, b * h * w, 200), variant
    n, h, w = 2, 7, 11
    flow = torch.randn((n, 2, h, w), device="cuda", generator=gen)
    mask = torch.randn((n, 576, h, w), device="cuda", generator=gen)
    whole, out = banded(n * 2 * 64 * h * w, torch.float32, -7.0)
    ofb200.check(lib.ofb_convex_upsample_f32(ofb200.ptr(flow), ofb200.ptr(mask), ofb200.ptr(out), n, h, w, ofb200.stream_ptr()), "up")
    torch.cuda.synchronize()
    assert intact(whole, n * 2 * 64 * h * w, -7.0)


# =============================================================================== randomized sweep
@pytest.mark.parametrize("seed", list(range(12)))
def test_random_shapes_corr_block_and_lookup(seed, monkeypatch):
    """Random (B, C, h, w), level count, radius, layout and CTA shape: the tcgen05 pyramid against the fp32
    CUDA-core builder, and the lookup on the stored pyramid against the oracle (indices and masks bit-exact)."""
    from model.corr import CorrBlock

    r = rng(1000 + seed)
    c = int(r.choice([64, 128, 192, 256]))
    h, w = int(r.integers(8, 70)), int(r.integers(8, 170))
    b = int(r.integers(1, 4))
    levels = int(r.integers(1, 5))
    while (h >> (levels - 1)) < 2 or (w >> (levels - 1)) < 2:     # keep every level at least 2x2 (1x1 divides by zero)
        levels -= 1
    radius = int(r.choice([3, 4]))
    monkeypatch.setenv("OFB200_PYRAMID_LAYOUT", str(r.choice(["qminor", "blocked"])))
    cta_group = int(r.choice([1, 2]))
    gen = torch.Generator(device="cuda").manual_seed(seed)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    ref_blk = CorrBlock(f1, f2, num_levels=levels, radius=radius, pyramid_dtype=torch.float32, builder="simt")
    blk = CorrBlock(f1, f2, num_levels=levels, radius=radius, cta_group=cta_group)
    assert blk.builder == "tcgen05"
    torch.cuda.synchronize()
    info = (b, c, h, w, levels, radius, cta_group)
    for lvl, (rel, mx) in enumerate(_pyr_errors(blk.corr_pyramid, [N(p) for p in ref_blk.corr_pyramid])):
        assert rel <= 4e-3 and mx <= 4e-2, (info, lvl, rel, mx)
    coords = (oracle.coords_grid(b, h, w) + float(r.choice([0.0, 0.5, 3.0, 25.0])) * r.standard_normal((b, 2, h, w))).astype(np.float32)
    out, idx, valid = blk(T(coords), return_index=True)
    stored = [np.ascontiguousarray(N(p.float())) for p in blk.corr_pyramid]
    ref, ridx, rvalid = oracle.corr_lookup(stored, coords, radius=radius, return_index=True)
    assert np.array_equal(N(idx), ridx) and np.array_equal(N(valid), rvalid), info
    assert maxabs(N(out), ref) <= tol(ref), info


@pytest.mark.parametrize("seed", list(range(12)))
def test_random_shapes_streaming_kernels(seed):
    """Random shapes / options for warp (every kernel variant), resize, convex upsampling and the metric reductions
    against the oracle."""
    from model.raft import upsample_flow
    from optical_flow import normalize, resize, warp
    from optical_flow.metrics import AverageEndPointError, OutlierRatio

    r = rng(2000 + seed)
    b, c = int(r.integers(1, 4)), int(r.integers(1, 6))
    h, w = int(r.integers(1, 90)), int(r.integers(1, 200))
    if seed == 3:
        h = 1
    if seed == 5:
        w = 1
    if seed % 2:
        w = (w + 3) // 4 * 4                                  # widths the TMA-window warp accepts
    pad = str(r.choice(["zeros", "border", "reflection"]))
    ac = bool(r.integers(0, 2))
    frame = r.random((b, c, h, w), dtype=np.float32)
    flow_px = (float(r.choice([0.5, 5.0, 40.0])) * r.standard_normal((b, 2, h, w))).astype(np.float32)
    flow = oracle.normalize(flow_px).astype(np.float32)
    ref, ref_mask = oracle.warp(frame, flow, padding_mode=pad, align_corners=ac, return_mask=True)
    outs = []
    for variant in warp_variants(w):
        out, mask = warp(T(frame), T(flow), padding_mode=pad, align_corners=ac, return_mask=True, variant=variant)
        assert maxabs(N(out), ref) <= 1e-5, (variant, b, c, h, w, pad, ac)
        assert np.array_equal(N(mask).astype(np.uint8), ref_mask)
        outs.append(N(out))
    assert all(np.array_equal(outs[0], o) for o in outs[1:])
    fused = warp(T(frame), T(flow_px), padding_mode=pad, align_corners=ac, pixel_flow=True)
    assert np.array_equal(N(fused), outs[2])
    # resize to a random size
    ho, wo = int(r.integers(1, 120)), int(r.integers(1, 260))
    got = N(resize(T(flow_px), size=(ho, wo)))
    want = oracle.resize(flow_px, size=(ho, wo))
    assert maxabs(got, want) <= tol(want), (h, w, ho, wo)
    # convex upsampling on a coarse grid of the same aspect
    hc, wc = max(h // 8, 1), max(w // 8, 1)
    fl = r.standard_normal((b, 2, hc, wc)).astype(np.float32)
    mk = (2 * r.standard_normal((b, 576, hc, wc))).astype(np.float32)
    up = N(upsample_flow(T(fl), T(mk)))
    want = oracle.upsample_flow(fl, mk)
    assert maxabs(up, want) <= tol(want)
    # metrics
    target = (flow_px + r.standard_normal(flow_px.shape)).astype(np.float32)
    valid = (r.random((b, h, w)) > 0.3).astype(np.float32)
    m, f1 = AverageEndPointError(), OutlierRatio(abs_threshold=0.5, rel_threshold=0.05)
    m.update(T(flow_px), T(target), T(valid)); f1.update(T(flow_px), T(target), T(valid))
    s, n = oracle.epe_sum_count(flow_px, target, valid)
    so, no = oracle.outlier_sum_count(flow_px, target, valid, 0.5, 0.05)
    assert int(m.total) == n and abs(float(m._acc[0]) - s) <= 1e-6 * max(1.0, s)
    assert int(f1.total) == no and float(f1._acc[0]) == so
