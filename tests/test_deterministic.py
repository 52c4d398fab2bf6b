"""Bit-reproducible gradients, and `torch.use_deterministic_algorithms` honoured.

The convex upsampling's d_flow and the bilinear resize's (`resize`, `upflow8`) gradient are fixed-order gathers, so
every backward the RAFT training step runs through the library -- correlation pyramid (bf16 / fp16, tcgen05 GEMMs),
lookups, their coordinates, `upsample_flow` and `sequence_loss` -- gives the same bits on every run.  The one
order-dependent gradient left, `warp`'s frame gradient (an atomic scatter), raises under
`torch.use_deterministic_algorithms(True)` as `F.grid_sample`'s backward does, and warns with `warn_only=True`.
"""
import os
import subprocess
import sys
import textwrap

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def det_flags():
    """Save and restore the determinism switches a test changes."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    saved = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled(),
             torch.backends.cudnn.deterministic, torch.utils.deterministic.fill_uninitialized_memory)
    yield
    torch.use_deterministic_algorithms(saved[0], warn_only=saved[1])
    torch.backends.cudnn.deterministic = saved[2]
    torch.utils.deterministic.fill_uninitialized_memory = saved[3]


def bits_equal(a, b):
    if a is None or b is None:
        return a is None and b is None
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    iview = {4: torch.int32, 2: torch.int16}[a.element_size()]
    return torch.equal(a.contiguous().view(iview), b.contiguous().view(iview))


def busy_side_stream():
    """Unrelated work on another stream, running while the backward under test runs."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        x = torch.empty(1 << 25, device="cuda").normal_()
        for _ in range(8):
            x = torch.sin(x) * 1.0001
    return side, x


def twice(fn):
    """fn() run twice, each behind a busy side stream; returns both results."""
    out = []
    for _ in range(2):
        side, keep = busy_side_stream()
        out.append(fn())
        torch.cuda.current_stream().wait_stream(side)
        del keep
    torch.cuda.synchronize()
    return out


# ---------------------------------------------------------------------------------------------------- convex upsampling

UP_SHAPES = [(16, 47, 156), (2, 19, 37), (1, 1, 1), (3, 15, 31), (1, 29, 61)]
MASK_DTYPES = [torch.float32, torch.bfloat16, torch.float16]


def up_inputs(shape, dt, seed):
    n, h, w = shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    flow = 2 * torch.randn((n, 2, h, w), device="cuda", generator=g)
    mask = (2 * torch.randn((n, 576, h, w), device="cuda", generator=g)).to(dt)
    d_out = torch.randn((n, 2, 8 * h, 8 * w), device="cuda", generator=g)
    return flow, mask, d_out


def up_backward(flow, mask, d_out, want_flow=True, want_mask=True):
    from ofb200.ops.raft_ops import upsample_flow

    f = flow.clone().requires_grad_(want_flow)
    m = mask.clone().requires_grad_(want_mask)
    inputs = [t for t in (f, m) if t.requires_grad]
    grads = torch.autograd.grad(upsample_flow(f, m), inputs, grad_outputs=d_out)
    it = iter(grads)
    return (next(it) if want_flow else None), (next(it) if want_mask else None)


@pytest.mark.parametrize("shape", UP_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dt", MASK_DTYPES, ids=str)
def test_upsample_backward_repeats_bit_for_bit(det_flags, dt, shape):
    flow, mask, d_out = up_inputs(shape, dt, 11)
    (f1, m1), (f2, m2) = twice(lambda: up_backward(flow, mask, d_out))
    assert bits_equal(f1, f2) and bits_equal(m1, m2)
    # d_mask does not depend on whether d_flow is wanted (the halo only feeds d_flow), nor d_flow on d_mask
    assert bits_equal(up_backward(flow, mask, d_out, want_flow=False)[1], m1)
    assert bits_equal(up_backward(flow, mask, d_out, want_mask=False)[0], f1)


def test_upsample_backward_accumulates_into_d_flow(det_flags):
    """The C ABI adds to d_flow: one add per element, of the value a zero-filled d_flow receives."""
    import ofb200

    flow, mask, d_out = up_inputs((2, 19, 37), torch.float32, 3)
    lib = ofb200.load()

    def run(d_flow):
        rc = lib.ofb_convex_upsample_backward(ofb200.ptr(flow), ofb200.ptr(mask), ofb200.DTYPE_F32, ofb200.ptr(d_out),
                                              ofb200.ptr(d_flow), None, 2, 19, 37, ofb200.stream_ptr())
        ofb200.check(rc, "ofb_convex_upsample_backward")
        return d_flow

    base = torch.randn_like(flow)
    got = run(base.clone())
    alone = run(torch.zeros_like(flow))
    assert bits_equal(got, base + alone)


@pytest.mark.parametrize("shape", [(2, 19, 37), (1, 1, 1), (3, 15, 31)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dt", MASK_DTYPES, ids=str)
def test_upsample_backward_values_against_float64_adjoint(det_flags, dt, shape):
    """d_flow and d_mask against the reference expression's autograd in float64 (oracle/torch_port.py), on the
    mask's logits widened exactly; the bounds of the existing upsampling gradient tests."""
    from oracle import torch_port

    flow, mask, d_out = up_inputs(shape, dt, 5)
    d_flow, d_mask = up_backward(flow, mask, d_out)
    f64 = flow.double().requires_grad_(True)
    m64 = mask.double().requires_grad_(True)
    rf, rm = torch.autograd.grad(torch_port.upsample_flow(f64, m64), (f64, m64), grad_outputs=d_out.double())
    assert float((d_flow.double() - rf).abs().max()) <= 1e-5 * max(1.0, float(rf.abs().max()))
    rel = {torch.float32: 1e-5, torch.bfloat16: 1e-2, torch.float16: 2e-3}[dt]
    assert float((d_mask.double() - rm).abs().max()) <= rel * float(rm.abs().max())


# ---------------------------------------------------------------------------------------------------- resize / upflow8

RESIZE_CASES = [  # (h, w, ho, wo)
    (47, 156, 376, 1248),    # 8x up: upflow8 at C4
    (19, 37, 38, 74),        # 2x up
    (19, 37, 9, 18),         # down
    (19, 37, 29, 50),        # non-integer up
    (24, 40, 17, 23),        # non-integer down
    (19, 37, 19, 37),        # identity
    (1, 7, 5, 1),            # single rows / columns
]


# against float64: the source coordinates are the forward's fp32 ones (the atomic kernel's too); with align_corners the
# fp32 ratio (W-1)/(Wo-1) times indices up to 155 alone moves upflow8's gradient by ~1e-5 of its largest element at C4
UPFLOW8_TOL = {0: 1e-5, 1: 5e-5}


def resize_backward(x, size, ac, mul_x, mul_y, g):
    from ofb200.ops.operator import _resize_raw

    xr = x.clone().requires_grad_(True)
    (d,) = torch.autograd.grad(_resize_raw(xr, size, ac, mul_x, mul_y, "resize"), (xr,), grad_outputs=g)
    return d


def resize_adjoint64(x, size, ac, mul_x, mul_y, g):
    """F.interpolate's autograd in float64 on the CPU, with the magnitude factor per channel pair."""
    x64 = x.detach().double().cpu().requires_grad_(True)
    out = F.interpolate(x64, size=size, mode="bilinear", align_corners=bool(ac))
    fac = torch.tensor([mul_x, mul_y], dtype=torch.float64).repeat(x.shape[1] // 2).view(1, -1, 1, 1)
    (d,) = torch.autograd.grad(out * fac, (x64,), grad_outputs=g.double().cpu())
    return d


@pytest.mark.parametrize("ac", [0, 1])
@pytest.mark.parametrize("case", RESIZE_CASES, ids=lambda c: "{}x{}-{}x{}".format(*c))
def test_resize_backward_repeats_and_matches_float64(det_flags, case, ac):
    h, w, ho, wo = case
    gen = torch.Generator(device="cuda").manual_seed(ho * 1000 + wo)
    x = torch.randn((2, 2, h, w), device="cuda", generator=gen)
    g = torch.randn((2, 2, ho, wo), device="cuda", generator=gen)
    mul_x, mul_y = wo / w, ho / h
    d1, d2 = twice(lambda: resize_backward(x, (ho, wo), ac, mul_x, mul_y, g))
    assert bits_equal(d1, d2)
    ref = resize_adjoint64(x, (ho, wo), ac, mul_x, mul_y, g)
    assert float((d1.double().cpu() - ref).abs().max()) <= UPFLOW8_TOL[ac] * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("ac", [0, 1])
def test_resize_backward_is_exact_where_every_term_is(det_flags, ac):
    """2x upsampling (align_corners=False: weights 1/4 and 3/4; align_corners=True on 2^k + 1 grids: weights k / 2^m)
    of small-integer gradients: every product and partial sum is exact in fp32, so the gradient is the float64
    adjoint rounded once."""
    h, w, ho, wo = (19, 37, 38, 74) if ac == 0 else (9, 17, 17, 33)
    gen = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn((3, 2, h, w), device="cuda", generator=gen)
    g = torch.randint(-8, 9, (3, 2, ho, wo), device="cuda", generator=gen).float()
    d = resize_backward(x, (ho, wo), ac, 2.0, 2.0, g)
    ref = resize_adjoint64(x, (ho, wo), ac, 2.0, 2.0, g)
    assert torch.equal(d.cpu(), ref.float())


def test_upflow8_and_resize_surfaces_repeat(det_flags):
    from model.utils import upflow8
    from optical_flow import resize

    gen = torch.Generator(device="cuda").manual_seed(9)
    flow = torch.randn((16, 2, 47, 156), device="cuda", generator=gen)
    g8 = torch.randn((16, 2, 376, 1248), device="cuda", generator=gen)
    gr = torch.randn((16, 2, 70, 234), device="cuda", generator=gen)

    def run():
        f = flow.clone().requires_grad_(True)
        (a,) = torch.autograd.grad(upflow8(f), (f,), grad_outputs=g8)
        (b,) = torch.autograd.grad(resize(f, scale_factor=1.5), (f,), grad_outputs=gr)
        return a, b

    (a1, b1), (a2, b2) = twice(run)
    assert bits_equal(a1, a2) and bits_equal(b1, b2)
    ref = resize_adjoint64(flow, (376, 1248), 1, 8.0, 8.0, g8)
    assert float((a1.double().cpu() - ref).abs().max()) <= UPFLOW8_TOL[1] * float(ref.abs().max())


# ---------------------------------------------------------------------------------------------------- correlation block

def corr_inputs(seed, b=2, c=64, h=23, w=37):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    from model.utils import coords_grid

    coords = coords_grid(b, h, w).cuda() + 3 * torch.randn((b, 2, h, w), device="cuda", generator=gen)
    g = torch.randn((b, 4 * 81, h, w), device="cuda", generator=gen)
    return f1, f2, coords, g


@pytest.mark.parametrize("pdt", [torch.bfloat16, torch.float16], ids=str)
def test_corr_block_backward_repeats_bit_for_bit(det_flags, pdt):
    """The tcgen05 pyramid backward, the lookup's pyramid gradient and its coordinate gradient, twice."""
    from model.corr import CorrBlock

    f1, f2, coords, g = corr_inputs(21)

    def run():
        a, b, c = (t.clone().requires_grad_(True) for t in (f1, f2, coords))
        blk = CorrBlock(a, b, num_levels=4, radius=4, pyramid_dtype=pdt)
        outs = [blk(c + 0.25 * k) for k in range(3)]
        return torch.autograd.grad(sum((o * g).sum() for o in outs), (a, b, c))

    r1, r2 = twice(run)
    assert all(bits_equal(x, y) for x, y in zip(r1, r2))


# ---------------------------------------------------------------------------------------------------- RAFT-shaped step

class Step(torch.nn.Module):
    """A RAFT-shaped training step: conv feature encoder -> CorrBlock -> 12 lookups with a conv update stand-in ->
    `upsample_flow` with a mask head run under autocast (or, as mask-less RAFT, `upflow8`) -> `sequence_loss`."""

    def __init__(self):
        super().__init__()
        self.fnet = torch.nn.Conv2d(3, 64, 8, stride=8)
        self.update = torch.nn.Conv2d(4 * 81 + 2, 2, 3, padding=1)
        self.mask = torch.nn.Conv2d(4 * 81 + 2, 576, 1)

    def forward(self, ops, img1, img2, gt, valid, half, convex=True):
        f1, f2 = self.fnet(img1), self.fnet(img2)
        b, _, h, w = f1.shape
        coords0 = ops["coords_grid"](b, h, w).to(img1.device)
        coords1 = coords0.clone()
        corr_fn = ops["corr"](f1, f2)
        preds = []
        for _ in range(12):
            coords1 = coords1.detach()
            corr = corr_fn(coords1)
            x = torch.cat([corr, coords1 - coords0], dim=1)
            coords1 = coords1 + 0.1 * self.update(x)
            with torch.autocast("cuda", dtype=half):
                mask = 0.25 * self.mask(x)
            preds.append(ops["upsample_flow"](coords1 - coords0, mask) if convex else ops["upflow8"](coords1 - coords0))
        return ops["sequence_loss"](preds, gt, valid)


def step_inputs(seed=4):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    img1 = torch.rand((2, 3, 128, 192), device="cuda", generator=gen)
    img2 = torch.roll(img1, shifts=(2, -3), dims=(2, 3))
    gt = 3 * torch.randn((2, 2, 128, 192), device="cuda", generator=gen)
    valid = (torch.rand((2, 128, 192), device="cuda", generator=gen) > 0.1).float()
    return img1, img2, gt, valid


def ours(pdt):
    from model.corr import CorrBlock
    from model.raft import sequence_loss, upsample_flow
    from model.utils import coords_grid, upflow8

    return {"coords_grid": coords_grid, "upsample_flow": upsample_flow, "upflow8": upflow8,
            "corr": lambda a, b: CorrBlock(a, b, num_levels=4, radius=4, pyramid_dtype=pdt),
            "sequence_loss": lambda p, g, v: sequence_loss(p, g, v)[0]}


def train_grads(ops, half, convex=True, seed=4):
    torch.manual_seed(1234)
    net = Step().cuda()
    loss = net(ops, *step_inputs(seed), half=half, convex=convex)
    loss.backward()
    return loss.detach(), [p.grad for p in net.parameters()]


@pytest.mark.parametrize("convex", [True, False], ids=["convex", "upflow8"])
@pytest.mark.parametrize("half", [torch.float16, torch.bfloat16], ids=str)
@pytest.mark.parametrize("pdt", [torch.bfloat16, torch.float16], ids=str)
def test_training_step_gradients_repeat_under_the_flag(det_flags, pdt, half, convex):
    torch.use_deterministic_algorithms(True)
    (l1, g1), (l2, g2) = twice(lambda: train_grads(ours(pdt), half, convex))
    assert bits_equal(l1, l2)
    assert len(g1) == 6 and all(g is not None for g in g1[:4])   # the mask head has no gradient without `convex`
    assert all(bits_equal(a, b) for a, b in zip(g1, g2))


# ---------------------------------------------------------------------------------------------------- forward under the flag

def test_forward_outputs_unchanged_with_nan_filled_allocations(det_flags):
    """torch NaN-fills every torch.empty under the flag: outputs equal to the ones without it prove no kernel reads
    memory it did not write (pyramid padding included)."""
    from model.corr import CorrBlock
    from model.raft import upsample_flow
    from optical_flow import warp

    f1, f2, coords, _ = corr_inputs(31)
    flow, mask, _ = up_inputs((2, 19, 37), torch.float16, 8)
    gen = torch.Generator(device="cuda").manual_seed(8)
    frame = torch.rand((2, 3, 152, 296), device="cuda", generator=gen)
    wflow = 0.05 * torch.randn((2, 2, 152, 296), device="cuda", generator=gen)

    def run():
        outs = []
        for pdt in (torch.bfloat16, torch.float16):
            blk = CorrBlock(f1, f2, num_levels=4, radius=4, pyramid_dtype=pdt)
            outs += [blk(coords), blk(coords + 0.5)]
        outs.append(upsample_flow(flow, mask))
        outs += list(warp(frame, wflow, return_mask=True))
        outs.append(warp(frame, wflow, padding_mode="zeros", align_corners=True))
        return outs

    torch.use_deterministic_algorithms(False)
    plain = run()
    torch.use_deterministic_algorithms(True)
    torch.utils.deterministic.fill_uninitialized_memory = True
    filled = run()
    assert all(torch.equal(a, b) for a, b in zip(plain, filled))
    assert all(not torch.isnan(t.float()).any() for t in filled if t.is_floating_point())


# ---------------------------------------------------------------------------------------------------- warp

def warp_inputs():
    gen = torch.Generator(device="cuda").manual_seed(12)
    frame = torch.rand((2, 16, 64, 96), device="cuda", generator=gen)
    flow = 0.1 * torch.randn((2, 2, 64, 96), device="cuda", generator=gen)
    g = torch.randn((2, 16, 64, 96), device="cuda", generator=gen)
    return frame, flow, g


def test_warp_flow_gradient_runs_and_repeats_under_the_flag(det_flags):
    from optical_flow import warp

    frame, flow, g = warp_inputs()
    torch.use_deterministic_algorithms(True)

    def run():
        f = flow.clone().requires_grad_(True)
        return torch.autograd.grad(warp(frame, f), (f,), grad_outputs=g)[0]

    d1, d2 = twice(run)
    assert bits_equal(d1, d2)


def test_warp_frame_gradient_raises_under_the_flag(det_flags):
    from optical_flow import warp

    frame, flow, g = warp_inputs()
    fr, fl = frame.clone().requires_grad_(True), flow.clone().requires_grad_(True)
    torch.use_deterministic_algorithms(True)
    with pytest.raises(RuntimeError, match="does not have a deterministic implementation, but you set "
                                           "'torch.use_deterministic_algorithms\\(True\\)'"):
        torch.autograd.grad(warp(fr, fl), (fr, fl), grad_outputs=g)
    # the reference's warp (F.grid_sample) refuses the same way
    from oracle import torch_port

    with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
        torch.autograd.grad(torch_port.warp(fr, fl), (fr,), grad_outputs=g)


def test_warp_frame_gradient_warns_with_warn_only(det_flags):
    from optical_flow import warp

    frame, flow, g = warp_inputs()
    fr = frame.clone().requires_grad_(True)
    torch.use_deterministic_algorithms(False)
    (ref,) = torch.autograd.grad(warp(fr, flow), (fr,), grad_outputs=g)
    torch.use_deterministic_algorithms(True, warn_only=True)
    with pytest.warns(UserWarning, match="does not have a deterministic implementation"):
        (got,) = torch.autograd.grad(warp(fr, flow), (fr,), grad_outputs=g)
    assert float((got - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


# ---------------------------------------------------------------------------------------------------- live reference

LIVE_STEP = textwrap.dedent("""
    import hashlib, json, sys
    sys.path.insert(0, {tests!r})
    import overlay_probe
    import torch
    overlay_probe.stub_third_party()
    overlay_probe.set_path("patch", {ref!r})
    import model
    import ofb200
    ofb200.patch_reference()
    import model.raft as raft_mod
    ns = sys.modules.get("model._reference_raft", raft_mod)
    torch.use_deterministic_algorithms(True)
    digests = []
    for rep in range(2):
        torch.manual_seed(1234)
        net = model.RAFT().cuda().train()
        g = torch.Generator(device="cuda").manual_seed(99)
        img0 = torch.rand((1, 3, 128, 192), device="cuda", generator=g) * 255.0
        img1 = torch.roll(img0, shifts=(2, -3), dims=(2, 3))
        gt = 2 * torch.randn((1, 2, 128, 192), device="cuda", generator=g)
        valid = torch.ones((1, 128, 192), device="cuda")
        preds = net(img0, img1, iters=12)
        loss = ns.sequence_loss(preds, gt, valid)[0]
        loss.backward()
        h = hashlib.sha256()
        for p in net.parameters():
            if p.grad is not None:
                h.update(p.grad.detach().cpu().numpy().tobytes())
        digests.append(h.hexdigest())
    print(json.dumps({{"digests": digests}}))
""")


def test_reference_raft_training_step_repeats_under_the_flag(det_flags):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from stage_reference import find_reference

    ref = find_reference()
    if ref is None:
        pytest.skip("no checkout of the upstream torch-optical-flow project: set OFB200_REFERENCE to one, or stage it "
                    "under oracle/_ref/ (tools/stage_reference.py)")
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    env.pop("PYTHONPATH", None)
    script = LIVE_STEP.format(tests=os.path.join(ROOT, "tests"), ref=ref)
    res = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-2000:] + "\n" + res.stderr[-4000:]
    import json

    d = json.loads(res.stdout.strip().splitlines()[-1])["digests"]
    assert d[0] == d[1]
