"""Gradients of `end_point_error` (`ofb_epe_backward_f32`) and of `warp_grid`.

The reference's end_point_error (optical_flow/metrics/epe.py:41-61) is torch.norm(pred - target, p=2, dim=dim), with
`.mean()` when reduce=True.  Autograd through it gives, bit for bit (ATen's norm, mean and subtraction backwards),
    d pred   = g * ((pred - target) / n).masked_fill(n == 0, 0)        d target = -d pred
with n the norm and g the map's upstream gradient, or the mean's divided by the number of pixels.  The kernel replays
that sequence on its own forward map, so it is tested
  * bit for bit against the formula evaluated with torch CUDA ops, n being this library's
    end_point_error(..., reduce=False) and g / N a true division; NaN positions included;
  * against autograd through the reference expression on the GPU and on the CPU: n differs from ATen's by its last bit
    or two (ATen sums x^2 + y^2 in its own order) and CUDA's mean backward multiplies by 1/N where the kernel divides
    by N, so |got - ref| <= 2^-21 |g| per element, on finite pixels with |pred - target| <= 1e3; pixels with
    pred == target get exactly 0 on both sides.
warp_grid (reference operator.py:36-56) is the base grid plus the flow: the flow's gradient is the grid's gradient.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
OFB_OK, OFB_EINVAL = 0, -1
REF_TOL = 2.0 ** -21

# (name, dim, permutation of the (B, 2, H, W) base tensor; "permuted" is a non-contiguous (B, 2, H, W) view of a
# (B, H, W, 2) tensor, "offset" a contiguous (B, 2, H, W) view 4 bytes into its storage)
LAYOUTS = [("b2hw", 1), ("bhw2", -1), ("2bhw", 0), ("bh2w", 2), ("permuted", 1), ("offset", 1)]
# H*W a multiple of 4 (float4 path when aligned), odd (scalar path), a 1-pixel map, an empty batch
SHAPES = [(3, 8, 12), (2, 7, 9), (1, 1, 1), (0, 5, 6)]
WHO = ("pred", "target", "both")


@pytest.fixture(scope="module")
def lib():
    import ofb200

    if not os.path.exists(ofb200.LIB_PATH):
        ofb200.build()
    return ofb200.load()


@pytest.fixture(scope="module")
def cuda_lib(lib):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return lib


# =============================================================================== C ABI (no device)
def test_epe_backward_validates_arguments_without_launch(lib):
    """Zero sizes and two NULL outputs return OK, NULL inputs and negative sizes OFB_EINVAL, all before any launch."""
    fake = ctypes.c_void_p(1 << 20)                      # never dereferenced: every call below returns before a launch

    def call(pred=fake, target=fake, d_epe=fake, scalar=0, d_pred=fake, d_target=fake, b=2, h=4, w=4):
        return lib.ofb_epe_backward_f32(pred, target, d_epe, scalar, d_pred, d_target, b, h, w, None)

    before = lib.ofb_launch_count()
    for scalar in (0, 1):
        for size in ({"b": 0}, {"h": 0}, {"w": 0}):
            assert call(None, None, None, scalar, None, None, **size) == OFB_OK
        assert call(pred=None, scalar=scalar) == OFB_EINVAL
        assert call(target=None, scalar=scalar) == OFB_EINVAL
        assert call(d_epe=None, scalar=scalar) == OFB_EINVAL
        for size in ({"b": -1}, {"h": -1}, {"w": -1}):
            assert call(scalar=scalar, **size) == OFB_EINVAL
        assert call(scalar=scalar, d_pred=None, d_target=None) == OFB_OK
    assert lib.ofb_launch_count() == before


# =============================================================================== helpers
def make_inputs(layout, shape, seed, device="cuda"):
    """(pred, target, dim) in `layout`, from (B, 2, H, W) normals; the first pixel of every batch has pred == target and
    the second pred == target in x only."""
    b, h, w = shape
    gen = torch.Generator().manual_seed(seed)
    base = [3 * torch.randn((b, 2, h, w), generator=gen) for _ in range(2)]
    if b and h * w > 1:
        base[1][:, :, 0, 0] = base[0][:, :, 0, 0]
        base[1][:, 0, 0, 1] = base[0][:, 0, 0, 1]
    elif b:
        base[1][0] = base[0][0]

    def lay(x):
        x = x.to(device)
        if layout == "bhw2":
            return x.permute(0, 2, 3, 1).contiguous()
        if layout == "2bhw":
            return x.permute(1, 0, 2, 3).contiguous()
        if layout == "bh2w":
            return x.permute(0, 2, 1, 3).contiguous()
        if layout == "permuted":
            return x.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
        if layout == "offset":
            buf = torch.empty(x.numel() + 1, device=device)
            buf[1:].copy_(x.flatten())
            return buf[1:].view(x.shape)
        return x.contiguous()

    dim = dict(LAYOUTS)[layout]
    return lay(base[0]), lay(base[1]), dim


def map_shape(x, dim):
    d = dim % x.dim()
    return tuple(x.shape[:d]) + tuple(x.shape[d + 1:])


def upstreams(reduce, shape, seed):
    """(name, fn(out) -> None calling backward) for the upstream gradients a caller hands over."""
    gen = torch.Generator().manual_seed(seed)
    if reduce:
        return [("mean_x0.3", lambda out: (0.3 * out).backward()),
                ("mean_-1.7", lambda out: out.backward(torch.tensor(-1.7, device=out.device)))]
    n = int(np.prod(shape))
    rnd = torch.randn(shape, generator=gen)
    rev = torch.randn(shape[::-1], generator=gen)
    off = torch.randn(n + 1, generator=gen)
    return [("map", lambda out: out.backward(rnd.to(out.device))),
            ("noncontig_map", lambda out: out.backward(rev.to(out.device).permute(*reversed(range(len(shape)))))),
            ("offset_map", lambda out: out.backward(off.to(out.device)[1:].view(shape))),
            ("sum", lambda out: out.sum().backward())]                     # a stride-0 expanded map gradient


def leaf_like(x, requires_grad):
    """A fresh leaf with x's values, sizes, strides and storage offset."""
    extent = 1 + sum((s - 1) * st for s, st in zip(x.shape, x.stride())) if x.numel() else 0
    y = torch.empty(x.storage_offset() + max(extent, 1), device=x.device).as_strided(x.shape, x.stride(), x.storage_offset())
    with torch.no_grad():
        y.copy_(x)
    return y.requires_grad_(requires_grad)


def run_grad(pred, target, dim, reduce, who, fire):
    """end_point_error forward + backward on fresh leaves in the inputs' layout -> (out, d_pred or None,
    d_target or None, the upstream gradient the output received)."""
    from optical_flow.metrics import end_point_error

    p, t = leaf_like(pred, who in ("pred", "both")), leaf_like(target, who in ("target", "both"))
    captured = []
    out = end_point_error(p, t, dim=dim, reduce=reduce)
    assert out.grad_fn is not None
    out.register_hook(lambda g: captured.append(g.detach().clone()))
    fire(out)
    return out.detach(), (p.grad if who != "target" else None), (t.grad if who != "pred" else None), captured[0]


def expected(pred, target, dim, reduce, g):
    """g * ((p - t) / m).masked_fill(m == 0, 0) with torch CUDA ops, m = this library's own end-point-error map."""
    from optical_flow.metrics import end_point_error

    with torch.no_grad():
        p, t = pred.detach().cuda(), target.detach().cuda()
        d = dim % p.dim()
        m = end_point_error(p, t, dim=dim, reduce=False).unsqueeze(d)
        g = g.cuda()
        g = g / torch.tensor(float(m.numel()), device="cuda") if reduce else g.unsqueeze(d)
        return g * ((p - t) / m).masked_fill(m == 0, 0), g


def reference(pred, target, dim, reduce, g, device):
    """Autograd through the reference's torch.norm(pred - target, p=2, dim=dim)[.mean()] on `device`."""
    p = pred.detach().to(device).requires_grad_(True)
    t = target.detach().to(device).requires_grad_(True)
    n = torch.norm(p - t, p=2, dim=dim)
    (n.mean() if reduce else n).backward(g.to(device))
    return p.grad, t.grad


def bits_equal(a, b):
    a, b = a.detach().cpu(), b.detach().cpu()
    if a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na].contiguous().view(torch.int32), b[~nb].contiguous().view(torch.int32))


def check_against_reference(got, pred, target, dim, reduce, g, g_eff, sign):
    """|got - ref| <= 2^-21 |g| on finite pixels with |pred - target| <= 1e3, exactly 0 where pred == target."""
    d = dim % pred.dim()
    delta = (pred.detach().cuda() - target.detach().cuda())
    ok = (torch.isfinite(delta) & (delta.abs() <= 1e3)).all(dim=d, keepdim=True).expand_as(delta)
    same = (delta == 0).all(dim=d, keepdim=True).expand_as(delta)
    bound = REF_TOL * g_eff.abs().expand_as(delta)
    got = got.detach().cuda()
    for device in ("cuda", "cpu"):
        ref = reference(pred, target, dim, reduce, g, device)[0 if sign > 0 else 1].cuda()
        err = (got - ref).abs()
        assert bool((err[ok] <= bound[ok]).all()), (device, float((err[ok] - bound[ok]).max()))
        assert bool((got[same] == 0).all()) and bool((ref[same] == 0).all()), device


# =============================================================================== end_point_error backward
@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("layout", [name for name, _ in LAYOUTS])
def test_epe_grad_layouts(cuda_lib, layout, shape):
    """Every layout x reduce x which input requires grad x upstream gradient: bit for bit the formula on this
    library's map (d target = -d pred exactly), within 2^-21 |g| of the reference's autograd (GPU and CPU), gradients
    in the inputs' shapes and strides-agnostic."""
    pred, target, dim = make_inputs(layout, shape, seed=sum(map(ord, layout)) + sum(shape))
    for reduce in (True, False):
        for name, fire in upstreams(reduce, map_shape(pred, dim), seed=7):
            for who in WHO:
                _, d_pred, d_target, g = run_grad(pred, target, dim, reduce, who, fire)
                want, g_eff = expected(pred, target, dim, reduce, g)
                tag = (layout, shape, reduce, name, who)
                if d_pred is not None:
                    assert d_pred.shape == pred.shape, tag
                    assert bits_equal(d_pred, want), tag
                    check_against_reference(d_pred, pred, target, dim, reduce, g, g_eff, +1)
                if d_target is not None:
                    assert d_target.shape == target.shape, tag
                    assert bits_equal(d_target, -want), tag
                    check_against_reference(d_target, pred, target, dim, reduce, g, g_eff, -1)
                if d_pred is not None and d_target is not None:
                    assert bits_equal(d_target, -d_pred), tag


@gpu
@pytest.mark.parametrize("layout", ["b2hw", "bhw2", "offset"])
def test_epe_grad_non_finite(cuda_lib, layout):
    """inf and NaN in pred or target: NaN exactly where the formula gives NaN, all other bits equal."""
    pred, target, dim = make_inputs(layout, (2, 6, 8), seed=3)
    with torch.no_grad():
        pv, tv = pred.view(-1), target.view(-1)
        pv[5], pv[17], tv[23], tv[40] = float("inf"), float("nan"), float("-inf"), float("nan")
        pv[60], tv[60] = float("inf"), float("inf")
        pv[70] = 3.0e38                                   # overflows the squared sum: n = inf, q = 0 or NaN
    for reduce in (True, False):
        for name, fire in upstreams(reduce, map_shape(pred, dim), seed=11):
            _, d_pred, d_target, g = run_grad(pred, target, dim, reduce, "both", fire)
            want, _ = expected(pred, target, dim, reduce, g)
            assert bool(torch.isnan(want).any()), (layout, reduce, name)
            assert bits_equal(d_pred, want) and bits_equal(d_target, -want), (layout, reduce, name)


@gpu
def test_epe_grad_golden_inputs(cuda_lib, golden):
    """The pred / target the reference's epe_map / epe_mean were recorded from (tests/golden/upsample_epe.npz)."""
    g = golden("upsample_epe")
    pred, target = torch.from_numpy(g["pred"]).cuda(), torch.from_numpy(g["target"]).cuda()
    for reduce in (True, False):
        for name, fire in upstreams(reduce, map_shape(pred, 1), seed=5):
            out, d_pred, d_target, up = run_grad(pred, target, 1, reduce, "both", fire)
            want_out = g["epe_mean"] if reduce else g["epe_map"]
            assert float(np.max(np.abs(out.cpu().numpy() - want_out))) <= 1e-6
            want, g_eff = expected(pred, target, 1, reduce, up)
            assert bits_equal(d_pred, want) and bits_equal(d_target, -want), (reduce, name)
            check_against_reference(d_pred, pred, target, 1, reduce, up, g_eff, +1)
            check_against_reference(d_target, pred, target, 1, reduce, up, g_eff, -1)


@gpu
@pytest.mark.parametrize("layout", ["b2hw", "bhw2", "permuted"])
def test_epe_grad_host_tensors(cuda_lib, layout):
    """Host inputs get host gradients, bit for bit the device ones."""
    pred, target, dim = make_inputs(layout, (2, 7, 12), seed=9)
    hp, ht = make_inputs(layout, (2, 7, 12), seed=9, device="cpu")[:2]
    for reduce in (True, False):
        for name, fire in upstreams(reduce, map_shape(pred, dim), seed=13):
            out_d, dp_d, dt_d, _ = run_grad(pred, target, dim, reduce, "both", fire)
            out_h, dp_h, dt_h, _ = run_grad(hp, ht, dim, reduce, "both", fire)
            assert not out_h.is_cuda and not dp_h.is_cuda and not dt_h.is_cuda, (reduce, name)
            assert bits_equal(out_h, out_d) and bits_equal(dp_h, dp_d) and bits_equal(dt_h, dt_d), (reduce, name)


@gpu
def test_epe_grad_in_a_combined_loss(cuda_lib):
    """sequence_loss + 0.1 * end_point_error: each prediction's gradient is the sum of the two terms' gradients (the
    EPE term is not silently dropped), and the ground truth gets its EPE gradient."""
    from model import sequence_loss
    from optical_flow.metrics import end_point_error

    gen = torch.Generator(device="cuda").manual_seed(21)
    b, h, w = 2, 24, 40
    preds = [(4 * torch.randn((b, 2, h, w), device="cuda", generator=gen)).requires_grad_(True) for _ in range(3)]
    gt = (4 * torch.randn((b, 2, h, w), device="cuda", generator=gen)).requires_grad_(True)
    valid = (torch.rand((b, h, w), device="cuda", generator=gen) > 0.2).float()

    g_seq = torch.autograd.grad(sequence_loss(preds, gt.detach(), valid)[0], preds)
    g_epe_pred, g_epe_gt = torch.autograd.grad(0.1 * end_point_error(preds[-1], gt), (preds[-1], gt))
    loss = sequence_loss(preds, gt.detach(), valid)[0] + 0.1 * end_point_error(preds[-1], gt)
    loss.backward()
    assert bits_equal(preds[-1].grad, g_seq[-1] + g_epe_pred)
    for p, gs in zip(preds[:-1], g_seq[:-1]):
        assert bits_equal(p.grad, gs)
    assert bits_equal(gt.grad, g_epe_gt) and float(g_epe_pred.abs().max()) > 0


@gpu
def test_epe_no_grad_path(cuda_lib):
    """Forward values with inputs requiring grad are bitwise those under torch.no_grad(); nothing requiring grad (or
    no_grad) gives an output without grad_fn and one launch; the metric classes stay non-differentiable."""
    import ofb200
    from optical_flow.metrics import AverageEndPointError, end_point_error

    for layout, shape in (("b2hw", (3, 8, 12)), ("bhw2", (2, 7, 9)), ("permuted", (2, 5, 8))):
        pred, target, dim = make_inputs(layout, shape, seed=17)
        for reduce in (True, False):
            n0 = ofb200.launch_count()
            plain = end_point_error(pred, target, dim=dim, reduce=reduce)
            assert plain.grad_fn is None and ofb200.launch_count() - n0 == 1
            with torch.no_grad():
                n0 = ofb200.launch_count()
                nograd = end_point_error(pred.clone().requires_grad_(True), target, dim=dim, reduce=reduce)
                assert nograd.grad_fn is None and ofb200.launch_count() - n0 == 1
            n0 = ofb200.launch_count()
            withgrad = end_point_error(pred.clone().requires_grad_(True), target, dim=dim, reduce=reduce)
            assert withgrad.grad_fn is not None and ofb200.launch_count() - n0 == 1
            assert bits_equal(withgrad, nograd) and bits_equal(plain, nograd), (layout, reduce)
        metric = AverageEndPointError(dim=dim)
        assert metric(pred.clone().requires_grad_(True), target).grad_fn is None


# =============================================================================== warp_grid backward
@gpu
def test_warp_grid_grad_is_the_incoming_gradient(cuda_lib):
    """d warp_grid / d flow is the identity: flow.grad is bitwise the grid's gradient, on the device and for host
    tensors, for a contiguous flow, a permuted (B, 2, H, W) one and the stride-0 gradient of .sum()."""
    from optical_flow.operator.operator import warp_grid

    gen = torch.Generator().manual_seed(4)
    b, h, w = 2, 9, 14
    base = torch.randn((b, h, w, 2), generator=gen) * 0.1
    g = torch.randn((b, h, w, 2), generator=gen)
    for device in ("cuda", "cpu"):
        flow = base.to(device, copy=True).requires_grad_(True)
        grid = warp_grid(flow)
        assert grid.device.type == device and grid.grad_fn is not None
        grid.backward(g.to(device))
        assert flow.grad.device.type == device and bits_equal(flow.grad, g)
        flow.grad = None
        warp_grid(flow).sum().backward()
        assert bits_equal(flow.grad, torch.ones_like(g))
        chw = base.permute(0, 3, 1, 2).contiguous().to(device).requires_grad_(True)
        warp_grid(chw.permute(0, 2, 3, 1)).backward(g.to(device))
        assert bits_equal(chw.grad, g.permute(0, 3, 1, 2))
