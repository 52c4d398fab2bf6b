"""The convex upsampling's backward with a half-precision mask: `ofb_convex_upsample_backward` and `upsample_flow`.

Under the reference's `precision: 16` the mask head's output is fp16 or bf16 and the softmax of raft.py:78 autocasts it
to fp32, so the reference's mask gradient is its fp32 softmax backward rounded once to the mask's dtype.  The kernel
widens each 16-bit logit exactly, computes d_mask in fp32 with the fp32 kernel's arithmetic and rounds it once, so:
  kernel     d_mask of a 16-bit mask == the fp32 kernel's d_mask on the widened mask, cast (`.to(dtype)`), bit for bit,
             NaN at the same positions, fp16 beyond +-65504 -> inf; d_flow (fp32, summed with atomics) within 1e-5 max|ref|
  surface    upsample_flow(flow, half_mask) differentiates like upsample_flow(flow, half_mask.float()), without the cast:
             the same mask-gradient bits in the mask's dtype, no fp32 copy of the mask kept for backward or made in it
  autocast   a stand-in for the mask head under torch.autocast gets the parameter gradients of the explicit cast path
"""
import os

import pytest
import torch

gpu = pytest.mark.gpu
HALF = {"fp16": torch.float16, "bf16": torch.bfloat16}
OFB_OK, OFB_EINVAL, OFB_EUNSUPPORTED, OFB_EALIGN = 0, -1, -2, -3
BAD_DTYPES = (-1, 3, 4, 99)          # 3 = OFB_DTYPE_F64
ALLOC_GRANULE = 512                  # the CUDA caching allocator rounds every block to 512 bytes


def bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}[t.dtype])


def dtype_code(dt):
    import ofb200

    return {torch.float32: ofb200.DTYPE_F32, torch.float16: ofb200.DTYPE_F16, torch.bfloat16: ofb200.DTYPE_BF16}[dt]


def assert_cast_equal(got, ref32, what):
    """got (16-bit) == ref32.to(got.dtype) bit for bit, NaN at the same positions (NaN payloads are not compared)."""
    want = ref32.to(got.dtype)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), what
    assert torch.equal(bits(got)[~nan], bits(want)[~nan]), (what, int((bits(got) != bits(want))[~nan].sum()))


def assert_atomic_close(got, ref, what):
    """d_flow is summed with atomics in an unspecified order: NaN at the same positions, the rest within 1e-5 max|ref|."""
    nan = torch.isnan(ref)
    assert torch.equal(torch.isnan(got), nan), what
    diff = float((got[~nan] - ref[~nan]).abs().max()) if bool((~nan).any()) else 0.0
    assert diff <= 1e-5 * float(ref[~nan].abs().max()), (what, diff)


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


def test_backward_entry_point_validates_arguments_without_launch(lib):
    """ofb_convex_upsample_backward returns OFB_EINVAL for an unknown mask dtype before anything else (empty sizes
    included) and for a null flow, mask or d_out; OFB_OK for empty sizes with null pointers; OFB_EALIGN for a mask or
    d_mask not aligned to its element size and a d_out not 16-byte aligned.  ofb_convex_upsample_backward_f32 returns
    the code of the new entry point with OFB_DTYPE_F32 in every case.  Nothing launches."""
    import ofb200

    fake = 1 << 20                       # 16-byte aligned, never dereferenced: every call below returns before a launch
    f32 = ofb200.DTYPE_F32
    good = (f32, ofb200.DTYPE_F16, ofb200.DTYPE_BF16)

    def call(dt, flow=fake, mask=fake, d_out=fake, d_flow=fake, d_mask=fake, n=2, h=3, w=5):
        return lib.ofb_convex_upsample_backward(flow, mask, dt, d_out, d_flow, d_mask, n, h, w, None)

    def call_f32(flow=fake, mask=fake, d_out=fake, d_flow=fake, d_mask=fake, n=2, h=3, w=5):
        return lib.ofb_convex_upsample_backward_f32(flow, mask, d_out, d_flow, d_mask, n, h, w, None)

    before = lib.ofb_launch_count()
    empty = ({"n": 0}, {"h": 0}, {"w": 0}, {"n": 0, "h": 0, "w": 0})
    nulls = {"flow": None, "mask": None, "d_out": None, "d_flow": None, "d_mask": None}
    for dt in BAD_DTYPES:
        for kw in ({},) + empty:
            assert call(dt, **kw) == OFB_EINVAL, (dt, kw)
            assert call(dt, **nulls, **kw) == OFB_EINVAL, (dt, kw)
    # (arguments, the code each valid dtype returns)
    elem = {f32: 2, ofb200.DTYPE_F16: 1, ofb200.DTYPE_BF16: 1}       # an offset that misaligns the element size
    cases = [({"flow": None}, OFB_EINVAL), ({"mask": None}, OFB_EINVAL), ({"d_out": None}, OFB_EINVAL),
             ({"flow": None, "d_flow": None, "d_mask": None}, OFB_EINVAL), ({"n": -1}, OFB_EINVAL),
             ({"h": -3}, OFB_EINVAL), ({"d_flow": None, "d_mask": None}, OFB_OK), ({"n": 65536}, OFB_EUNSUPPORTED),
             ({"d_out": fake + 8}, OFB_EALIGN), ({"d_out": fake + 4, "d_mask": None}, OFB_EALIGN),
             ({"d_out": fake + 2, "d_flow": None}, OFB_EALIGN)]
    cases += [({**nulls, **kw}, OFB_OK) for kw in empty]
    for dt in good:
        for kw, want in cases + [({"mask": fake + elem[dt]}, OFB_EALIGN), ({"d_mask": fake + elem[dt]}, OFB_EALIGN),
                                 ({"mask": fake + elem[dt], "d_mask": None}, OFB_EALIGN),
                                 ({"d_mask": fake + elem[dt], "d_flow": None}, OFB_EALIGN)]:
            got = call(dt, **kw)
            assert got == want, (dt, kw, got)
            if dt == f32:
                assert call_f32(**kw) == got, kw
    assert lib.ofb_launch_count() == before


# =============================================================================== kernel (GPU)
SHAPES = [(1, 1, 1), (2, 19, 37), (3, 5, 64), (16, 47, 156)]


def inputs(shape, dt, extreme, seed):
    """flow (N,2,h,w), mask (N,576,h,w) in dt, d_out (N,2,8h,8w).  extreme: logits up to 1e4 in magnitude (fp16: up to
    6e4), +inf logits at a few coarse pixels (NaN gradients there), and flow and d_out large enough at one pixel in
    seven that |d_mask| exceeds 65504."""
    n, h, w = shape
    gen = torch.Generator(device="cuda").manual_seed(seed)
    flow = 2 * torch.randn((n, 2, h, w), device="cuda", generator=gen)
    logits = 2 * torch.randn((n, 576, h, w), device="cuda", generator=gen)
    d_out = torch.randn((n, 2, 8 * h, 8 * w), device="cuda", generator=gen)
    if extreme:
        p = torch.arange(h * w, device="cuda").view(1, 1, h, w)
        big = (p % 3 == 1)
        logits = torch.where(big, logits * (6e4 / 8 if dt == torch.float16 else 1e4 / 2), logits)
        logits.view(n, 9, 64, h, w)[:, 2, 5][(p[0, 0] % 11 == 5).expand(n, h, w)] = float("inf")
        huge = (p % 7 == 0)
        flow = torch.where(huge, flow * 500, flow)
        d_out = torch.where(huge.repeat_interleave(8, 2).repeat_interleave(8, 3), d_out * 200, d_out)
    return flow.contiguous(), logits.to(dt).contiguous(), d_out.contiguous()


def run_backward(flow, mask, d_out, want_flow=True, want_mask=True, d_mask=None):
    """ofb_convex_upsample_backward -> (d_flow or None, d_mask or None); d_mask is NaN-filled first unless given."""
    import ofb200

    n, _, h, w = flow.shape
    d_flow = torch.zeros((n, 2, h, w), device="cuda") if want_flow else None
    if want_mask and d_mask is None:
        d_mask = torch.full(mask.shape, float("nan"), dtype=mask.dtype, device="cuda")
    rc = ofb200.load().ofb_convex_upsample_backward(ofb200.ptr(flow), ofb200.ptr(mask), dtype_code(mask.dtype),
                                                    ofb200.ptr(d_out), ofb200.ptr(d_flow), ofb200.ptr(d_mask if want_mask else None),
                                                    n, h, w, ofb200.stream_ptr())
    ofb200.check(rc, "ofb_convex_upsample_backward")
    return d_flow, (d_mask if want_mask else None)


@gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("name", list(HALF))
def test_half_mask_gradient_is_the_cast_fp32_gradient(cuda_lib, name, shape):
    """d_mask of an fp16 / bf16 mask is the fp32 kernel's d_mask on the widened mask, cast, bit for bit (NaN at the same
    positions, fp16 overflow to inf); d_flow matches the fp32 kernel's within the atomics' tolerance.  With d_flow NULL
    the kernel writes the same d_mask bits; with d_mask NULL the same d_flow."""
    dt = HALF[name]
    for extreme in (False, True):
        what = (name, shape, extreme)
        flow, mask, d_out = inputs(shape, dt, extreme, 3000 + sum(shape) + extreme)
        ref_flow, ref_mask = run_backward(flow, mask.float(), d_out)
        d_flow, d_mask = run_backward(flow, mask, d_out)
        assert d_mask.dtype == dt
        assert_cast_equal(d_mask, ref_mask, what)
        assert_atomic_close(d_flow, ref_flow, what)
        _, only_mask = run_backward(flow, mask, d_out, want_flow=False)
        assert torch.equal(bits(only_mask), bits(d_mask)), what
        only_flow, _ = run_backward(flow, mask, d_out, want_mask=False)
        assert_atomic_close(only_flow, ref_flow, what)
        if extreme and shape[1] * shape[2] > 11:
            assert bool(torch.isnan(d_mask).any()), what
            if dt == torch.float16:
                assert bool(torch.isinf(d_mask).any()) and bool(ref_mask.abs().gt(65504).logical_and(ref_mask.isfinite()).any()), what


@gpu
@pytest.mark.parametrize("name", list(HALF))
def test_half_mask_needs_only_element_alignment(cuda_lib, name):
    """A 16-bit mask and d_mask that start 2 bytes past a 4-byte boundary are read and written in place: the same
    d_mask bits as from aligned copies, and nothing outside d_mask is touched."""
    dt = HALF[name]
    flow, mask, d_out = inputs((2, 19, 37), dt, False, 3100)
    _, want = run_backward(flow, mask, d_out)
    mask_buf = torch.empty(mask.numel() + 1, dtype=dt, device="cuda")
    mask_buf[1:] = mask.view(-1)
    out_buf = torch.full((mask.numel() + 2,), 7.0, dtype=dt, device="cuda")
    d_mask = out_buf[1:-1].view(mask.shape)
    mask_odd = mask_buf[1:].view(mask.shape)
    assert mask_odd.data_ptr() % 4 == 2 and d_mask.data_ptr() % 4 == 2
    run_backward(flow, mask_odd, d_out, d_mask=d_mask)
    assert torch.equal(bits(d_mask), bits(want))
    assert float(out_buf[0]) == 7.0 and float(out_buf[-1]) == 7.0


# =============================================================================== upsample_flow (GPU)
def surface_inputs(dt, seed, n=2, h=19, w=37, device="cuda"):
    gen = torch.Generator().manual_seed(seed)
    flow = 2 * torch.randn((n, 2, h, w), generator=gen)
    mask = (2 * torch.randn((n, 576, h, w), generator=gen)).to(dt)
    wgt = torch.randn((n, 2, 8 * h, 8 * w), generator=gen)
    return flow.to(device), mask.to(device), wgt.to(device)


def grads(flow, mask, wgt, flow_grad=True, mask_grad=True, cast=False):
    """(output, d flow, d mask) of sum(upsample_flow(flow, mask) * wgt); cast: the parent's path, mask.float() first."""
    from model.raft import upsample_flow

    f = flow.clone().requires_grad_(flow_grad)
    m = mask.clone().requires_grad_(mask_grad)
    out = upsample_flow(f, m.float() if cast else m)
    (out * wgt).sum().backward()
    return out.detach(), f.grad, m.grad


@gpu
@pytest.mark.parametrize("name", list(HALF))
def test_upsample_flow_half_mask_gradient(cuda_lib, name):
    """The mask gradient of a half mask is, bit for bit, the gradient through upsample_flow(flow, mask.float()) (which
    autograd casts to the mask's dtype), in the mask's dtype; the output is unchanged and the flow gradient matches
    within the atomics' tolerance.  Flow-only and mask-only gradients work."""
    dt = HALF[name]
    flow, mask, wgt = surface_inputs(dt, 3200)
    ref_out, ref_df, ref_dm = grads(flow, mask, wgt, cast=True)
    out, df, dm = grads(flow, mask, wgt)
    assert torch.equal(out, ref_out)
    assert dm.dtype == dt and ref_dm.dtype == dt
    assert torch.equal(bits(dm), bits(ref_dm))
    assert_atomic_close(df, ref_df, name)
    _, only_df, none = grads(flow, mask, wgt, mask_grad=False)
    assert none is None
    assert_atomic_close(only_df, ref_df, name)
    _, none, only_dm = grads(flow, mask, wgt, flow_grad=False)
    assert none is None and torch.equal(bits(only_dm), bits(dm))


@gpu
@pytest.mark.parametrize("name", list(HALF))
def test_upsample_flow_half_mask_gradient_on_host_tensors(cuda_lib, name):
    """Host flow and host half mask: output and gradients arrive on the host, the mask gradient in the mask's dtype with
    the device run's bits."""
    dt = HALF[name]
    flow, mask, wgt = surface_inputs(dt, 3300, device="cpu")
    out, df, dm = grads(flow, mask, wgt)
    assert out.device.type == "cpu" and df.device.type == "cpu" and dm.device.type == "cpu"
    assert dm.dtype == dt
    dev_out, dev_df, dev_dm = grads(flow.cuda(), mask.cuda(), wgt.cuda())
    assert torch.equal(out, dev_out.cpu())
    assert torch.equal(bits(dm), bits(dev_dm.cpu()))
    assert_atomic_close(df, dev_df.cpu(), name)


@gpu
@pytest.mark.parametrize("name", list(HALF))
def test_upsample_flow_half_mask_keeps_no_fp32_copy(cuda_lib, name):
    """A forward with a half mask that requires grad allocates only its output (the graph keeps the caller's mask), and
    the backward's peak adds only the two gradients, d_mask in the mask's dtype: no fp32 mask-sized buffer either way."""
    from model.raft import upsample_flow

    dt = HALF[name]
    flow, mask, _ = surface_inputs(dt, 3400, n=4, h=47, w=156)
    flow.requires_grad_(True)
    mask.requires_grad_(True)
    g = torch.randn((4, 2, 8 * 47, 8 * 156), device="cuda")
    upsample_flow(flow, mask)                            # warm-up: module load, allocator pools
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    out = upsample_flow(flow, mask)
    torch.cuda.synchronize()
    out_bytes = out.numel() * out.element_size()
    assert 0 <= torch.cuda.memory_allocated() - before - out_bytes < ALLOC_GRANULE
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    d_flow, d_mask = torch.autograd.grad(out, (flow, mask), grad_outputs=g)
    torch.cuda.synchronize()
    assert d_mask.dtype == dt
    grad_bytes = d_mask.numel() * d_mask.element_size() + d_flow.numel() * d_flow.element_size()
    fp32_mask_bytes = mask.numel() * 4
    extra = torch.cuda.max_memory_allocated() - base
    assert extra <= grad_bytes + 2 * ALLOC_GRANULE, (extra, grad_bytes, fp32_mask_bytes)


@gpu
@pytest.mark.parametrize("name", list(HALF))
def test_upsample_flow_half_mask_runs_three_kernels(cuda_lib, name):
    """Forward plus backward of upsample_flow with a half mask that requires grad, driven by torch.autograd.grad with a
    precomputed output gradient, runs the two library kernels and the d_flow zero-fill, and no copy or cast."""
    from model.raft import upsample_flow
    from torch.profiler import ProfilerActivity, profile

    dt = HALF[name]
    flow, mask, _ = surface_inputs(dt, 3500)
    flow.requires_grad_(True)
    mask.requires_grad_(True)
    g = torch.randn((2, 2, 8 * 19, 8 * 37), device="cuda")
    torch.autograd.grad(upsample_flow(flow, mask), (flow, mask), grad_outputs=g)        # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        torch.autograd.grad(upsample_flow(flow, mask), (flow, mask), grad_outputs=g)
        torch.cuda.synchronize()
    events = prof.events()
    kernels = [e.name for e in events if e.device_type == torch.autograd.DeviceType.CUDA]
    ops = {e.name for e in events if e.device_type == torch.autograd.DeviceType.CPU}
    assert not ops & {"aten::copy_", "aten::_to_copy"}, sorted(ops)
    assert len(kernels) == 3, kernels
    assert sum("convex_upsample_kernel" in k for k in kernels) == 1, kernels
    assert sum("convex_upsample_bwd_kernel" in k for k in kernels) == 1, kernels
    assert sum(("fill" in k.lower() or "memset" in k.lower()) for k in kernels) == 1, kernels


# =============================================================================== autocast end to end (GPU)
def ulp(ref, dt):
    """The spacing of dt at |ref| (subnormal spacing below the smallest normal)."""
    mant, emin = {torch.float16: (10, -14), torch.bfloat16: (7, -126)}[dt]
    r = ref.float().abs()
    _, e = torch.frexp(torch.where(r > 0, r, torch.ones_like(r)))
    e = torch.where(r > 0, e, torch.full_like(e, emin + 1))
    return torch.exp2((torch.clamp(e - 1, min=emin) - mant).double()).float()


@gpu
@pytest.mark.parametrize("name", list(HALF))
def test_autocast_mask_head_gradients(cuda_lib, name):
    """A stand-in for BasicUpdateBlock's mask head (reference update.py:140-144,160: 3x3 conv -> ReLU -> 1x1 conv to 576
    channels, then .25 *) under torch.autocast, then upsample_flow, a weighted sum and backward: the head's parameter
    gradients and the mask gradient equal those of the explicit mask.float() path bit for bit, the flow gradient is
    within the atomics' tolerance, and the mask gradient is within the fp32 tolerance plus one ulp of the dtype of
    autograd through oracle/torch_port.upsample_flow under the same autocast."""
    from model.raft import upsample_flow
    from oracle import torch_port as tp

    dt = HALF[name]
    n, h, w = 2, 19, 37
    torch.manual_seed(3600)
    head = torch.nn.Sequential(torch.nn.Conv2d(128, 256, 3, padding=1), torch.nn.ReLU(inplace=True),
                               torch.nn.Conv2d(256, 576, 1, padding=0)).cuda()
    gen = torch.Generator(device="cuda").manual_seed(3610)
    net = torch.randn((n, 128, h, w), device="cuda", generator=gen)
    flow = 2 * torch.randn((n, 2, h, w), device="cuda", generator=gen)
    wgt = torch.randn((n, 2, 8 * h, 8 * w), device="cuda", generator=gen)

    def step(upsample, cast):
        head.zero_grad(set_to_none=True)
        f = flow.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=dt):
            mask = .25 * head(net)
            mask.retain_grad()
            loss = (upsample(f, mask.float() if cast else mask) * wgt).sum()
        loss.backward()
        assert mask.dtype == dt and mask.grad.dtype == dt
        return loss.detach(), [p.grad.clone() for p in head.parameters()], f.grad, mask.grad

    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        step(upsample_flow, False)                                                   # warm-up: cuDNN plans
        ref = step(upsample_flow, True)
        got = step(upsample_flow, False)
        oracle = step(tp.upsample_flow, False)
    finally:
        torch.backends.cudnn.deterministic = det
    assert torch.equal(got[0], ref[0])
    for k, (a, b) in enumerate(zip(got[1], ref[1])):
        assert a.dtype == b.dtype and torch.equal(a, b), k
    assert_atomic_close(got[2], ref[2], name)
    assert torch.equal(bits(got[3]), bits(ref[3]))
    want = oracle[3].float()
    err = (got[3].float() - want).abs()
    bound = 2e-5 * max(1.0, float(want.abs().max())) + ulp(want, dt)
    assert bool((err <= bound).all()), float((err - bound).max())
