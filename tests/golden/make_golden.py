"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU.

`OFB200_REFERENCE=<checkout> python tests/golden/make_golden.py`; the tests themselves need
only the stored vectors.  Every array stored here is an input or an output of a reference call;
the reference call that produced it is named in the `ref_call` string of each case.

The lookup *index / validity* vectors are produced by replaying, with eager torch fp32 ops,
exactly the expressions the reference evaluates (methods/raft/model/utils.py:70-71,77 and
ATen GridSampler.h:30) -- the reference never returns its floor indices, so this is the
index oracle (SURVEY.md section 8c).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from _refimport import load_reference  # noqa: E402

torch.manual_seed(0)
torch.set_num_threads(1)
of, corr_mod, utils, RAFT = load_reference()
from optical_flow.metrics import AverageEndPointError  # noqa: E402
from optical_flow.metrics.epe import end_point_error  # noqa: E402
from optical_flow.operator.operator import warp_grid  # noqa: E402


def g(seed):
    return torch.Generator().manual_seed(seed)


def save(name, **arrays):
    out = {}
    for k, v in arrays.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        out[k] = v
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


# ------------------------------------------------------------------ warp (operator.py:8-56)
def make_warp():
    cases = {}
    idx = 0
    for (b, c, h, w, sigma) in [(2, 3, 17, 23, 3.0), (1, 1, 9, 40, 12.0), (1, 4, 33, 6, 1.0), (1, 3, 1, 7, 2.0), (1, 2, 5, 1, 2.0)]:
        frame = torch.rand(b, c, h, w, generator=g(10 + idx))
        flow_px = sigma * torch.randn(b, 2, h, w, generator=g(20 + idx))
        flow = of.normalize(flow_px)
        cases[f"frame{idx}"] = frame
        cases[f"flow_px{idx}"] = flow_px
        cases[f"flow{idx}"] = flow
        cases[f"out{idx}"] = of.warp(frame, flow)
        cases[f"grid{idx}"] = warp_grid(flow.permute(0, 2, 3, 1))
        idx += 1
    cases["n"] = np.int64(idx)
    # every mode / padding / align_corners combination the kernel implements
    frame = torch.rand(2, 3, 12, 15, generator=g(31))
    flow = of.normalize(4.0 * torch.randn(2, 2, 12, 15, generator=g(32)))
    cases["opt_frame"] = frame
    cases["opt_flow"] = flow
    for mode in ("bilinear", "nearest"):
        for pad in ("zeros", "border", "reflection"):
            for ac in (False, True):
                cases[f"opt_{mode}_{pad}_{int(ac)}"] = of.warp(frame, flow, mode=mode, padding_mode=pad, align_corners=ac)
    save("warp", ref_call="optical_flow.warp(frame, optical_flow.normalize(flow_px)); warp_grid", **cases)


# ------------------------------------------------------------------ warp gradients (autograd through operator.py:8-56)
def make_warp_grad():
    """d(sum(weight * warp(frame, flow)))/d frame and /d flow from autograd through the UNMODIFIED reference warp."""
    cases = {}
    frame0 = torch.rand(2, 3, 12, 16, generator=g(90))
    flow0 = of.normalize(5.0 * torch.randn(2, 2, 12, 16, generator=g(91)))
    weight = torch.randn(2, 3, 12, 16, generator=g(92))
    cases.update(frame=frame0, flow=flow0, weight=weight)
    for pad in ("zeros", "border", "reflection"):
        for ac in (False, True):
            frame, flow = frame0.clone().requires_grad_(True), flow0.clone().requires_grad_(True)
            out = of.warp(frame, flow, padding_mode=pad, align_corners=ac)
            (out * weight).sum().backward()
            cases[f"dframe_{pad}_{int(ac)}"], cases[f"dflow_{pad}_{int(ac)}"] = frame.grad, flow.grad
    save("warp_grad", ref_call="autograd of (weight * optical_flow.warp(frame, flow, padding_mode, align_corners)).sum()", **cases)


# ------------------------------------------- scale / normalize / resize / integrate / upflow8
def make_resize():
    cases = {}
    flow = 10.0 * torch.randn(2, 2, 9, 13, generator=g(40))
    cases["flow"] = flow
    cases["scale_2"] = of.scale(flow, 2)
    cases["scale_3_m1"] = of.scale(flow, (3, -1))
    cases["normalize"] = of.normalize(flow)
    cases["denormalize"] = of.denormalize(flow)
    cases["resize_20_31"] = of.resize(flow, size=(20, 31))
    cases["resize_4_5"] = of.resize(flow, size=(4, 5))
    cases["resize_9_13"] = of.resize(flow, size=(9, 13))
    cases["resize_sf2"] = of.resize(flow, scale_factor=2)
    cases["resize_sf2p5"] = of.resize(flow, scale_factor=2.5)
    cases["resize_sf0p5"] = of.resize(flow, scale_factor=0.5)
    small = 5.0 * torch.randn(2, 2, 6, 11, generator=g(41))
    cases["small"] = small
    cases["upflow8"] = utils.upflow8(small)
    f1 = of.normalize(2.0 * torch.randn(1, 2, 10, 14, generator=g(42)))
    f2 = of.normalize(2.0 * torch.randn(1, 2, 10, 14, generator=g(43)))
    f3 = of.normalize(2.0 * torch.randn(1, 2, 10, 14, generator=g(44)))
    cases["int_f1"], cases["int_f2"], cases["int_f3"] = f1, f2, f3
    cases["integrate"] = of.integrate(f1, f2, f3)
    save("resize", ref_call="optical_flow.scale/normalize/denormalize/resize/integrate; model.utils.upflow8", **cases)


# -------------------------------------------------- CorrBlock (corr.py:38-87, utils.py:64-86)
def lookup_index_oracle(coords, pyramid, radius):
    """floor indices and validity bits of every lookup tap, replayed with eager torch fp32 ops."""
    b, _, h, w = coords.shape
    d = 2 * radius + 1
    c = coords.permute(0, 2, 3, 1).reshape(b * h * w, 2)
    off = torch.linspace(-radius, radius, d)
    idx = torch.empty(b * h * w, len(pyramid), 2, d, dtype=torch.int32)
    valid = torch.empty(b * h * w, len(pyramid), d * d, dtype=torch.uint8)
    for lvl, p in enumerate(pyramid):
        H, W = p.shape[-2:]
        cen = c / 2 ** lvl
        x = cen[:, 0:1] + off[None]            # (Q, d)  x + dy[i]   (corr.py:66-70)
        y = cen[:, 1:2] + off[None]            # (Q, d)  y + dx[j]
        xg = 2 * x / (W - 1) - 1               # utils.py:70
        yg = 2 * y / (H - 1) - 1               # utils.py:71
        ix = ((xg + 1) / 2) * (W - 1)          # GridSampler.h:30
        iy = ((yg + 1) / 2) * (H - 1)
        idx[:, lvl, 0] = torch.floor(ix).to(torch.int32)
        idx[:, lvl, 1] = torch.floor(iy).to(torch.int32)
        m = (xg[:, :, None] > -1) & (yg[:, None, :] > -1) & (xg[:, :, None] < 1) & (yg[:, None, :] < 1)  # utils.py:77
        valid[:, lvl] = m.reshape(-1, d * d).to(torch.uint8)
    return idx, valid


def make_corr():
    cases = {}
    # main case: default CorrBlock (4 levels, radius 4) on a 16x16 feature grid
    b, c, h, w = 1, 64, 16, 16
    f1 = torch.randn(b, c, h, w, generator=g(50))
    f2 = torch.randn(b, c, h, w, generator=g(51))
    blk = corr_mod.CorrBlock(f1, f2, num_levels=4, radius=4)
    cases["fmap1"], cases["fmap2"] = f1, f2
    cases["volume_shape"] = np.array(corr_mod.CorrBlock.corr(f1, f2).shape)
    for i, p in enumerate(blk.corr_pyramid):
        cases[f"pyr{i}"] = p
    grid = utils.coords_grid(b, h, w)
    cases["coords_grid"] = grid
    coord_sets = {
        "int": grid.clone(),                                                  # RAFT iteration 0
        "noise": grid + 2.5 * torch.randn(b, 2, h, w, generator=g(52)),
    }
    for name, co in coord_sets.items():
        cases[f"coords_{name}"] = co
        cases[f"lookup_{name}"] = blk(co)
        idx, valid = lookup_index_oracle(co, blk.corr_pyramid, 4)
        cases[f"idx_{name}"] = idx
        cases[f"valid_{name}"] = valid
    # batch 2, non-square, 3 levels: far-out-of-bounds and half-pixel coordinates
    b, c, h, w = 2, 32, 8, 14
    f1 = torch.randn(b, c, h, w, generator=g(150))
    f2 = torch.randn(b, c, h, w, generator=g(151))
    blk = corr_mod.CorrBlock(f1, f2, num_levels=3, radius=4)
    cases["b2_fmap1"], cases["b2_fmap2"] = f1, f2
    for i, p in enumerate(blk.corr_pyramid):
        cases[f"b2_pyr{i}"] = p
    grid = utils.coords_grid(b, h, w)
    coord_sets = {
        "far": grid + 15.0 * torch.randn(b, 2, h, w, generator=g(53)),        # many taps out of bounds
        "half": grid + 0.5,
    }
    for name, co in coord_sets.items():
        cases[f"coords_{name}"] = co
        cases[f"lookup_{name}"] = blk(co)
        idx, valid = lookup_index_oracle(co, blk.corr_pyramid, 4)
        cases[f"idx_{name}"] = idx
        cases[f"valid_{name}"] = valid
    # odd sizes: pyramid floor semantics 13x21 -> 6x10 -> 3x5 -> 1x2 ; radius 3, 3 levels
    f1o = torch.randn(1, 32, 13, 21, generator=g(54))
    f2o = torch.randn(1, 32, 13, 21, generator=g(55))
    blk_o = corr_mod.CorrBlock(f1o, f2o, num_levels=3, radius=3)
    co = utils.coords_grid(1, 13, 21) + 3.0 * torch.randn(1, 2, 13, 21, generator=g(56))
    cases["odd_fmap1"], cases["odd_fmap2"], cases["odd_coords"] = f1o, f2o, co
    for i, p in enumerate(blk_o.corr_pyramid):
        cases[f"odd_pyr{i}"] = p
    cases["odd_lookup"] = blk_o(co)
    idx, valid = lookup_index_oracle(co, blk_o.corr_pyramid, 3)
    cases["odd_idx"], cases["odd_valid"] = idx, valid
    # bilinear_sampler with mask=True (utils.py:76-78)
    img = torch.rand(3, 2, 7, 9, generator=g(57))
    pts = torch.rand(3, 5, 4, 2, generator=g(58)) * torch.tensor([10.0, 8.0]) - 1.0
    pts[0, 0, 0] = torch.tensor([0.0, 0.0])
    pts[0, 0, 1] = torch.tensor([8.0, 6.0])
    pts[0, 0, 2] = torch.tensor([4.0, 3.0])
    s, m = utils.bilinear_sampler(img, pts, mask=True)
    cases["bs_img"], cases["bs_pts"], cases["bs_out"], cases["bs_mask"] = img, pts, s, m
    save("corr", ref_call="model.corr.CorrBlock(f1,f2)(coords); CorrBlock.corr; model.utils.bilinear_sampler/coords_grid", **cases)


# ------------------------------------------------------ convex upsample (raft.py:73-85) + EPE
def make_upsample_epe():
    cases = {}
    flow = 2.0 * torch.randn(2, 2, 6, 9, generator=g(60))
    mask = 3.0 * torch.randn(2, 576, 6, 9, generator=g(61))
    cases["flow"], cases["mask"] = flow, mask
    cases["up"] = RAFT.upsample_flow(flow, mask)
    pred = 3.0 * torch.randn(3, 2, 11, 17, generator=g(62))
    target = pred + torch.randn(3, 2, 11, 17, generator=g(63))
    valid = (torch.rand(3, 11, 17, generator=g(64)) > 0.2).float()
    cases["pred"], cases["target"], cases["valid"] = pred, target, valid
    cases["epe_map"] = end_point_error(pred, target, reduce=False)
    cases["epe_mean"] = end_point_error(pred, target)
    m = AverageEndPointError()
    m.update(pred, target, valid)
    cases["m1_sum"], cases["m1_total"], cases["m1_compute"] = m.sum_epe.clone(), m.total.clone(), m.compute()
    m.update(pred * 0.5, target)
    cases["m2_sum"], cases["m2_total"], cases["m2_compute"] = m.sum_epe.clone(), m.total.clone(), m.compute()
    # OutlierRatio (f1.py): flows large enough that the 3 px / 5 % thresholds split the pixels
    from optical_flow.metrics.f1 import OutlierRatio
    f1_target = 8.0 * torch.randn(3, 2, 11, 17, generator=g(65))
    f1_pred = f1_target + 3.0 * torch.randn(3, 2, 11, 17, generator=g(66))
    f1_target[0, :, 0, 0] = 0.0                      # |target| = 0: epe / 0 = inf (an outlier when epe > 3)
    cases["f1_pred"], cases["f1_target"] = f1_pred, f1_target
    fm = OutlierRatio(abs_threshold=3.0, rel_threshold=0.05)
    fm.update(f1_pred, f1_target, valid)
    cases["f1a_sum"], cases["f1a_total"], cases["f1a_compute"] = fm.sum_outliers.clone(), fm.total.clone(), fm.compute()
    fm.update(f1_pred, f1_target)
    cases["f1b_sum"], cases["f1b_total"], cases["f1b_compute"] = fm.sum_outliers.clone(), fm.total.clone(), fm.compute()
    save("upsample_epe", ref_call="RAFT.upsample_flow; optical_flow.metrics.epe.end_point_error / AverageEndPointError", **cases)


# ------------------------------------------------------ sequence_loss (raft.py:231-260)
def make_sequence_loss():
    from model.raft import sequence_loss

    cases = {}
    gt = 6.0 * torch.randn(2, 2, 20, 28, generator=g(80))
    gt[0, :, 3, 4] = 500.0                                   # |gt| >= max_flow: dropped
    valid = (torch.rand(2, 20, 28, generator=g(81)) > 0.25).float()
    preds = [gt + (3.0 / (i + 1)) * torch.randn(2, 2, 20, 28, generator=g(82 + i)) for i in range(5)]
    loss, metrics = sequence_loss(preds, gt, valid)
    cases.update(gt=gt, valid=valid, preds=torch.stack(preds), loss=loss,
                 m=torch.tensor([metrics["1px"], metrics["3px"], metrics["5px"]], dtype=torch.float64))
    loss2, metrics2 = sequence_loss(preds[:1], gt, valid, gamma=0.5, max_flow=10.0)
    cases.update(loss2=loss2, m2=torch.tensor([metrics2["1px"], metrics2["3px"], metrics2["5px"]], dtype=torch.float64))
    save("sequence_loss", ref_call="model.raft.sequence_loss(flow_preds, flow_gt, valid, gamma, max_flow)", **cases)


# ------------------------------------------------------ gradients of upsample_flow / sequence_loss (autograd)
def make_raft_grad():
    """Gradients autograd produces through the UNMODIFIED RAFT.upsample_flow and sequence_loss."""
    from model.raft import sequence_loss

    cases = {}
    flow = (2.0 * torch.randn(2, 2, 5, 7, generator=g(100))).requires_grad_(True)
    mask = (3.0 * torch.randn(2, 576, 5, 7, generator=g(101))).requires_grad_(True)
    weight = torch.randn(2, 2, 40, 56, generator=g(102))
    (RAFT.upsample_flow(flow, mask) * weight).sum().backward()
    cases.update(up_flow=flow.detach(), up_mask=mask.detach(), up_weight=weight, up_dflow=flow.grad, up_dmask=mask.grad)
    gt = 6.0 * torch.randn(2, 2, 12, 20, generator=g(103))
    gt[1, :, 2, 3] = 900.0
    valid = (torch.rand(2, 12, 20, generator=g(104)) > 0.25).float()
    preds = [(gt + (2.0 / (i + 1)) * torch.randn(2, 2, 12, 20, generator=g(105 + i))).requires_grad_(True) for i in range(4)]
    preds[1].data[0, 0, 0, 0] = gt[0, 0, 0, 0]               # an exact zero difference: sign(0) = 0
    loss, _ = sequence_loss(preds, gt, valid, gamma=0.8)
    (3.0 * loss).backward()
    cases.update(sl_gt=gt, sl_valid=valid, sl_preds=torch.stack([p.detach() for p in preds]),
                 sl_dpreds=torch.stack([p.grad for p in preds]))
    save("raft_grad", ref_call="autograd through RAFT.upsample_flow and model.raft.sequence_loss", **cases)


# ------------------------------------------------------ gradients of the correlation block (autograd)
def make_corr_grad():
    """d(sum_k weight_k * CorrBlock(fmap1, fmap2)(coords_k))/d fmap1, /d fmap2 through the UNMODIFIED reference
    (matmul, avg_pool2d chain, grid_sample), two lookups accumulating into the same pyramid."""
    cases = {}
    b, c, h, w = 1, 64, 16, 20
    f1 = torch.randn(b, c, h, w, generator=g(120)).requires_grad_(True)
    f2 = torch.randn(b, c, h, w, generator=g(121)).requires_grad_(True)
    base = utils.coords_grid(b, h, w)
    blk = corr_mod.CorrBlock(f1, f2, num_levels=4, radius=4)
    total = 0.0
    for k in range(2):
        coords = base + 3.0 * torch.randn(b, 2, h, w, generator=g(122 + k))
        if k == 0:
            coords[0, :, 0, :4] = base[0, :, 0, :4]           # integer coordinates (RAFT's first iteration)
            coords[0, 0, 3, 3] = -40.0                        # a window entirely outside
        weight = torch.randn(b, 4 * 81, h, w, generator=g(130 + k))
        total = total + (blk(coords) * weight).sum()
        cases[f"coords{k}"], cases[f"weight{k}"] = coords, weight
    total.backward()
    cases.update(fmap1=f1.detach(), fmap2=f2.detach(), dfmap1=f1.grad, dfmap2=f2.grad)
    save("corr_grad", ref_call="autograd through CorrBlock(fmap1, fmap2, 4, 4)(coords) x2", **cases)


# ------------------------------------------------------ RAFT.forward trace (raft.py:87-147)
def make_raft_trace():
    """Run the UNMODIFIED reference RAFT (random weights, eval mode) on one small image pair and record
    every tensor that crosses the hot-path boundary inside forward(): the feature maps handed to
    CorrBlock (raft.py:112), the coordinates and result of each corr_fn call (raft.py:128), the inputs
    and result of each upsample_flow call (raft.py:140).  The GPU test replays those calls on the B200
    kernels (section 8f, row 1: the accelerated block inside the unmodified model)."""
    import model.raft as raft_mod

    torch.manual_seed(1234)
    net = RAFT()
    net.eval()
    rec = {"coords": [], "corr": [], "up_flow": [], "up_mask": [], "up_out": []}

    class Recorder(corr_mod.CorrBlock):
        def __init__(self, fmap1, fmap2, num_levels=4, radius=4):
            rec["fmap1"], rec["fmap2"] = fmap1.clone(), fmap2.clone()
            super().__init__(fmap1, fmap2, num_levels=num_levels, radius=radius)

        def __call__(self, coords):
            out = super().__call__(coords)
            rec["coords"].append(coords.clone())
            rec["corr"].append(out.clone())
            return out

    orig_up = RAFT.upsample_flow

    def up(flow, mask):
        out = orig_up(flow, mask)
        rec["up_flow"].append(flow.clone()); rec["up_mask"].append(mask.clone()); rec["up_out"].append(out.clone())
        return out

    raft_mod.CorrBlock = Recorder
    net.upsample_flow = up
    img0 = 255.0 * torch.rand(1, 3, 128, 192, generator=g(70))   # 16x24 features: level 3 is 2x3 (1x1 would divide by zero, utils.py:70)
    img1 = torch.roll(img0, shifts=(2, -3), dims=(2, 3)) + 4.0 * torch.randn(1, 3, 128, 192, generator=g(71))
    with torch.no_grad():
        flow_lo, flow_up = net(img0, img1, iters=2, test_mode=True)
    raft_mod.CorrBlock = corr_mod.CorrBlock
    save("raft_trace", ref_call="RAFT()(img0, img1, iters=2, test_mode=True), hooks on CorrBlock / upsample_flow",
         fmap1=rec["fmap1"], fmap2=rec["fmap2"], coords=torch.stack(rec["coords"]), corr=torch.stack(rec["corr"]),
         up_flow=torch.stack(rec["up_flow"]), up_mask=torch.stack(rec["up_mask"]), up_out=torch.stack(rec["up_out"]),
         flow_lo=flow_lo, flow_up=flow_up)


if __name__ == "__main__":
    if sys.argv[1:] == ["raft_trace"]:
        make_raft_trace()
        sys.exit(0)
    if sys.argv[1:] == ["sequence_loss"]:
        make_sequence_loss()
        sys.exit(0)
    if sys.argv[1:] == ["warp_grad"]:
        make_warp_grad()
        sys.exit(0)
    if sys.argv[1:] == ["raft_grad"]:
        make_raft_grad()
        sys.exit(0)
    if sys.argv[1:] == ["corr_grad"]:
        make_corr_grad()
        sys.exit(0)
    make_warp()
    make_warp_grad()
    make_resize()
    make_corr()
    make_upsample_epe()
    make_sequence_loss()
    make_raft_grad()
    make_corr_grad()
    make_raft_trace()
