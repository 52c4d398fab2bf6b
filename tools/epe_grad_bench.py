"""end_point_error forward + backward: this library's kernels (`ofb_epe_reduce_f32` / `ofb_epe_map_f32`, then
`ofb_epe_backward_f32`) against autograd through the reference's expression `torch.norm(pred - target, p=2, dim=1)`
[`.mean()`] on stock torch CUDA ops, the two arms alternating in one process, plus the backward kernel alone.

    python tools/epe_grad_bench.py [--reps 20] [--warmup 3] [--shapes c4,bench] [--label TEXT] [--out FILE]

Shapes (full-resolution flows, (B, 2, H, W)): `c4` = B = 16, 376 x 1248; `bench` = bench.py's 8 pairs at 1088 x 1920.
Cases: both inputs requiring grad or `pred` only, reduce True (mean; upstream gradient 1) or False (map; a random
upstream map).  Each timed window runs SETS calls, each on its own (pred, target) pair, SETS x 8 bytes per pixel of
inputs (0.48 GB at c4, 1.07 GB at bench) against 126 MB of L2, so every call streams from HBM.  Each window starts
behind a ~20 ms spin kernel (torch.cuda._sleep), so every launch is queued before the first runs and the time is the
GPU's, not Python autograd's; `host_bound_reps` counts windows the GPU reached before the last launch was queued
(expected 0).  Per case: median / min / mean per call (ms) of each arm and their ratio, the backward kernel alone
(median per call) with its algorithmic bytes per pixel -- 16 read, + 4 for a map gradient, + 8 written per requested
gradient -- the rate that reaches and its share of 6565.5 GB/s (the HBM copy rate DESIGN.md section 4 divides by), and
the largest difference between the arms' gradients in units of the upstream gradient |g| (the kernel's contract:
<= 2^-21).  The first line names the GPU, its power limit and max SM clock, read in the same run."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import ofb200  # noqa: E402
from ofb200.ops.epe import end_point_error  # noqa: E402
from pyramid_dtype_bench import Window, gpu_info  # noqa: E402

SHAPES = {"c4": (16, 376, 1248), "bench": (8, 1088, 1920)}
SETS = 4
PEAK_GBS = 6565.5
SLEEP_CYCLES = 40_000_000          # ~20 ms at 1965 MHz: longer than queueing one window of either arm
CASES = [(who, reduce) for who in ("both", "pred") for reduce in (True, False)]


def stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}


def bwd_bytes(who, reduce):
    return 16 + (0 if reduce else 4) + 8 * (2 if who == "both" else 1)


def ours(p, t, reduce):
    return end_point_error(p, t, reduce=reduce)


def reference(p, t, reduce):
    n = torch.norm(p - t, p=2, dim=1)
    return n.mean() if reduce else n


def step(fn, p, t, g, who, reduce):
    inputs = (p, t) if who == "both" else (p,)
    return torch.autograd.grad(fn(p, t, reduce), inputs, grad_outputs=g)


def time_windows(arms, reps, warmup):
    """arms: name -> fn() running one window's work; alternating order every repetition -> per-arm window times."""
    times = {key: [] for key in arms}
    host_bound = {key: 0 for key in arms}
    keys = list(arms)
    for r in range(warmup + reps):
        for key in (keys if r % 2 == 0 else reversed(keys)):
            torch.cuda._sleep(SLEEP_CYCLES)
            with Window() as win:
                arms[key]()
            reached = win.e0.query()
            torch.cuda.synchronize()
            if r >= warmup:
                times[key].append(win.ms() / SETS)
                host_bound[key] += int(reached)
    return times, host_bound


def bench_shape(name, reps, warmup):
    b, h, w = SHAPES[name]
    px = b * h * w
    gen = torch.Generator(device="cuda").manual_seed(2031)
    preds = [4 * torch.randn((b, 2, h, w), device="cuda", generator=gen) for _ in range(SETS)]
    targets = [4 * torch.randn((b, 2, h, w), device="cuda", generator=gen) for _ in range(SETS)]
    maps = [torch.randn((b, h, w), device="cuda", generator=gen) for _ in range(SETS)]
    one = torch.ones((), device="cuda")
    lib = ofb200.load()
    recs = []
    for who, reduce in CASES:
        ps = [p.requires_grad_(True) for p in preds]
        ts = [t.requires_grad_(who == "both") for t in targets]
        gs = [one] * SETS if reduce else maps

        def arm(fn):
            return lambda: [step(fn, ps[k], ts[k], gs[k], who, reduce) for k in range(SETS)]

        d_p = torch.empty_like(preds[0])
        d_t = torch.empty_like(preds[0]) if who == "both" else None

        def kernel_only():
            for k in range(SETS):
                rc = lib.ofb_epe_backward_f32(ofb200.ptr(preds[k]), ofb200.ptr(targets[k]), ofb200.ptr(gs[k]), int(reduce),
                                              ofb200.ptr(d_p), ofb200.ptr(d_t), b, h, w, ofb200.stream_ptr())
                ofb200.check(rc, "ofb_epe_backward_f32")

        times, host_bound = time_windows({"ofb200": arm(ours), "torch": arm(reference), "bwd_kernel": kernel_only},
                                         reps, warmup)
        got = step(ours, ps[0], ts[0], gs[0], who, reduce)
        ref = step(reference, ps[0], ts[0], gs[0], who, reduce)
        g_abs = float(gs[0].abs().max()) / (px if reduce else 1)
        diff = max(float((a - r).abs().max()) for a, r in zip(got, ref)) / g_abs
        per = statistics.median(times["bwd_kernel"])
        gbs = bwd_bytes(who, reduce) * px / (per * 1e-3) / 1e9
        rec = {"shape": name, "B": b, "H": h, "W": w, "grad": who, "reduce": reduce, "reps": reps, "sets": SETS,
               "ofb200_ms": stats(times["ofb200"]), "torch_ms": stats(times["torch"]),
               "ofb200_over_torch": round(statistics.median(times["ofb200"]) / statistics.median(times["torch"]), 3),
               "bwd_kernel_ms": stats(times["bwd_kernel"]), "bwd_bytes_per_px": bwd_bytes(who, reduce),
               "bwd_GB_s": round(gbs, 1), "bwd_frac_of_6565_GB_s": round(gbs / PEAK_GBS, 3),
               "max_grad_diff_over_g": diff, "within_2^-21": diff <= 2.0 ** -21,
               "host_bound_reps": host_bound}
        recs.append(rec)
        del got, ref
    for p in preds + targets:
        p.requires_grad_(False)
    del preds, targets, maps
    torch.cuda.empty_cache()
    return recs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c4,bench")
    ap.add_argument("--label", default=None, help="added to every JSON line as \"label\" (e.g. the build measured)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("epe_grad_bench.py needs a CUDA device (B200)")
    if args.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")
    ofb200.load()
    tag = {"label": args.label} if args.label else {}
    lines = [dict(gpu_info(), **tag)]
    print(json.dumps(lines[0]), flush=True)
    for name in args.shapes.split(","):
        for rec in bench_shape(name, args.reps, args.warmup):
            rec = dict(rec, **tag)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
