"""Convex upsampling forward + backward (`upsample_flow`, then `torch.autograd.grad` for the flow and the mask) with an
fp32 mask, with a half-precision mask through an fp32 cast (what `precision: 16` ran before the backward read the mask
in its own dtype: `mask.float()`, the fp32 kernels, autograd's cast of d_mask back), and with the half-precision mask
read and its gradient written directly.  12 iterations of each variant (one RAFT forward's worth of upsamplings, each
with its own flow, mask and output gradient) timed with CUDA events, all variants alternating in one process.

    python tools/upsample_mask_dtype_bench.py [--reps 20] [--warmup 3] [--shapes c4,bench] [--label TEXT] [--out FILE]

Shapes (coarse grid): `c4` = B = 16, 47 x 156; `bench` = bench.py's micro-batch (8 pairs, 136 x 240).  Variants:
    fp32                    fp32 mask
    fp16_via_fp32, bf16_via_fp32
                            half mask, upsample_flow(flow, mask.float()): a cast kernel before the forward, the fp32
                            kernels, a cast of the fp32 d_mask after the backward (5 kernels with the d_flow zero-fill)
    fp16, bf16              half mask passed as it is: the forward reads it, the backward reads it and writes d_mask in
                            its dtype (3 kernels)
Per shape one JSON line gives, per variant, the median / min / mean of the 12 iterations (ms), the median per iteration
and the algorithmic HBM bytes per coarse pixel and iteration with the rate they reach and its share of 6565.5 GB/s (the
HBM copy bandwidth measured on a B200, DESIGN.md section 4):
    forward          576 * esize mask + 8 flow + 512 upsampled flow                     fp32 2824 B, 16-bit 1672 B
    backward         576 * esize mask + 8 flow + 512 d_out + 576 * esize d_mask + 8 d_flow   fp32 5136 B, 16-bit 2832 B
    each fp32 cast   576 * (2 + 4)                                                                     3456 B
    so fp32 7960 B, via fp32 14872 B, direct 4504 B.
Each window starts behind a ~20 ms spin kernel (torch.cuda._sleep), so all 12 iterations are queued before the first
runs and the time is the GPU's, not the Python autograd's; `host_bound_reps` counts windows whose start the GPU reached
before the last launch was queued (expected 0).  The run also checks that the timed direct d_mask has the bits of the
via-fp32 d_mask (the fp32 gradient cast).  The first line names the GPU, its power limit and max SM clock, read in the
same run.  Each variant's 12 masks (1.6 GB in fp16 at c4, 3.6 GB at bench) are larger than L2, so every kernel streams
from HBM."""
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
from ofb200.ops.raft_ops import upsample_flow  # noqa: E402
from pyramid_dtype_bench import Window, gpu_info  # noqa: E402

SHAPES = {"c4": (16, 47, 156), "bench": (8, 136, 240)}
ITERS = 12
PEAK_GBS = 6565.5
SLEEP_CYCLES = 40_000_000          # ~20 ms at 1965 MHz: longer than queueing 12 iterations of any variant
HALF = {"fp16": torch.float16, "bf16": torch.bfloat16}


def px_bytes():
    fwd = {es: 576 * es + 8 + 512 for es in (4, 2)}
    bwd = {es: 576 * es + 8 + 512 + 576 * es + 8 for es in (4, 2)}
    cast = 576 * (2 + 4)
    via = cast + fwd[4] + bwd[4] + cast
    return {"fp32": fwd[4] + bwd[4], "fp16_via_fp32": via, "fp16": fwd[2] + bwd[2], "bf16_via_fp32": via,
            "bf16": fwd[2] + bwd[2]}


def stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}


def step(flow, mask, g, cast):
    out = upsample_flow(flow, mask.float() if cast else mask)
    return torch.autograd.grad(out, (flow, mask), grad_outputs=g)


def bench_shape(name, reps, warmup):
    b, h, w = SHAPES[name]
    px = b * h * w
    gen = torch.Generator(device="cuda").manual_seed(2027)
    flows = [(2 * torch.randn((b, 2, h, w), device="cuda", generator=gen)).requires_grad_(True) for _ in range(ITERS)]
    grads = [torch.randn((b, 2, 8 * h, 8 * w), device="cuda", generator=gen) for _ in range(ITERS)]
    logits = [2 * torch.randn((b, 576, h, w), device="cuda", generator=gen) for _ in range(ITERS)]
    masks = {key: [m.to(dt).requires_grad_(True) for m in logits] for key, dt in HALF.items()}
    masks["fp32"] = [m.to(torch.float16).float().requires_grad_(True) for m in logits]
    del logits

    def variant(key, cast):
        return lambda k: step(flows[k], masks[key][k], grads[k], cast)

    variants = {"fp32": variant("fp32", False), "fp16_via_fp32": variant("fp16", True), "fp16": variant("fp16", False),
                "bf16_via_fp32": variant("bf16", True), "bf16": variant("bf16", False)}
    times = {key: [] for key in variants}
    host_bound = {key: 0 for key in variants}
    keys = list(variants)
    for r in range(warmup + reps):
        for key in (keys if r % 2 == 0 else reversed(keys)):             # alternate the order every repetition
            fn = variants[key]
            torch.cuda._sleep(SLEEP_CYCLES)
            with Window() as win:
                for k in range(ITERS):
                    fn(k)
            reached = win.e0.query()
            torch.cuda.synchronize()
            if r >= warmup:
                times[key].append(win.ms())
                host_bound[key] += int(reached)
    pb = px_bytes()
    rec = {"shape": name, "B": b, "h": h, "w": w, "iterations": ITERS, "reps": reps}
    for key, v in times.items():
        per = statistics.median(v) / ITERS
        gbs = pb[key] * px / (per * 1e-3) / 1e9
        rec[key] = {"ms_12": stats(v), "ms_per_iter": round(per, 4), "bytes_per_px": pb[key], "GB_s": round(gbs, 1),
                    "frac_of_6565_GB_s": round(gbs / PEAK_GBS, 3), "host_bound_reps": host_bound[key]}
    med = {key: statistics.median(v) for key, v in times.items()}
    for key in HALF:
        rec[f"{key}_over_{key}_via_fp32"] = round(med[key] / med[f"{key}_via_fp32"], 3)
        rec[f"{key}_over_fp32"] = round(med[key] / med["fp32"], 3)
    # the timed direct d_mask is the via-fp32 d_mask (the fp32 gradient cast) bit for bit; d_flow within the atomics'
    # tolerance (its sums run in an unspecified order)
    k = ITERS - 1
    for key in HALF:
        d_flow, d_mask = step(flows[k], masks[key][k], grads[k], False)
        ref_flow, ref_mask = step(flows[k], masks[key][k], grads[k], True)
        rec[f"{key}_d_mask_bits_equal"] = bool(d_mask.dtype == ref_mask.dtype and torch.equal(d_mask.view(torch.int16),
                                                                                             ref_mask.view(torch.int16)))
        rec[f"{key}_d_flow_max_rel_diff"] = float((d_flow - ref_flow).abs().max() / ref_flow.abs().max())
    del flows, grads, masks
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c4,bench")
    ap.add_argument("--label", default=None, help="added to every JSON line as \"label\" (e.g. the build measured)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("upsample_mask_dtype_bench.py needs a CUDA device (B200)")
    if args.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")
    ofb200.load()
    tag = {"label": args.label} if args.label else {}
    lines = [dict(gpu_info(), **tag)]
    print(json.dumps(lines[0]), flush=True)
    for name in args.shapes.split(","):
        rec = dict(bench_shape(name, args.reps, args.warmup), **tag)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
