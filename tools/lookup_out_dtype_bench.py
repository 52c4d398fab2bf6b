"""The correlation lookup with a half-precision output (`ofb_corr_lookup_to`) and gradient (`ofb_corr_lookup_backward`,
`ofb_corr_lookup_coords_backward_from`) against the fp32 output and what autocast does with it today.  12 launches of
each variant (one RAFT forward's worth of lookups, each with its own coordinates and output gradient) timed with CUDA
events, all variants alternating in one process.

    python tools/lookup_out_dtype_bench.py [--reps 20] [--warmup 3] [--shapes c4,bench] [--out FILE]

Shapes: `c4` = B = 16, 47 x 156; `bench` = bench.py's micro-batch (8 pairs, 136 x 240); C = 256, 4 levels, radius 4, the
bf16 query-minor 8x4 pyramid of the tcgen05 builder.  Forward variants:
    fp32            the fp32 lookup (the reference's output)
    fp32_then_half  the fp32 lookup, then .half(): what torch.autocast does before BasicMotionEncoder.convc1
    fp16, bf16      the lookup writing its output in that dtype
Backward variants: the pyramid backward (into a dense fp32 gradient pyramid, as CorrBlock's) plus the coordinate
backward, with an fp32 d_out and with an fp16 d_out (the same values).  Per shape one JSON line gives, per variant, the
median / min / mean of the 12 launches (ms), the median per launch and the algorithmic HBM bytes per query with the rate
they reach and its share of 6565.5 GB/s (the HBM copy bandwidth measured on a B200, DESIGN.md section 4):
    forward         L (2r+2)^2 * 2 window + 8 coordinates + L (2r+1)^2 * esize output          fp32 2104 B, 16-bit 1456 B
    + .half()       reads the 1296 B fp32 output, writes 648 B                                          4048 B
    backward        pyramid backward: 8 coordinates + L (2r+1)^2 * esize d_out + L (2r+2)^2 * 4 gradient updates;
                    coordinate backward: L (2r+2)^2 * 2 window + L (2r+1)^2 * esize d_out + 8 + 8    fp32 5016 B, fp16 3720 B
It also checks that the timed half-precision outputs are the fp32 output cast (bit for bit) and that both backward
variants give the same d coords bits.  The first line names the GPU, its power limit and max SM clock, read in the same
run.  The pyramid (2.3 GB at c4, 22.6 GB at bench), the gradient pyramid and the 12 output gradients are larger than L2,
so every kernel streams from HBM."""
import argparse
import ctypes
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import ofb200  # noqa: E402
from model.utils import coords_grid  # noqa: E402
from ofb200.ops.corr import CorrBlock  # noqa: E402
from pyramid_dtype_bench import Window, gpu_info  # noqa: E402

SHAPES = {"c4": (16, 256, 47, 156), "bench": (8, 256, 136, 240)}
LEVELS, RADIUS, ITERS = 4, 4, 12
PEAK_GBS = 6565.5
CODE = {torch.float32: ofb200.DTYPE_F32, torch.float16: ofb200.DTYPE_F16, torch.bfloat16: ofb200.DTYPE_BF16}


def query_bytes():
    win = LEVELS * (2 * RADIUS + 2) ** 2 * 2
    chans = LEVELS * (2 * RADIUS + 1) ** 2
    upd = LEVELS * (2 * RADIUS + 2) ** 2 * 4
    bwd = {es: (8 + chans * es + upd) + (win + chans * es + 16) for es in (4, 2)}
    return {"fp32": win + 8 + 4 * chans, "fp32_then_half": win + 8 + 4 * chans + 4 * chans + 2 * chans,
            "fp16": win + 8 + 2 * chans, "bf16": win + 8 + 2 * chans, "bwd_fp32": bwd[4], "bwd_fp16": bwd[2]}


def stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}


def bench_shape(name, reps, warmup):
    b, c, h, w = SHAPES[name]
    q = b * h * w
    d = 2 * RADIUS + 1
    lib = ofb200.load()
    st = ofb200.stream_ptr()
    gen = torch.Generator(device="cuda").manual_seed(2026)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    coords = [coords_grid(b, h, w).cuda() + 4 * torch.randn((b, 2, h, w), device="cuda", generator=gen) for _ in range(ITERS)]
    g16 = [torch.randn((b, LEVELS * d * d, h, w), device="cuda", generator=gen).half() for _ in range(ITERS)]
    g32 = [g.float() for g in g16]
    blk = CorrBlock(f1, f2, num_levels=LEVELS, radius=RADIUS, pyramid_dtype=torch.bfloat16)
    assert blk.builder == "tcgen05" and blk._pyr.layout == ofb200.LAYOUT_QMINOR8X4
    outs = {dt: torch.empty((b, LEVELS * d * d, h, w), dtype=dt, device="cuda") for dt in CODE}
    d_coords = torch.empty((b, 2, h, w), device="cuda")
    # the dense fp32 gradient pyramid CorrBlock's backward accumulates into (tight rows)
    dpyr = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    ofb200.check(lib.ofb_pyramid_layout(h, w, LEVELS, 0, ctypes.byref(dpyr), ctypes.byref(elems)), "ofb_pyramid_layout")
    dpyr.dtype = ofb200.DTYPE_F32
    dbufs = [torch.zeros(q * int(elems[lvl]), device="cuda") for lvl in range(LEVELS)]
    for lvl, t in enumerate(dbufs):
        dpyr.base[lvl] = t.data_ptr()

    def lookup(k, dt):
        ofb200.check(lib.ofb_corr_lookup_to(ctypes.byref(blk._pyr), ofb200.ptr(coords[k]), ofb200.ptr(outs[dt]), CODE[dt],
                                            None, None, b, h, w, RADIUS, st), "ofb_corr_lookup_to")
        return outs[dt]

    def backward(k, g):
        g = g[k]
        ofb200.check(lib.ofb_corr_lookup_backward(ctypes.byref(dpyr), ofb200.ptr(coords[k]), ofb200.ptr(g), CODE[g.dtype],
                                                  b, h, w, RADIUS, st), "ofb_corr_lookup_backward")
        ofb200.check(lib.ofb_corr_lookup_coords_backward_from(ctypes.byref(blk._pyr), ofb200.ptr(coords[k]), ofb200.ptr(g),
                                                              CODE[g.dtype], ofb200.ptr(d_coords), b, h, w, RADIUS, st),
                     "ofb_corr_lookup_coords_backward_from")

    variants = {
        "fp32": lambda k: lookup(k, torch.float32),
        "fp32_then_half": lambda k: lookup(k, torch.float32).half(),
        "fp16": lambda k: lookup(k, torch.float16),
        "bf16": lambda k: lookup(k, torch.bfloat16),
        "bwd_fp32": lambda k: backward(k, g32),
        "bwd_fp16": lambda k: backward(k, g16),
    }
    times = {key: [] for key in variants}
    keys = list(variants)
    for r in range(warmup + reps):
        for key in (keys if r % 2 == 0 else reversed(keys)):             # alternate the order every repetition
            fn = variants[key]
            with Window() as win:
                for k in range(ITERS):
                    fn(k)
            torch.cuda.synchronize()
            if r >= warmup:
                times[key].append(win.ms())
    qb = query_bytes()
    rec = {"shape": name, "B": b, "C": c, "h": h, "w": w, "levels": LEVELS, "radius": RADIUS, "pyramid": "bf16",
           "layout": "qminor8x4", "launches": ITERS, "reps": reps}
    for key, v in times.items():
        per = statistics.median(v) / ITERS
        gbs = qb[key] * q / (per * 1e-3) / 1e9
        rec[key] = {"ms_12": stats(v), "ms_per_launch": round(per, 4), "bytes_per_query": qb[key], "GB_s": round(gbs, 1),
                    "frac_of_6565_GB_s": round(gbs / PEAK_GBS, 3)}
    med = {key: statistics.median(v) for key, v in times.items()}
    rec["fp16_over_fp32"] = round(med["fp16"] / med["fp32"], 3)
    rec["fp16_over_fp32_then_half"] = round(med["fp16"] / med["fp32_then_half"], 3)
    rec["bwd_fp16_over_bwd_fp32"] = round(med["bwd_fp16"] / med["bwd_fp32"], 3)
    # the timed kernels compute what they should: the half outputs are the fp32 output cast, both gradients agree
    ref = lookup(ITERS - 1, torch.float32).clone()
    rec["half_outputs_are_the_cast"] = all(
        torch.equal(lookup(ITERS - 1, dt).view(torch.int16), ref.to(dt).view(torch.int16)) for dt in (torch.float16, torch.bfloat16))
    backward(ITERS - 1, g32)
    dc32 = d_coords.clone()
    backward(ITERS - 1, g16)
    rec["d_coords_equal"] = bool(torch.equal(dc32.view(torch.int32), d_coords.view(torch.int32)))
    del blk, dbufs
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c4,bench")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lookup_out_dtype_bench.py needs a CUDA device (B200)")
    if args.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")
    ofb200.load()
    lines = [gpu_info()]
    print(json.dumps(lines[0]), flush=True)
    for name in args.shapes.split(","):
        rec = bench_shape(name, args.reps, args.warmup)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
