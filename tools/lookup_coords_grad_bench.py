"""The correlation lookup's coordinate backward (`ofb_corr_lookup_coords_backward`) against the forward lookup
(`ofb_corr_lookup`) on the same pyramid: 12 launches of each (one RAFT forward's worth of lookups, each with its own
coordinates and output gradient) timed with CUDA events, forward and backward alternating in one process.

    python tools/lookup_coords_grad_bench.py [--reps 20] [--warmup 3] [--shapes c4,bench] [--out FILE]

Shapes: `c4` = B = 16, 47 x 156; `bench` = bench.py's micro-batch (8 pairs, 136 x 240); C = 256, 4 levels, radius 4.
Pyramids: the default bf16 query-minor 8x4 layout of the tcgen05 builder, and fp16.  Per shape and dtype one JSON line
gives the median / min / mean of the 12 launches (ms), the median per launch, backward / forward, and the algorithmic
HBM bytes per query of each kernel with the rate they reach and its share of 6565.5 GB/s (the HBM copy bandwidth
measured on a B200, DESIGN.md section 4):
    forward   L (2r+2)^2 esize window + 8 coordinates + 4 L (2r+1)^2 output          = 2104 B in bf16 / fp16
    backward  L (2r+2)^2 esize window + 4 L (2r+1)^2 d_out + 8 coordinates + 8 d coords = 2112 B
The first line names the GPU and its power limit, read in the same run.  The pyramids (2.3 GB per dtype at c4, 22.6 GB
at bench) and the 12 output gradients are larger than L2, so both kernels stream from HBM."""
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
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
LEVELS, RADIUS, ITERS = 4, 4, 12
PEAK_GBS = 6565.5


def query_bytes(esize):
    win = LEVELS * (2 * RADIUS + 2) ** 2 * esize
    chans = 4 * LEVELS * (2 * RADIUS + 1) ** 2
    return {"forward": win + 8 + chans, "backward": win + chans + 8 + 8}


def stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}


def bench_shape(name, reps, warmup):
    b, c, h, w = SHAPES[name]
    q = b * h * w
    d = 2 * RADIUS + 1
    lib = ofb200.load()
    gen = torch.Generator(device="cuda").manual_seed(2025)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    coords = [coords_grid(b, h, w).cuda() + 4 * torch.randn((b, 2, h, w), device="cuda", generator=gen) for _ in range(ITERS)]
    d_out = [torch.randn((b, LEVELS * d * d, h, w), device="cuda", generator=gen) for _ in range(ITERS)]
    out = torch.empty((b, LEVELS * d * d, h, w), device="cuda")
    d_coords = torch.empty((b, 2, h, w), device="cuda")
    blocks = {}
    for key, dt in DTYPES.items():
        blk = CorrBlock(f1, f2, num_levels=LEVELS, radius=RADIUS, pyramid_dtype=dt)
        assert blk.builder == "tcgen05" and blk._pyr.layout == ofb200.LAYOUT_QMINOR8X4
        blocks[key] = blk
    times = {key: {"forward": [], "backward": []} for key in DTYPES}

    def forward(blk):
        for k in range(ITERS):
            blk._lookup(coords[k], out, None, None)

    def backward(blk):
        for k in range(ITERS):
            ofb200.check(lib.ofb_corr_lookup_coords_backward(ctypes.byref(blk._pyr), ofb200.ptr(coords[k]),
                                                             ofb200.ptr(d_out[k]), ofb200.ptr(d_coords), b, h, w, RADIUS,
                                                             ofb200.stream_ptr()), "ofb_corr_lookup_coords_backward")

    for r in range(warmup + reps):
        for key in (DTYPES if r % 2 == 0 else reversed(list(DTYPES))):           # alternate the order every repetition
            parts = [("forward", forward), ("backward", backward)]
            for part, fn in (parts if r % 2 == 0 else reversed(parts)):
                with Window() as win:
                    fn(blocks[key])
                torch.cuda.synchronize()
                if r >= warmup:
                    times[key][part].append(win.ms())
    recs = []
    for key, dt in DTYPES.items():
        qb = query_bytes(torch.finfo(dt).bits // 8)
        rec = {"shape": name, "B": b, "C": c, "h": h, "w": w, "levels": LEVELS, "radius": RADIUS, "dtype": key,
               "layout": "qminor8x4", "launches": ITERS, "reps": reps}
        for part, v in times[key].items():
            per = statistics.median(v) / ITERS
            gbs = qb[part] * q / (per * 1e-3) / 1e9
            rec[part] = {"ms_12": stats(v), "ms_per_launch": round(per, 4), "bytes_per_query": qb[part],
                         "GB_s": round(gbs, 1), "frac_of_6565_GB_s": round(gbs / PEAK_GBS, 3)}
        rec["backward_over_forward"] = round(statistics.median(times[key]["backward"]) / statistics.median(times[key]["forward"]), 3)
        # the timed kernel does real work: its last gradient is finite and not all zero
        backward(blocks[key])
        rec["d_coords_finite_nonzero"] = bool(torch.isfinite(d_coords).all()) and bool((d_coords != 0).any())
        recs.append(rec)
    del blocks
    torch.cuda.empty_cache()
    return recs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c4,bench")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lookup_coords_grad_bench.py needs a CUDA device (B200)")
    if args.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")
    ofb200.load()
    lines = [gpu_info()]
    print(json.dumps(lines[0]), flush=True)
    for name in args.shapes.split(","):
        for rec in bench_shape(name, args.reps, args.warmup):
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
