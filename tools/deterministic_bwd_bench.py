"""The deterministic backward kernels against the atomic ones they replace: the convex upsampling's backward (fp32 and
fp16 masks, d_flow and d_mask) and `upflow8`'s backward (bilinear resize, align_corners=True, 8x), each called through
the C ABI of this build and of a baseline libofb200.so (the build before the kernels became gathers) loaded in the same
process.  12 launches per window (one RAFT forward's worth, each with its own inputs) timed with CUDA events, the two
builds alternating.

    python tools/deterministic_bwd_bench.py --baseline PATH/libofb200.so [--reps 20] [--warmup 3] [--shapes c4,bench]
                                            [--out FILE]

Build the baseline from the commit before, e.g. `git worktree add /tmp/base <commit> && make -C
/tmp/base/torch-optical-flow_b200/csrc`, and pass its `ofb200/libofb200.so`.  Shapes (coarse grid): `c4` = B = 16,
47 x 156; `bench` = bench.py's micro-batch (8 pairs, 136 x 240).  Each window starts behind a ~20 ms spin kernel
(torch.cuda._sleep), so all 12 launches are queued before the first runs; `host_bound_reps` counts windows whose start
the GPU reached before the last launch was queued (expected 0).  The 12 input sets of every variant are larger than
L2.  Per shape one JSON line gives, per variant and build, the median / min / mean of the window (ms) and the ratio
new / baseline of the medians.  It also checks, on the timed inputs, that the new d_mask has the baseline's bits, that
d_flow and the upflow8 gradient are within 1e-5 (relative to the largest element) of the baseline's atomic sums, and that
two runs of the new kernels give the same bits.  A last line times `tools/microbench.py:bench_corr_train_c4` (CorrBlock
forward + backward at C4) with each build, in a subprocess each; the line before it, the cost of torch's NaN fill of
uninitialised memory under `torch.use_deterministic_algorithms(True)` on a CorrBlock's construction at the bench
shape.  The first line names the GPU, its power limit and max
SM clock, read in the same run."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import ofb200  # noqa: E402
from pyramid_dtype_bench import Window, gpu_info  # noqa: E402

SHAPES = {"c4": (16, 47, 156), "bench": (8, 136, 240)}
ITERS = 12
SLEEP_CYCLES = 40_000_000          # ~20 ms at 1965 MHz: longer than queueing 12 launches
MASKS = {"fp32": torch.float32, "fp16": torch.float16}
DT = {torch.float32: ofb200.DTYPE_F32, torch.float16: ofb200.DTYPE_F16}


def bind(path):
    lib = ctypes.CDLL(path)
    for name, (res, args) in ofb200.SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}


def bench_shape(name, libs, reps, warmup):
    b, h, w = SHAPES[name]
    gen = torch.Generator(device="cuda").manual_seed(2028)
    flows = [2 * torch.randn((b, 2, h, w), device="cuda", generator=gen) for _ in range(ITERS)]
    d_outs = [torch.randn((b, 2, 8 * h, 8 * w), device="cuda", generator=gen) for _ in range(ITERS)]
    masks = {k: [(2 * torch.randn((b, 576, h, w), device="cuda", generator=gen)).to(dt) for _ in range(ITERS)]
             for k, dt in MASKS.items()}
    d_flows = [torch.zeros_like(f) for f in flows]
    d_masks = {k: [torch.empty_like(m) for m in v] for k, v in masks.items()}
    st = ofb200.stream_ptr()

    def upsample(lib, key, k, d_flow=None, d_mask=None):
        d_flow = d_flows[k] if d_flow is None else d_flow
        d_mask = d_masks[key][k] if d_mask is None else d_mask
        m = masks[key][k]
        rc = lib.ofb_convex_upsample_backward(ofb200.ptr(flows[k]), ofb200.ptr(m), DT[m.dtype], ofb200.ptr(d_outs[k]),
                                              ofb200.ptr(d_flow), ofb200.ptr(d_mask), b, h, w, st)
        ofb200.check(rc, "ofb_convex_upsample_backward")

    def upflow8(lib, k, d_in=None):
        d_in = d_flows[k] if d_in is None else d_in
        rc = lib.ofb_resize_bilinear_backward_f32(ofb200.ptr(d_outs[k]), ofb200.ptr(d_in), b, 2, h, w, 8 * h, 8 * w, 1,
                                                  8.0, 8.0, st)
        ofb200.check(rc, "ofb_resize_bilinear_backward_f32")

    variants = {}
    for which, lib in libs.items():
        for key in MASKS:
            variants[f"upsample_{key}_{which}"] = (lambda lib, key: lambda k: upsample(lib, key, k))(lib, key)
        variants[f"upflow8_{which}"] = (lambda lib: lambda k: upflow8(lib, k))(lib)
    times = {key: [] for key in variants}
    host_bound = {key: 0 for key in variants}
    keys = list(variants)
    for r in range(warmup + reps):
        for key in (keys if r % 2 == 0 else reversed(keys)):
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
    rec = {"shape": name, "B": b, "h": h, "w": w, "launches": ITERS, "reps": reps}
    for key, v in times.items():
        rec[key] = {"ms_12": stats(v), "host_bound_reps": host_bound[key]}
    med = {key: statistics.median(v) for key, v in times.items()}
    for base in [f"upsample_{k}" for k in MASKS] + ["upflow8"]:
        rec[f"{base}_new_over_baseline"] = round(med[f"{base}_new"] / med[f"{base}_baseline"], 3)

    # results on the last timed input set: new against baseline, and new against itself
    k = ITERS - 1

    def rel(a, ref):
        return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))

    for key in MASKS:
        out = {}
        for which in ("new", "baseline", "new_again"):
            df, dm = torch.zeros_like(flows[k]), torch.empty_like(masks[key][k])
            upsample(libs["new" if which != "baseline" else "baseline"], key, k, df, dm)
            out[which] = (df, dm)
        iv = torch.int32 if masks[key][k].element_size() == 4 else torch.int16
        rec[f"upsample_{key}_d_mask_bits_equal_baseline"] = bool(torch.equal(out["new"][1].view(iv), out["baseline"][1].view(iv)))
        rec[f"upsample_{key}_d_flow_max_rel_diff_baseline"] = rel(out["new"][0], out["baseline"][0])
        rec[f"upsample_{key}_repeat_bits_equal"] = bool(torch.equal(out["new"][0].view(torch.int32), out["new_again"][0].view(torch.int32))
                                                     and torch.equal(out["new"][1].view(iv), out["new_again"][1].view(iv)))
    out = {}
    for which in ("new", "baseline", "new_again"):
        d = torch.zeros_like(flows[k])
        upflow8(libs["new" if which != "baseline" else "baseline"], k, d)
        out[which] = d
    rec["upflow8_max_rel_diff_baseline"] = rel(out["new"], out["baseline"])
    rec["upflow8_repeat_bits_equal"] = bool(torch.equal(out["new"].view(torch.int32), out["new_again"].view(torch.int32)))
    torch.cuda.synchronize()
    del flows, d_outs, masks, d_flows, d_masks
    torch.cuda.empty_cache()
    return rec


def nan_fill_cost(reps, warmup):
    """CorrBlock construction (bf16 pyramid) at bench.py's micro-batch, with torch's NaN fill of uninitialised memory
    (what `torch.use_deterministic_algorithms(True)` turns on) and without, alternating; the pyramids must be equal."""
    from model.corr import CorrBlock

    b, c, h, w = 8, 256, 136, 240
    gen = torch.Generator(device="cuda").manual_seed(2029)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    saved = (torch.are_deterministic_algorithms_enabled(), torch.utils.deterministic.fill_uninitialized_memory)
    times = {"plain": [], "nan_filled": []}
    pyrs = {}
    try:
        for r in range(warmup + reps):
            for key in (("plain", "nan_filled") if r % 2 == 0 else ("nan_filled", "plain")):
                torch.use_deterministic_algorithms(key == "nan_filled")
                torch.utils.deterministic.fill_uninitialized_memory = True
                torch.cuda.synchronize()
                with Window() as win:
                    blk = CorrBlock(f1, f2, num_levels=4, radius=4)
                torch.cuda.synchronize()
                if r >= warmup:
                    times[key].append(win.ms())
                if r == warmup + reps - 1:
                    pyrs[key] = [t.clone() for t in blk.corr_pyramid]
                del blk
    finally:
        torch.use_deterministic_algorithms(saved[0])
        torch.utils.deterministic.fill_uninitialized_memory = saved[1]
    med = {k: statistics.median(v) for k, v in times.items()}
    equal = all(torch.equal(a, b) for a, b in zip(pyrs["plain"], pyrs["nan_filled"]))
    return {"kernel": "CorrBlock(bf16) construction, 8 x 256 x 136 x 240, with / without the NaN fill (ms)",
            "plain": stats(times["plain"]), "nan_filled": stats(times["nan_filled"]),
            "added_ms": round(med["nan_filled"] - med["plain"], 4), "pyramids_equal": equal}


CORR_TRAIN = """
import json, sys
sys.path[:0] = [{pkg!r}, {tools!r}]
import ofb200
ofb200.LIB_PATH = {lib!r}
import microbench
print(json.dumps(microbench.bench_corr_train_c4()))
"""


def corr_train(paths):
    rec = {"kernel": "tools/microbench.py:bench_corr_train_c4, min of 3 reps (ms)"}
    for which, path in paths.items():
        code = CORR_TRAIN.format(pkg=os.path.join(ROOT, "torch-optical-flow_b200"), tools=os.path.join(ROOT, "tools"),
                                 lib=path)
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800)
        if res.returncode != 0:
            raise SystemExit(f"bench_corr_train_c4 with {path} failed:\n{res.stderr[-3000:]}")
        rec[which] = json.loads(res.stdout.strip().splitlines()[-1])
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--baseline", required=True, help="libofb200.so of the build before the deterministic kernels")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c4,bench")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_bwd_bench.py needs a CUDA device (B200)")
    if args.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")
    baseline = os.path.abspath(args.baseline)
    if os.path.realpath(baseline) == os.path.realpath(ofb200.LIB_PATH):
        raise SystemExit("--baseline is this build's own library")
    libs = {"new": ofb200.load(), "baseline": bind(baseline)}
    lines = [gpu_info()]
    print(json.dumps(lines[0]), flush=True)
    for name in args.shapes.split(","):
        lines.append(bench_shape(name, libs, args.reps, args.warmup))
        print(json.dumps(lines[-1]), flush=True)
    lines.append(nan_fill_cost(args.reps, args.warmup))
    print(json.dumps(lines[-1]), flush=True)
    lines.append(corr_train({"new": ofb200.LIB_PATH, "baseline": baseline}))
    print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
