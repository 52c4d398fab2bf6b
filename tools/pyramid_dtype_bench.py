"""bf16 against fp16 correlation pyramids: the tcgen05 builder (K2) and 12 lookups (K3, one RAFT forward's worth) timed
with CUDA events, the two dtypes alternating in one process so both see the same clocks and neighbours.

    python tools/pyramid_dtype_bench.py [--reps 20] [--warmup 3] [--shapes bench,c4] [--out FILE]

Shapes: `bench` = bench.py's micro-batch (8 pairs, C = 256, 136 x 240), `c4` = B = 16, C = 256, 47 x 156.  Per dtype and
shape it prints one JSON line with the median / min / mean of the operand prep, the builder and the 12 lookups over the
timed repetitions (ms), and the relative difference of the medians (fp16 / bf16 - 1).  The first line names the GPU and
its power limit (read-only `nvidia-smi --query-gpu`): the times belong to that card at that limit.  Both pyramids stay
resident (2 x 22.6 GB at the bench shape), far larger than L2, so every build and lookup streams from HBM."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
import torch  # noqa: E402

import ofb200  # noqa: E402
from model.utils import coords_grid  # noqa: E402
from ofb200.ops.corr import CorrBlock, build_pyramid, prepare_operands  # noqa: E402

SHAPES = {"bench": (8, 256, 136, 240), "c4": (16, 256, 47, 156)}
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
ITERS = 12


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = res.stdout.strip().splitlines()[0] if res.returncode == 0 and res.stdout.strip() else res.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


class Window:
    """CUDA events around one piece of work on the current stream."""

    def __init__(self):
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def __enter__(self):
        self.e0.record()
        return self

    def __exit__(self, *exc):
        self.e1.record()
        return False

    def ms(self):
        return self.e0.elapsed_time(self.e1)


def bench_shape(name, reps, warmup):
    b, c, h, w = SHAPES[name]
    gen = torch.Generator(device="cuda").manual_seed(2024)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    coords = [coords_grid(b, h, w).cuda() + 4 * torch.randn((b, 2, h, w), device="cuda", generator=gen) for _ in range(ITERS)]
    out = torch.empty((b, 4 * 81, h, w), device="cuda")
    state = {}
    for key, dt in DTYPES.items():
        blk = CorrBlock(f1, f2, num_levels=4, radius=4, pyramid_dtype=dt)
        assert blk.builder == "tcgen05"
        state[key] = (blk, prepare_operands(f1, f2, 4, dt))
    times = {key: {"prep": [], "build": [], "lookup12": []} for key in DTYPES}

    def one(key, keep):
        blk, ops = state[key]
        dt = DTYPES[key]
        with Window() as tp:
            prepare_operands(f1, f2, 4, dt)
        with Window() as tb:
            ofb200.check(build_pyramid(ops, blk._pyr, b, c, h, w, dt), "build_pyramid")
        with Window() as tl:
            for k in range(ITERS):
                blk._lookup(coords[k], out, None, None)
        torch.cuda.synchronize()
        if keep:
            times[key]["prep"].append(tp.ms())
            times[key]["build"].append(tb.ms())
            times[key]["lookup12"].append(tl.ms())

    for r in range(warmup + reps):
        order = list(DTYPES) if r % 2 == 0 else list(reversed(DTYPES))      # alternate which dtype runs first
        for key in order:
            one(key, r >= warmup)
    recs = []
    med = {}
    for key in DTYPES:
        rec = {"shape": name, "B": b, "C": c, "h": h, "w": w, "dtype": key, "reps": reps}
        for part, v in times[key].items():
            rec[part] = {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}
        med[key] = {part: statistics.median(v) for part, v in times[key].items()}
        recs.append(rec)
    recs.append({"shape": name, "fp16_vs_bf16": {part: round(med["fp16"][part] / med["bf16"][part] - 1.0, 4)
                                                 for part in med["bf16"]}})
    # both builders computed the same correlations: a sanity check that the timed kernels did real work
    a, bb = state["bf16"][0].corr_pyramid[0][:4096].float(), state["fp16"][0].corr_pyramid[0][:4096].float()
    recs[-1]["l0_rel_diff_bf16_fp16"] = float((a - bb).norm() / bb.norm())
    del state
    torch.cuda.empty_cache()
    return recs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="bench,c4")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pyramid_dtype_bench.py needs a CUDA device (B200)")
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
