"""The warp (`optical_flow.warp`, pixel-unit flow with the fused normalize) with fp32 inputs, with half-precision inputs
through the fp32 cast autocast runs (`frame.float()`, `flow.float()`, the fp32 warp, and in the backward the casts of
the gradients back), and with the half-precision frame and flow read directly.  12 launches of each variant (each
with its own frame, flow and output gradient) timed with CUDA events, all variants alternating in one process; then
one end-to-end arm: bench.py's host-staged pass with the half-precision producers' tensors, fp32 frame against fp16
frame, in the same call.

    python tools/warp_half_bench.py [--reps 20] [--warmup 3] [--shapes c2,bench,feature] [--e2e-steps 10]
                                    [--label TEXT] [--out FILE]

Shapes (B x C x H x W): `c2` = 2 x 3 x 436 x 1024 (Sintel), `bench` = 8 x 3 x 1088 x 1920 (bench.py's frame), `feature`
= 8 x 128 x 136 x 240 (a feature warp of a coarse-to-fine network).  Variants, forward (`fwd`) and forward + backward
(`fwdbwd`, torch.autograd.grad for the frame and the flow):
    fp32                      fp32 frame and flow (holding the fp16-rounded values, so every variant computes the same)
    fp16_via_fp32, bf16_via_fp32
                              half frame and flow, warp(frame.float(), flow.float()): two cast kernels before the fp32
                              warp, and in the backward the casts of d_frame and d_flow to the inputs' dtypes
    fp16, bf16                half frame and flow passed as they are
Per shape and pass one JSON line gives, per variant, the median / min / mean of the 12 launches (ms), the median per
launch and the algorithmic HBM bytes per pixel with the rate they reach and its share of 6565.5 GB/s (the HBM copy
bandwidth measured on a B200, DESIGN.md section 4); e_i, e_v = element sizes of the frame and the flow:
    forward            C e_i frame + 2 e_v flow + 4C output
    backward           4C zero-fill + C e_i frame + 2 e_v flow + 4C d_out + 8C d_frame read-modify-write + 2 e_v d_flow,
                       plus the d_frame cast 4C + C e_i when the frame is 16-bit
    each fp32 cast     (2 + 4) per element: C for the frame, 2 for the flow (forward); d_frame, d_flow (backward)
Each window starts behind a ~20 ms spin kernel (torch.cuda._sleep), so all 12 launches are queued before the first
runs; `host_bound_reps` counts windows whose start the GPU reached before the last launch was queued (expected 0).
The run checks that the last timed outputs are bit-identical: fp16, fp16_via_fp32 and fp32 (which holds the same
values), bf16 and bf16_via_fp32; d_flow bit for bit and d_frame within one ulp of the dtype (its atomics add in a
varying order) between each half variant and its cast path.  Every line names the GPU, its power limit and max SM
clock, read in the same run.  The 12 inputs of a variant (>= 200 MB at c2 in fp32) exceed L2, so every launch streams from HBM.

The end-to-end line runs HostStagedRunner over pinned PairArena inputs as bench.py's `e2e_half_precision_producers`
arm does (8 pairs per step, fmap1 / fmap2 bf16, up_mask fp16), once with an fp32 frame and once with an fp16 frame,
alternating, and reports pairs/s (median over repetitions) and the host->device bytes per step of each."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import ofb200  # noqa: E402
from optical_flow import warp  # noqa: E402
from pyramid_dtype_bench import Window, gpu_info  # noqa: E402

SHAPES = {"c2": (2, 3, 436, 1024), "bench": (8, 3, 1088, 1920), "feature": (8, 128, 136, 240)}
ITERS = 12
PEAK_GBS = 6565.5
SLEEP_CYCLES = 40_000_000          # ~20 ms at 1965 MHz: longer than queueing 12 launches of any variant
HALF = {"fp16": torch.float16, "bf16": torch.bfloat16}
KEYS = ["fp32", "fp16_via_fp32", "fp16", "bf16_via_fp32", "bf16"]


def px_bytes(c, key, backward):
    """Algorithmic HBM bytes per output pixel (module docstring)."""
    ei = ev = 4 if key in ("fp32",) or key.endswith("via_fp32") else 2
    cast = key.endswith("via_fp32")
    fwd = c * ei + 2 * ev + 4 * c
    fwd += (c + 2) * 6 if cast else 0
    if not backward:
        return fwd
    bwd = 4 * c + c * ei + 2 * ev + 4 * c + 8 * c + 2 * ev
    if key in HALF:
        bwd += 4 * c + 2 * c                         # the d_frame cast after the kernel
    if cast:
        bwd += (c + 2) * 6                           # autograd's casts of d_frame and d_flow
    return fwd + bwd


def stats(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "mean": round(statistics.fmean(v), 4)}


def bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def same_bits(a, b):
    return bool(a.dtype == b.dtype and torch.equal(bits(a), bits(b)))


def bench_shape(name, reps, warmup):
    b, c, h, w = SHAPES[name]
    px = b * h * w
    gen = torch.Generator(device="cuda").manual_seed(2028)
    frames, flows, grads = [], [], []
    for _ in range(ITERS):
        frames.append(torch.rand((b, c, h, w), device="cuda", generator=gen).half().float())
        coarse = 8 * torch.randn((b, 2, h // 8, w // 8), device="cuda", generator=gen)      # pixel units, smooth
        flows.append(torch.nn.functional.interpolate(coarse, size=(h, w), mode="bilinear").half().float())
        grads.append(torch.randn((b, c, h, w), device="cuda", generator=gen))
    inputs = {"fp32": (frames, flows)}
    for key, dt in HALF.items():
        inputs[key] = ([f.to(dt) for f in frames], [f.to(dt) for f in flows])
    for key in list(inputs):
        for t in inputs[key][0] + inputs[key][1]:
            t.requires_grad_(True)

    def fn(key, backward):
        src = "fp32" if key == "fp32" else key.split("_")[0]
        cast = key.endswith("via_fp32")

        def run(k):
            fr, fl = inputs[src][0][k], inputs[src][1][k]
            if not backward:
                with torch.no_grad():
                    return warp(fr.float() if cast else fr, fl.float() if cast else fl, pixel_flow=True)
            out = warp(fr.float() if cast else fr, fl.float() if cast else fl, pixel_flow=True)
            return (out,) + torch.autograd.grad(out, (fr, fl), grad_outputs=grads[k])
        return run

    recs = []
    for backward in (False, True):
        times = {key: [] for key in KEYS}
        host_bound = {key: 0 for key in KEYS}
        last = {}
        for r in range(warmup + reps):
            for key in (KEYS if r % 2 == 0 else list(reversed(KEYS))):            # alternate the order every repetition
                run = fn(key, backward)
                torch.cuda._sleep(SLEEP_CYCLES)
                with Window() as win:
                    for k in range(ITERS):
                        res = run(k)
                reached = win.e0.query()
                torch.cuda.synchronize()
                if r >= warmup:
                    times[key].append(win.ms())
                    host_bound[key] += int(reached)
                last[key] = res
                del res
        rec = {"shape": name, "B": b, "C": c, "H": h, "W": w, "pass": "fwdbwd" if backward else "fwd",
               "launches": ITERS, "reps": reps}
        for key, v in times.items():
            per = statistics.median(v) / ITERS
            pb = px_bytes(c, key, backward)
            gbs = pb * px / (per * 1e-3) / 1e9
            rec[key] = {"ms_12": stats(v), "ms_per_launch": round(per, 4), "bytes_per_px": pb, "GB_s": round(gbs, 1),
                        "frac_of_6565_GB_s": round(gbs / PEAK_GBS, 3), "host_bound_reps": host_bound[key]}
        med = {key: statistics.median(v) for key, v in times.items()}
        for key in HALF:
            rec[f"{key}_over_{key}_via_fp32"] = round(med[key] / med[f"{key}_via_fp32"], 3)
            rec[f"{key}_over_fp32"] = round(med[key] / med["fp32"], 3)
        # the last timed launch of every variant: the same output bits; d_flow bits between the half variants and
        # their cast paths; d_frame within one ulp of the dtype (atomics)
        out = lambda key: last[key][0] if backward else last[key]       # noqa: E731
        rec["out_bits_equal"] = (same_bits(out("fp16"), out("fp32")) and same_bits(out("fp16_via_fp32"), out("fp32"))
                                 and same_bits(out("bf16"), out("bf16_via_fp32")))
        if backward:
            for key, dt in HALF.items():
                d, v = last[key][1:], last[f"{key}_via_fp32"][1:]
                rec[f"{key}_d_flow_bits_equal"] = same_bits(d[1], v[1])
                diff = (d[0].float() - v[0].float()).abs()
                spacing = torch.where(v[0].float() == 0, torch.ones_like(diff), v[0].float().abs()) * (
                    2.0 ** -10 if dt == torch.float16 else 2.0 ** -7)
                rec[f"{key}_d_frame_within_1ulp"] = bool((diff <= spacing).all())
        recs.append(rec)
        del last
    del inputs, frames, flows, grads
    torch.cuda.empty_cache()
    return recs


def bench_e2e(reps, steps):
    """bench.py's host-staged arm with the half-precision producers' tensors, fp32 frame against fp16 frame."""
    import bench
    from ofb200.runner import HostStagedRunner, PairArena
    from ofb200.ops.epe import AverageEndPointError

    device = torch.device("cuda", 0)
    pairs = 8
    batch = bench.make_batch(pairs, device, 1234, torch)
    producers = {"fmap1": torch.bfloat16, "fmap2": torch.bfloat16, "up_mask": torch.float16}
    arms = {"frame_fp32": dict(producers), "frame_fp16": dict(producers, frame=torch.float16)}
    hosts = {k: PairArena(pairs, PairArena.shapes_of(batch), pin=True, dtypes=d).fill(batch) for k, d in arms.items()}
    runners = {k: HostStagedRunner(device, 1) for k in arms}
    rates = {k: [] for k in arms}
    h2d = {}
    for r in range(2 + reps):
        for key in (list(arms) if r % 2 == 0 else list(reversed(list(arms)))):
            runner, host, m = runners[key], hosts[key], AverageEndPointError()
            runner.h2d_bytes = 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(steps):
                runner.run(host, m, prefetch=host if i + 1 < steps else None)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            if r >= 2:
                rates[key].append(pairs * steps / (ms * 1e-3))
                h2d[key] = runner.h2d_bytes // steps
    rec = {"shape": "e2e", "pairs_per_step": pairs, "steps": steps, "reps": reps, "micro_batch": 1,
           "producer_dtypes": "fmap1, fmap2: bf16; up_mask: fp16; coords, flow_lo, target, valid: fp32"}
    for key in arms:
        rec[key] = {"pairs_s": stats(rates[key]), "h2d_bytes_per_step": h2d[key],
                    "payload_bytes_per_pair": hosts[key].payload_bytes_per_pair}
    rec["frame_fp16_over_frame_fp32"] = round(statistics.median(rates["frame_fp16"]) /
                                              statistics.median(rates["frame_fp32"]), 3)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c2,bench,feature")
    ap.add_argument("--e2e-steps", type=int, default=10, help="steps per end-to-end repetition (0: skip the arm)")
    ap.add_argument("--label", default=None, help="added to every JSON line as \"label\" (e.g. the build measured)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("warp_half_bench.py needs a CUDA device (B200)")
    if args.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")
    ofb200.load()
    tag = dict(gpu_info(), **({"label": args.label} if args.label else {}))
    lines = []
    for name in args.shapes.split(","):
        for rec in bench_shape(name, args.reps, args.warmup):
            lines.append(dict(rec, **tag))
            print(json.dumps(lines[-1]), flush=True)
    if args.e2e_steps > 0:
        lines.append(dict(bench_e2e(args.reps, args.e2e_steps), **tag))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
