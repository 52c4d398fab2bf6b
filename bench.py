#!/usr/bin/env python
"""bench.py -- image-pairs/s of the hot path (corr + lookup, warp, EPE) on N B200s, one JSON line.

Workload (BASELINE.json configs[4], "C5"): 1088x1920 image pairs, 256-channel feature maps at 1/8
resolution (136x240), 4-level correlation pyramid, radius-4 lookup over 12 refinement iterations,
convex 8x upsampling, backward warp + validity mask of the 3x1088x1920 frame, masked EPE, and the
(sum, count) all-reduce over ranks.  Every rank processes `--pairs` pairs per step (8 by default, so
8 GPUs = the config's batch of 64): weak scaling, no data-path collective.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference ...                            # the CPU path on the host cores
    python bench.py --dump-outputs DIR ...                          # also write the last timed step's outputs

`--dump-outputs DIR` (rank 0): after the timed steps, DIR/<name>.npy holds what the last timed step of the
           device-resident arm computed -- `corr` (the last lookup), `flow_up`, `warped`, `mask` as float32
           (pairs, n) arrays, and `epe_state`, the float64 (sum, count) the step returned (the EPE metric
           accumulated over the timed steps).  Row p of output i (in that order) holds pair p's values at the
           flat C-order positions np.sort(np.random.default_rng(i).choice(size, n, replace=False)) of its
           per-pair array, n = 60e6 // (16 * pairs), or at every position when size <= n: under 64 MB in all.
           The inputs are seeded, so two builds run with the same arguments can be compared output for output.
           The last micro-batch is sampled after the timed window; with several micro-batches per step the
           others are sampled inside it (the next one overwrites the shared lookup buffer), which adds a gather
           of at most 60 MB to the timed time.

`value`  : pairs/s with inputs resident in HBM (CUDA events, barrier + synchronize on both sides,
           max over ranks).
`e2e`    : pairs/s through ofb200.runner.HostStagedRunner with PINNED HOST inputs: host->device
           copies of every input and the device->host read of the EPE state are inside the timed
           region.
`roofline`: the dominant kernel (K2, the tcgen05 correlation-pyramid builder) against the measured
           peaks of MEASURED_PEAKS.json; `kernels` lists every kernel class of the pass the same way
           and the named single-kernel configs (C2 warp, C3 corr, C4 lookup / upsample).
`cpu_baseline`: the reference's op sequence on a bounded sample of the same workload, timed on this box's
           host cores (rank 0, N=1 only) through both CPU restatements under oracle/ -- the C + OpenMP + numpy
           BLAS oracle and the ATen-op port (the ops the reference itself calls); the faster one is reported.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "torch-optical-flow_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "image-pairs/sec (corr+lookup, warp)"
UNIT = "pairs/s"
H, W, C, ITERS, RADIUS, LEVELS = 1088, 1920, 256, 12, 4, 4
h8, w8 = H // 8, W // 8
WORKLOAD = "c5_1080p_pipeline: fmaps 256x136x240, 4-level bf16 pyramid, r=4 lookup x12, convex upsample, warp 3x1088x1920 + mask, EPE"

PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
try:
    PEAKS.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
    PEAKS["source"] = "measured"
except Exception:
    pass


# ------------------------------------------------------------------------------ algorithmic work
def pyramid_elems(h, w, levels=LEVELS):
    return sum((h >> lv) * (w >> lv) for lv in range(levels))


def algorithmic(pairs):
    """Algorithmic bytes / flops per pass over `pairs` pairs (DESIGN.md section 4), per kernel class."""
    n = h8 * w8
    d2 = (2 * RADIUS + 1) ** 2
    return {
        # K2: bf16 operands read + bf16 pyramid written (both runs: levels 0-1, levels 2-3)
        "corr_pyramid_kernel": {"launches": 2, "flops": 2.0 * pairs * n * n * C,
                                "bytes": pairs * (2 * n * C * 2 + n * pyramid_elems(h8, w8) * 2)},
        # prep: fmap1 and fmap2 read in fp32 (fmap2 twice), K-major bf16 operands written
        "corr_prep": {"launches": 3, "bytes": pairs * n * C * (3 * 4 + 2 * 2 + 2 / 16)},
        "lookup": {"launches": ITERS,
                   "bytes": ITERS * pairs * n * (LEVELS * (2 * RADIUS + 2) ** 2 * 2 + 8 + LEVELS * d2 * 4)},
        "convex_upsample": {"launches": 1, "bytes": pairs * n * 4 * (576 + 2 + 128)},
        "warp": {"launches": 1, "bytes": pairs * H * W * (4 * (3 + 2 + 3) + 1)},        # normalize fused
        "epe": {"launches": 1, "bytes": pairs * H * W * 20},
    }


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self, t0, t1):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, f[2:]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------ synthetic inputs
def make_batch(pairs, device, seed, torch):
    g = torch.Generator(device=device).manual_seed(seed)
    from model.utils import coords_grid

    def rn(*s):
        return torch.randn(s, device=device, generator=g)

    base = coords_grid(pairs, h8, w8).to(device)
    batch = {
        "fmap1": rn(pairs, C, h8, w8), "fmap2": rn(pairs, C, h8, w8),
        "coords": (base[None] + 4 * rn(ITERS, pairs, 2, h8, w8)).contiguous(),
        "flow_lo": 1.5 * rn(pairs, 2, h8, w8),
        "up_mask": rn(pairs, 576, h8, w8),
        "frame": torch.rand((pairs, 3, H, W), device=device, generator=g),
        "target": 12 * rn(pairs, 2, H, W),
        "valid": (torch.rand((pairs, H, W), device=device, generator=g) > 0.1).float(),
    }
    batch["coords"][0] = base          # iteration 0 of RAFT looks up exact integer coordinates
    return batch


# ------------------------------------------------------------------------------ --dump-outputs
# per-pair shape of every array hot_path() returns
DUMP_SHAPES = {"corr": (LEVELS * (2 * RADIUS + 1) ** 2, h8, w8), "flow_up": (2, H, W), "warped": (3, H, W), "mask": (H, W)}
DUMP_BYTES = 60_000_000


class OutputSampler:
    """Fixed, seeded positions of hot_path()'s outputs, the same in every pair.  `take` gathers them on the device as
    soon as a micro-batch is done (the next one overwrites the shared lookup buffer); `write` saves the float32
    (pairs, n) arrays once the timed window has closed."""

    def __init__(self, pairs, device, torch):
        import numpy as np

        per_output = DUMP_BYTES // (len(DUMP_SHAPES) * 4 * pairs)
        self.index, self.parts = {}, []
        for seed, (name, shape) in enumerate(DUMP_SHAPES.items()):
            n = int(np.prod(shape))
            pick = np.arange(n) if n <= per_output else np.sort(np.random.default_rng(seed).choice(n, per_output, replace=False))
            self.index[name] = torch.from_numpy(pick).to(device)

    def take(self, out):
        self.parts.append({k: out[k].reshape(out[k].shape[0], -1)[:, i] for k, i in self.index.items()})

    def write(self, path, epe_state):
        import numpy as np

        os.makedirs(path, exist_ok=True)
        for k in self.index:
            arr = np.concatenate([p[k].float().cpu().numpy() for p in self.parts])
            np.save(os.path.join(path, k + ".npy"), arr)
        np.save(os.path.join(path, "epe_state.npy"), epe_state.double().cpu().numpy())


# ------------------------------------------------------------------------------ CPU path (oracle port)
def cpu_pass(sample):
    """The reference's op sequence for one pass, on the host, through the oracle port."""
    import oracle

    pyr = oracle.corr_pyramid(sample["fmap1"], sample["fmap2"], LEVELS)
    for it in range(sample["coords"].shape[0]):
        oracle.corr_lookup(pyr, sample["coords"][it], RADIUS)
    flow_up = oracle.upsample_flow(sample["flow_lo"], sample["up_mask"])
    oracle.warp(sample["frame"], oracle.normalize(flow_up), return_mask=True)
    return oracle.epe_sum_count(flow_up, sample["target"], sample["valid"])


def cpu_pass_torch(sample):
    """The same pass through oracle/torch_port.py: the ATen CPU ops the reference itself calls."""
    import torch

    from oracle import torch_port as tp

    t = {k: torch.from_numpy(v) for k, v in sample.items()}
    with torch.no_grad():
        pyr = tp.corr_pyramid(t["fmap1"], t["fmap2"], LEVELS)
        for it in range(t["coords"].shape[0]):
            tp.corr_lookup(pyr, t["coords"][it], RADIUS)
        flow_up = tp.upsample_flow(t["flow_lo"], t["up_mask"])
        tp.warp(t["frame"], tp.normalize(flow_up))
        return tp.epe_sum_count(flow_up, t["target"], t["valid"])


def cpu_sample(pairs, seed=99):
    import numpy as np

    r = np.random.default_rng(seed)
    ys, xs = np.meshgrid(np.arange(h8), np.arange(w8), indexing="ij")
    base = np.stack([xs, ys], 0).astype(np.float32)[None]

    def rn(*s):
        return r.standard_normal(s, dtype=np.float32)

    return {
        "fmap1": rn(pairs, C, h8, w8), "fmap2": rn(pairs, C, h8, w8),
        "coords": (base[None] + 4 * rn(ITERS, pairs, 2, h8, w8)).astype(np.float32),
        "flow_lo": 1.5 * rn(pairs, 2, h8, w8), "up_mask": rn(pairs, 576, h8, w8),
        "frame": r.random((pairs, 3, H, W), dtype=np.float32), "target": 12 * rn(pairs, 2, H, W),
        "valid": (r.random((pairs, H, W)) > 0.1).astype(np.float32),
    }


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def time_cpu(steps, warmup, pairs=1):
    """Both CPU restatements of the reference on one bounded sample; the faster one is the baseline."""
    import torch

    torch.set_num_threads(host_cores())
    sample = cpu_sample(pairs)
    rates = {}
    for name, fn in (("c_openmp_numpy", cpu_pass), ("torch_aten", cpu_pass_torch)):
        for _ in range(warmup):
            fn(sample)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn(sample)
        rates[name] = pairs * steps / (time.perf_counter() - t0)
    best = max(rates, key=rates.get)
    return {"value": rates[best], "unit": UNIT, "cores": host_cores(), "kind": "port",
            "sample": f"{pairs} pair(s) per step of the same 1080p pass (fp32 volume), {steps} timed step(s) after "
                      f"{warmup} warm-up, all host cores; two restatements of the reference timed, the faster reported: "
                      + ", ".join(f"{k} {v:.3f} pairs/s" for k, v in rates.items()),
            "ports": {k: round(v, 4) for k, v in rates.items()},
            "s_per_pair": 1.0 / rates[best]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core (numpy / the
    # oracle library are imported after this point, so the setting takes effect)
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(host_cores())
    steps, warm = args.steps, max(1, min(args.warmup, 1))
    cb = time_cpu(steps, warm, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": cb["s_per_pair"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "pairs_per_step": 1, "iters": ITERS, "radius": RADIUS, "levels": LEVELS},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "ports")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ single-kernel configs
def named_kernel_table(torch):
    """C2 warp, C3 corr pyramid, C4 lookup x12 + convex upsample at their BASELINE.json shapes."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import microbench

    recs = []
    # C2 / C3 / C4 forward kernels, then the training-path numbers (VERDICT r1 item 8: a driver line with clocks has to
    # carry them): the long-K backward GEMM alone at the C4 and C5 level-0 shapes, and one CorrBlock train step at KITTI size
    def backward_gemm():
        return microbench.bench_gemm_nt(shapes=((16, 7332, 256, 7332), (8, 32640, 256, 32640)))

    def corr_train_step():
        return microbench.bench_corr_train_c4(b=4)

    for fn in (microbench.bench_warp_c2, microbench.bench_corr_c3, microbench.bench_lookup_c4, backward_gemm, corr_train_step):
        try:
            recs.extend(fn())
        except Exception as e:  # a side table must never take the headline down
            recs.append({"kernel": fn.__name__, "error": repr(e)[:200]})
        torch.cuda.empty_cache()
    return recs


def bind_to_gpu_numa_node(torch, local):
    """Pin this rank to the CPUs next to its GPU (sysfs local_cpulist) BEFORE the pinned host buffers are
    allocated, so first-touch places them on the GPU's NUMA node: with 8 ranks staging 1.5 GB per step each,
    cross-socket pinned memory is what limits the host->device copies."""
    try:
        pr = torch.cuda.get_device_properties(local)
        path = f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"numa-local ({len(cpus)} cpus)"
    except Exception as e:  # topology not exposed: keep the default placement
        return f"default ({type(e).__name__})"
    return "default"


# ------------------------------------------------------------------------------ main arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    import ofb200
    from ofb200.runner import FIELDS, HostStagedRunner, KernelTimers, PairArena, hot_path
    from optical_flow.metrics.epe import AverageEndPointError

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU fallback (use --impl reference for the CPU arm)")
    ofb200.load()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    placement = {"chosen": "default"}
    dev_index = local
    if world > 1:
        # gloo for the CPU-side coordination of the placement probe, NCCL for everything on the device
        import datetime

        dist.init_process_group("cpu:gloo,cuda:nccl", timeout=datetime.timedelta(seconds=300))
        if not args.no_placement:
            from ofb200.runner import choose_device_set

            dev_index, placement = choose_device_set(rank, world, local)
    torch.cuda.set_device(dev_index)
    device = torch.device("cuda", dev_index)
    affinity = bind_to_gpu_numa_node(torch, dev_index) if world > 1 else "default"
    if world != args.gpus and rank == 0:
        sys.stderr.write(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}\n")
    sync_flag = torch.zeros(1, device=device)

    def barrier():
        if world > 1:
            dist.all_reduce(sync_flag)                 # a device collective (NCCL): every rank's stream has reached this point
        torch.cuda.synchronize()

    pairs, micro = args.pairs, min(args.micro, args.pairs)
    chunks = [(lo, min(lo + micro, pairs)) for lo in range(0, pairs, micro)]
    batch = make_batch(pairs, device, 1234 + rank, torch)
    views = [{k: (batch[k][:, lo:hi] if k == "coords" else batch[k][lo:hi]) for k in FIELDS} for lo, hi in chunks]
    views = [{k: v.contiguous() for k, v in d.items()} for d in views]
    lookup_out = torch.empty((micro, LEVELS * (2 * RADIUS + 1) ** 2, h8, w8), device=device)
    metric = AverageEndPointError()

    def step(timers=None, sampler=None):
        """One pass over every micro-batch.  With `sampler`, each micro-batch but the last is sampled before the next
        one overwrites the shared lookup buffer; the last one's outputs are returned, to be sampled by the caller."""
        out = None
        for v in views:
            if sampler is not None and out is not None:
                sampler.take(out)
            lo = lookup_out if v["fmap1"].shape[0] == micro else None
            out = hot_path(v, metric, timers=timers, lookup_out=lo, cta_group=args.cta_group)
        # (sum, count) all-reduce of a copy: the only collective
        return metric.sync(), (out if sampler is not None else None)

    # ---- device-resident arm
    for _ in range(args.warmup):
        step()
    metric.reset()
    dump = OutputSampler(pairs, device, torch) if args.dump_outputs and rank == 0 else None
    sampler = ClockSampler(dev_index)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    timers = KernelTimers()
    barrier()
    l0 = ofb200.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        state, last = step(timers, dump if i == args.steps - 1 else None)
    e1.record()
    if dump is not None:
        dump.take(last)                                # after e1: the last micro-batch's sample is not timed
    barrier()
    t_wall1 = time.time()
    if dump is not None:
        dump.write(args.dump_outputs, state)
        del dump
    launches = ofb200.launch_count() - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    epe_dev = float(metric.compute())
    ksum = timers.summary()
    value = world * pairs * args.steps / (ms * 1e-3)

    # ---- end-to-end arm: pinned host inputs, copies inside the timed region
    # the producer writes each pair's inputs into a pinned pair-major arena (ofb200.runner.PairArena): the runner
    # then moves one micro-batch -- all eight input tensors -- with a single host->device DMA
    def time_e2e(dtypes):
        host = PairArena(pairs, PairArena.shapes_of(batch), pin=True, dtypes=dtypes).fill(batch)
        runner = HostStagedRunner(device, min(args.e2e_micro, pairs))
        m2 = AverageEndPointError()
        steps = max(1, min(args.steps, args.e2e_steps))
        for _ in range(2):
            runner.run(host, m2)
        m2.reset()
        runner.h2d_bytes = runner.d2h_bytes = 0
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            # every step copies its own inputs; the next step's first pair is already in flight while this step's last
            # pair computes and its metric is read back
            epe = runner.run(host, m2, prefetch=host if i + 1 < steps else None)
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ms_ = max(e0.elapsed_time(e1), wall_ms)        # host-side staging is part of the cost: take the slower clock
        if world > 1:
            t = torch.tensor([ms_], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_ = float(t.item())
        res = {"value": round(world * pairs * steps / (ms_ * 1e-3), 2), "unit": UNIT, "steps": steps,
               "h2d_bytes_per_step": runner.h2d_bytes // steps, "d2h_bytes_per_step": runner.d2h_bytes // steps,
               "ms_per_step": round(ms_ / steps, 3), "micro_batch": runner.micro, "epe": epe}
        del host, runner
        return res

    # headline: the feature maps travel in bf16, the precision the reference's shipped configs produce them in
    # (`precision: 16`, methods/raft/config/train/default.yaml:20); everything else fp32.  The correlation operands
    # are bf16 either way (1/sqrt(256) is a power of two), so the pyramid is bit-identical to the fp32-input pass.
    half = {"fmap1": torch.bfloat16, "fmap2": torch.bfloat16}
    e2e = time_e2e(half)
    e2e["input_dtypes"] = "fmap1, fmap2: bf16 (read directly by ofb_corr_prep_from); coords, flow_lo, up_mask, frame, target, valid: fp32"
    e2e_fp32 = time_e2e(None)
    e2e_fp32["input_dtypes"] = "all fp32 (round-1 configuration)"
    epe_e2e = e2e.pop("epe")
    e2e_fp32.pop("epe")
    # informational: every tensor a `precision: 16` network produces in half precision travels that way -- the two
    # feature maps (bf16) AND the 576-channel upsampling mask (fp16: the mask head's autocast output; 46 % of a pair's
    # payload), read directly by ofb_convex_upsample.  Not the headline: the mask's rounding changes the upsampled flow
    # at the 1e-3 level, so this is a different input, reported separately.
    e2e_half = time_e2e(dict(half, up_mask=torch.float16))
    e2e_half["input_dtypes"] = "fmap1, fmap2: bf16; up_mask: fp16; coords, flow_lo, frame, target, valid: fp32"
    e2e_half.pop("epe")
    if rank == 0:
        sampler.stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines
    alg = algorithmic(micro)
    kernels = []
    for name, k in ksum.items():
        a = alg[name]
        groups = k["launches"] / a["launches"]            # passes timed
        ms_pass = k["ms_total"] / groups
        rec = {"kernel": name, "launches_per_pass": a["launches"], "ms_per_pass": round(ms_pass, 4),
               "share_of_step": round(k["ms_total"] / ms, 4),
               "gbs": round(a["bytes"] / ms_pass / 1e6, 1),
               "hbm_frac": round(a["bytes"] / ms_pass / 1e6 / PEAKS["hbm_gbs"], 4)}
        if "flops" in a:
            rec["tflops"] = round(a["flops"] / ms_pass / 1e9, 1)
            rec["tensor_frac_sustained"] = round(rec["tflops"] / PEAKS["bf16_tflops_sustained"], 4)
        kernels.append(rec)
    k2 = next(r for r in kernels if r["kernel"] == "corr_pyramid_kernel")
    roofline = {
        "kernel": "corr_pyramid_kernel (K2, tcgen05): the levels 0-1 run and the levels 2-3 run of one pyramid build",
        "bound": "hbm", "achieved": k2["gbs"], "peak": PEAKS["hbm_gbs"], "unit": "GB/s",
        "frac": k2["hbm_frac"], "traffic": None,
        "peak_source": PEAKS["source"] + " (MEASURED_PEAKS.json hbm_gbs)" if PEAKS["source"] == "measured" else "fallback",
        "tensor": {"achieved": k2["tflops"], "peak": PEAKS["bf16_tflops_sustained"], "unit": "TFLOP/s",
                   "frac": k2["tensor_frac_sustained"]},
        "note": "K=256 makes the builder write-bound on paper: 2*N^2*C flops need 0.39 ms/pair of tensor time, the bf16 "
                "pyramid write 0.44 ms/pair of HBM time; measured limit in steady state is the 1 kW power cap "
                "(992 W, 1.42 GHz when run back to back: profiles/r02_k2_power1.jsonl, DESIGN.md section 4)",
    }
    # dram__bytes_read + dram__bytes_write of both K2 launches at this shape come from ONE `ncu --set full` capture
    # committed under profiles/ (a profiler cannot run inside a timed region): a static figure, labelled as such
    traffic_file = os.path.join(ROOT, "profiles", "k2_traffic.json")
    if os.path.exists(traffic_file):
        try:
            tj = json.load(open(traffic_file))
            roofline["traffic"] = tj.get("dram_bytes_per_launch_at_bench_shape")
            roofline["traffic_source"] = "static: " + tj.get("source", "profiles/k2_traffic.json") + " -- not measured in this run"
            roofline["algorithmic_bytes"] = tj.get("algorithmic_bytes")
        except Exception:
            pass

    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "dtype_detail": "correlation: bf16 x bf16 -> f32 accumulate, bf16 stored; lookup / warp / upsample / EPE: f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "pairs_per_gpu_per_step": pairs, "global_pairs_per_step": pairs * world,
                   "micro_batch": micro, "iters": ITERS, "radius": RADIUS, "levels": LEVELS,
                   "l2": "inputs larger than L2 (pyramid 2.83 GB/pair, 196 MB of inputs per pair)",
                   "parallelism": f"batch-sharded x{world}, NCCL all-reduce of (sum_epe, count) only",
                   "host_affinity": affinity, "device_placement": placement},
        "e2e": dict(e2e, api="ofb200.runner.HostStagedRunner.run(pinned PairArena: one DMA per pair) -> CorrBlock / warp / upsample_flow / AverageEndPointError -> libofb200 C ABI"),
        "e2e_fp32_inputs": e2e_fp32,
        "e2e_half_precision_producers": e2e_half,
        "gpu_launches": int(launches),
        "clocks": sampler.summary(t_wall0, t_wall1),
        "roofline": roofline,
        "kernels": kernels,
        "epe": {"device": epe_dev, "e2e": epe_e2e},
    }
    if world == 1 and not args.no_named:
        line["named_configs"] = named_kernel_table(torch)
    if world == 1 and not args.no_cpu:
        del batch, views
        torch.cuda.empty_cache()
        cb = time_cpu(1, 0, 1)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "ports")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=8, help="image pairs per GPU per step")
    ap.add_argument("--micro", type=int, default=8, help="pairs per pyramid build (device-resident arm)")
    ap.add_argument("--e2e-micro", type=int, default=1, help="pairs per staged micro-batch (host arm)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cta-group", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-named", action="store_true", help="skip the single-kernel named configs")
    ap.add_argument("--no-placement", action="store_true", help="ranks use cuda:LOCAL_RANK without probing the host links")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3                                   # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
