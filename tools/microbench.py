"""Per-kernel micro-benchmarks at the BASELINE.json shapes (CUDA events on the launching stream,
3 warm-ups, inputs rotated / larger than L2).  One record per kernel with the algorithmic
bytes / flops of SURVEY.md section 8d and the achieved fraction of the measured peaks.

    python tools/microbench.py [warp] [corr] [lookup] [upsample] [corr_big] [ondemand]

bench.py imports bench_warp_c2 / bench_corr_c3 / bench_lookup_c4 for its `named_configs` table."""
import ctypes
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
import torch  # noqa: E402

import ofb200  # noqa: E402
from model.corr import CorrBlock, prepare_operands  # noqa: E402
from ofb200.ops.corr import _default_pyramid_dtype, build_pyramid  # noqa: E402
from model.utils import coords_grid  # noqa: E402
from optical_flow import normalize  # noqa: E402

PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
try:
    PEAKS.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
except Exception:
    pass


def timeit(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def record(name, ms, nbytes=None, flops=None, **extra):
    rec = {"kernel": name, "ms": round(ms, 4)}
    if nbytes is not None:
        gbs = nbytes / ms / 1e6
        rec.update(gbs=round(gbs, 1), hbm_frac=round(gbs / PEAKS["hbm_gbs"], 3))
    if flops is not None:
        tf = flops / ms / 1e9
        rec.update(tflops=round(tf, 1), tensor_frac_sustained=round(tf / PEAKS["bf16_tflops_sustained"], 3),
                   tensor_frac_burst=round(tf / PEAKS["bf16_tflops"], 3))
    rec.update(extra)
    return rec


def smooth_flow(b, h, w, sigma, gen, spacing=16):
    low = torch.randn((b, 2, h // spacing + 2, w // spacing + 2), device="cuda", generator=gen) * sigma
    return torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=True).contiguous()


def bench_warp_c2(variants=(0,), flows=("white5px", "smooth5px"), masks=(1,)):
    """C2: batched bilinear warp + validity mask, 32x3x436x1024 fp32."""
    b, c, h, w = 32, 3, 436, 1024
    gen = torch.Generator(device="cuda").manual_seed(1234)
    frames = [torch.rand((b, c, h, w), device="cuda", generator=gen) for _ in range(2)]
    mk = {"white5px": lambda: normalize(5 * torch.randn((b, 2, h, w), device="cuda", generator=gen)),
          "smooth5px": lambda: normalize(smooth_flow(b, h, w, 5.0, gen)),
          # control points every 64 px: gradients <= ~0.1 px/px, the regime of real flow fields away from motion edges
          "smooth5px64": lambda: normalize(smooth_flow(b, h, w, 5.0, gen, 64)),
          "smooth20px64": lambda: normalize(smooth_flow(b, h, w, 20.0, gen, 64))}
    px = b * h * w
    lib = ofb200.load()
    out = torch.empty_like(frames[0])
    mask = torch.empty((b, h, w), dtype=torch.uint8, device="cuda")
    recs, k = [], [0]
    for fname in flows:
        flow = mk[fname]()
        for variant in variants:
            for with_mask in masks:
                def run():
                    k[0] ^= 1
                    rc = lib.ofb_warp_f32(ofb200.ptr(frames[k[0]]), ofb200.ptr(flow), ofb200.ptr(out),
                                          ofb200.ptr(mask) if with_mask else None, b, c, h, w, 0, 1, 0, 0, variant,
                                          1.0, 1.0, ofb200.stream_ptr())
                    assert rc == 0
                ms = timeit(run)
                recs.append(record(f"C2 K1 warp 32x3x436x1024 variant={variant} flow={fname} mask={with_mask}", ms,
                                   nbytes=px * (32 + with_mask), img_per_s=round(b / ms * 1e3)))
    return recs


def bench_warp_bwd_c2(flows=("white5px", "smooth5px")):
    """C2 backward: d frame (scatter-add) + d flow, 32x3x436x1024 fp32.  Bytes: frame, flow, d_out read; d_flow written;
    d_frame read-modify-written = 4 * (C + 2 + C + 2 + 2C) per pixel."""
    b, c, h, w = 32, 3, 436, 1024
    gen = torch.Generator(device="cuda").manual_seed(1234)
    frame = torch.rand((b, c, h, w), device="cuda", generator=gen)
    d_out = torch.randn((b, c, h, w), device="cuda", generator=gen)
    mk = {"white5px": lambda: normalize(5 * torch.randn((b, 2, h, w), device="cuda", generator=gen)),
          "smooth5px": lambda: normalize(smooth_flow(b, h, w, 5.0, gen))}
    lib = ofb200.load()
    d_frame = torch.zeros_like(frame)
    d_flow = torch.empty((b, 2, h, w), device="cuda")
    recs = []
    for fname in flows:
        flow = mk[fname]()

        def run():
            rc = lib.ofb_warp_backward_f32(ofb200.ptr(frame), ofb200.ptr(flow), ofb200.ptr(d_out), ofb200.ptr(d_frame),
                                           ofb200.ptr(d_flow), b, c, h, w, 1, 0, 1.0, 1.0, ofb200.stream_ptr())
            assert rc == 0
        ms = timeit(run)
        recs.append(record(f"C2 K1 warp backward 32x3x436x1024 flow={fname}", ms, nbytes=b * h * w * 4 * (4 * c + 4)))
    return recs


def _corr_setup(b, c, h, w, seed=1):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    return gen, f1, f2


def bench_corr(name, b, c, h, w, cta_groups=(0,), prep=True):
    gen, f1, f2 = _corr_setup(b, c, h, w)
    n = h * w
    recs = []
    # the operands of the pyramid CorrBlock(f1, f2) builds (OFB200_PYRAMID_DTYPE): fp16 for an fp16 pyramid, else bf16
    op_dt = torch.float16 if _default_pyramid_dtype() == torch.float16 else torch.bfloat16
    a_km, b_km, q_km = prepare_operands(f1, f2, 4, op_dt)
    ms = timeit(lambda: prepare_operands(f1, f2, 4, op_dt))
    if prep:
        recs.append(record(f"{name} K2 prep (fmap1, fmap2, fmap2/4x4)", ms, nbytes=b * c * n * (3 * 4 + 2 * 2 + 2 / 16)))
    blk = CorrBlock(f1, f2)
    elems = sum(int(blk._pyr.lvl_h[lv]) * int(blk._pyr.lvl_w[lv]) for lv in range(4)) * b * n
    for cg in cta_groups:
        def run():
            rc = build_pyramid((a_km, b_km, q_km), blk._pyr, b, c, h, w, op_dt, cg)
            assert rc == 0
        ms = timeit(run, reps=10)
        recs.append(record(f"{name} K2 corr pyramid cta_group={cg}", ms, nbytes=elems * 2 + 2 * b * n * c * 2,
                           flops=2.0 * b * n * n * c, pairs_per_s=round(b / ms * 1e3, 1)))
    return recs, blk, gen


def bench_corr_c3(cta_groups=(0,)):
    """C3: all-pairs correlation, 256-ch features at 1/8 of 436x1024 (55x128), 4-level pyramid, batch 16."""
    recs, blk, _ = bench_corr("C3 B16 55x128", 16, 256, 55, 128, cta_groups)
    del blk
    return recs


def bench_lookup(name, blk, gen, b, h, w, iters=12):
    lib = ofb200.load()
    st = ofb200.stream_ptr()
    n = h * w
    coords = coords_grid(b, h, w).cuda()[None] + 4 * torch.randn((iters, b, 2, h, w), device="cuda", generator=gen)
    out = torch.empty((b, 324, h, w), device="cuda")
    dt = blk._buffers[0].dtype
    esz = dt.itemsize

    def look():
        for it in range(iters):
            rc = lib.ofb_corr_lookup(ctypes.byref(blk._pyr), ofb200.ptr(coords[it]), ofb200.ptr(out), None, None,
                                     b, h, w, 4, st)
            assert rc == 0
    ms = timeit(look, reps=5) / iters
    return record(f"{name} K3 lookup r=4 x{iters} ({ {torch.bfloat16: 'bf16', torch.float16: 'fp16'}.get(dt, 'fp32')} pyramid), per iteration", ms,
                  nbytes=b * n * (4 * 100 * esz + 8 + 324 * 4), iters_ms=round(iters * ms, 3))


def bench_ondemand(name, b, c, h, w, iters=12, sigma=4.0):
    """On-demand correlation lookup (no materialised volume): time per iteration, and the memory it needs.
    sigma: px of white noise on the lookup coordinates (4 = the bench's; 0.25 = a smooth flow field)."""
    gen, f1, f2 = _corr_setup(b, c, h, w, seed=3)
    torch.cuda.reset_peak_memory_stats()
    m0 = torch.cuda.memory_allocated()
    blk = CorrBlock(f1, f2, on_demand=True)
    mem = torch.cuda.memory_allocated() - m0
    coords = coords_grid(b, h, w).cuda()[None] + sigma * torch.randn((iters, b, 2, h, w), device="cuda", generator=gen)
    out = torch.empty((b, 324, h, w), device="cuda")

    def look():
        for it in range(iters):
            blk(coords[it], out=out)
    ms = timeit(look, reps=3, warm=1) / iters
    n = h * w
    macs = 4 * 121 * c                                    # <= 11 x 11 positions per level
    return record(f"{name} on-demand corr lookup r=4 x{iters}, coords noise {sigma} px, per iteration", ms, flops=2.0 * b * n * macs,
                  operand_bytes_per_pair=round(mem / b), pyramid_bytes_per_pair_bf16=2 * n * sum((h >> l) * (w >> l) for l in range(4)))


def bench_lookup_c4():
    """C4: pyramid lookup radius 4 over 12 iterations at KITTI 375x1242 (47x156), batch 16, + convex upsampling."""
    b, c, h, w = 16, 256, 47, 156
    gen, f1, f2 = _corr_setup(b, c, h, w, seed=2)
    blk = CorrBlock(f1, f2)
    recs = [bench_lookup("C4 B16 47x156", blk, gen, b, h, w)]
    del blk
    recs.extend(bench_upsample_c4(epe=False, upflow=False))
    return recs


def bench_backward_c4():
    """C4 backward kernels: lookup backward (one iteration into the fp32 gradient pyramid), convex-upsample backward."""
    import ctypes
    b, c, h, w = 16, 256, 47, 156
    gen = torch.Generator(device="cuda").manual_seed(9)
    lib = ofb200.load()
    desc = ofb200.Pyramid()
    elems = (ctypes.c_int64 * ofb200.MAX_LEVELS)()
    ofb200.check(lib.ofb_pyramid_layout(h, w, 4, 0, ctypes.byref(desc), ctypes.byref(elems)), "layout")
    desc.dtype = ofb200.DTYPE_F32
    bufs = [torch.zeros(b * h * w * int(elems[l]), device="cuda") for l in range(4)]
    for l in range(4):
        desc.base[l] = bufs[l].data_ptr()
    base = torch.stack(torch.meshgrid(torch.arange(w, device="cuda"), torch.arange(h, device="cuda"), indexing="xy"), 0)[None].float()
    coords = (base + 4 * torch.randn((b, 2, h, w), device="cuda", generator=gen)).contiguous()
    d_out = torch.randn((b, 324, h, w), device="cuda", generator=gen)

    def lk():
        rc = lib.ofb_corr_lookup_backward_f32(ctypes.byref(desc), ofb200.ptr(coords), ofb200.ptr(d_out), b, h, w, 4, ofb200.stream_ptr())
        assert rc == 0
    ms = timeit(lk)
    q = b * h * w
    recs = [record("C4 B16 47x156 K3 lookup backward r=4, per iteration (fp32 gradient pyramid RMW)", ms,
                   nbytes=q * (4 * 81 * 4 + 4 * 100 * 8 + 8))]
    flow = torch.randn((b, 2, h, w), device="cuda", generator=gen)
    mask = torch.randn((b, 576, h, w), device="cuda", generator=gen)
    g_up = torch.randn((b, 2, 8 * h, 8 * w), device="cuda", generator=gen)
    d_flow = torch.zeros_like(flow)
    d_mask = torch.empty_like(mask)

    def up():
        rc = lib.ofb_convex_upsample_backward_f32(ofb200.ptr(flow), ofb200.ptr(mask), ofb200.ptr(g_up), ofb200.ptr(d_flow),
                                                  ofb200.ptr(d_mask), b, h, w, ofb200.stream_ptr())
        assert rc == 0
    ms = timeit(up)
    recs.append(record("C4 B16 47x156 K4b convex upsample backward", ms, nbytes=q * 4 * (576 * 2 + 128 + 4)))
    return recs


def bench_corr_train_c4(b=4, iters=12):
    """CorrBlock forward + backward at the KITTI size: build, `iters` lookups, then the backward pass (lookup backward
    kernels into the fp32 gradient pyramid, feature-map gradients through the library GEMMs), fp32 and bf16 GEMMs."""
    import os
    from model import CorrBlock
    c, h, w = 256, 47, 156
    gen = torch.Generator(device="cuda").manual_seed(11)
    f1 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    f2 = torch.randn((b, c, h, w), device="cuda", generator=gen)
    base = torch.stack(torch.meshgrid(torch.arange(w, device="cuda"), torch.arange(h, device="cuda"), indexing="xy"), 0)[None].float()
    coords = [(base + 3 * torch.randn((b, 2, h, w), device="cuda", generator=gen)).contiguous() for _ in range(iters)]
    wts = [torch.randn((b, 324, h, w), device="cuda", generator=gen) for _ in range(iters)]
    recs = []
    for mode in ("fp32", "bf16", "tcgen05"):
        os.environ["OFB200_BWD_GEMM"] = mode
        times = {"fwd": [], "bwd": []}
        for rep in range(4):
            a1, a2 = f1.clone().requires_grad_(True), f2.clone().requires_grad_(True)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            torch.cuda.synchronize()
            ev[0].record()
            blk = CorrBlock(a1, a2, num_levels=4, radius=4)
            total = sum((blk(cd) * wt).sum() for cd, wt in zip(coords, wts))
            ev[1].record()
            total.backward()
            ev[2].record()
            torch.cuda.synchronize()
            if rep:
                times["fwd"].append(ev[0].elapsed_time(ev[1]))
                times["bwd"].append(ev[1].elapsed_time(ev[2]))
        recs.append({"kernel": f"C4 B{b} 47x156 CorrBlock train step, {iters} lookups, d-fmap GEMMs in {mode}",
                     "fwd_ms": round(min(times["fwd"]), 3), "bwd_ms": round(min(times["bwd"]), 3)})
    del os.environ["OFB200_BWD_GEMM"]
    return recs


def bench_gemm_nt(shapes=((16, 7332, 256, 7332), (8, 32640, 256, 32640), (16, 7332, 256, 1833))):
    """The backward GEMM kernel alone: D[M x N] = A[M x K] . B[N x K]^T, bf16 in, fp32 out (level-0 shapes of C4 / C5)."""
    lib = ofb200.load()
    recs = []
    for (b, m, n, k) in shapes:
        gen = torch.Generator(device="cuda").manual_seed(2)
        pk = (k + 7) // 8 * 8
        a = torch.randn((b, m, pk), device="cuda", generator=gen).to(torch.bfloat16)
        bb = torch.randn((b, n, pk), device="cuda", generator=gen).to(torch.bfloat16)
        d = torch.empty((b, m, n), device="cuda")

        def run():
            rc = lib.ofb_gemm_nt_bf16(ofb200.ptr(a), ofb200.ptr(bb), ofb200.ptr(d), b, m, n, k, pk, pk, n, m * pk, n * pk, m * n,
                                      1.0, 0, ofb200.stream_ptr())
            assert rc == 0
        ms = timeit(run)
        flops = 2.0 * b * m * n * k
        recs.append({"kernel": f"backward GEMM B{b} M{m} N{n} K{k} (bf16 -> fp32)", "ms": round(ms, 4),
                     "tflops": round(flops / ms / 1e9, 1), "tensor_frac_sustained": round(flops / ms / 1e9 / 1391.6, 3),
                     "gbs_A_stream": round(b * m * pk * 2 / ms / 1e6, 1)})
    return recs


def bench_sequence_loss_c4(n_pred=12):
    """sequence_loss over 12 full-resolution predictions at the C4 (KITTI) size: 8 B/px per prediction + 12 B/px."""
    import ctypes
    n, h, w = 16, 376, 1248
    gen = torch.Generator(device="cuda").manual_seed(5)
    gt = 8 * torch.randn((n, 2, h, w), device="cuda", generator=gen)
    valid = (torch.rand((n, h, w), device="cuda", generator=gen) > 0.1).float()
    preds = [gt + torch.randn((n, 2, h, w), device="cuda", generator=gen) for _ in range(n_pred)]
    acc = torch.zeros(6, dtype=torch.float64, device="cuda")
    ptrs = (ctypes.c_void_p * n_pred)(*[p.data_ptr() for p in preds])
    lib = ofb200.load()

    def run():
        rc = lib.ofb_sequence_loss_f32(ptrs, n_pred, ofb200.ptr(gt), ofb200.ptr(valid), ofb200.ptr(acc), n, h, w, 0.8, 400.0,
                                       ofb200.stream_ptr())
        assert rc == 0
    ms = timeit(run)
    return [record(f"C4 B16 376x1248 K4d sequence_loss x{n_pred} predictions", ms, nbytes=n * h * w * (8 * n_pred + 12))]


def bench_upsample_c4(epe=True, upflow=True):
    n, h, w = 16, 47, 156
    gen = torch.Generator(device="cuda").manual_seed(3)
    masks = [torch.randn((n, 576, h, w), device="cuda", generator=gen) for _ in range(2)]
    flow = torch.randn((n, 2, h, w), device="cuda", generator=gen)
    lib = ofb200.load()
    out = torch.empty((n, 2, 8 * h, 8 * w), device="cuda")
    k = [0]
    recs = []

    def run():
        k[0] ^= 1
        rc = lib.ofb_convex_upsample_f32(ofb200.ptr(flow), ofb200.ptr(masks[k[0]]), ofb200.ptr(out), n, h, w, ofb200.stream_ptr())
        assert rc == 0
    ms = timeit(run)
    recs.append(record("C4 B16 47x156 K4b convex upsample", ms, nbytes=n * h * w * (578 * 4 + 128 * 4), pairs_per_s=round(n / ms * 1e3)))
    if upflow:
        flows = [torch.randn((n, 2, h, w), device="cuda", generator=gen) for _ in range(4)]
        outs = [torch.empty((n, 2, 8 * h, 8 * w), device="cuda") for _ in range(4)]

        def up():
            k[0] = (k[0] + 1) % 4
            rc = lib.ofb_resize_bilinear_f32(ofb200.ptr(flows[k[0]]), ofb200.ptr(outs[k[0]]), n, 2, h, w, 8 * h, 8 * w, 1, 8.0, 8.0, ofb200.stream_ptr())
            assert rc == 0
        ms = timeit(up)
        recs.append(record("C4 K4a upflow8", ms, nbytes=n * 2 * h * w * 4 * 65))
    if epe:
        preds = [torch.randn((n, 2, 8 * h, 8 * w), device="cuda", generator=gen) for _ in range(3)]
        tgts = [torch.randn((n, 2, 8 * h, 8 * w), device="cuda", generator=gen) for _ in range(3)]
        valid = (torch.rand((n, 8 * h, 8 * w), device="cuda", generator=gen) > 0.1).float()
        acc = torch.zeros(2, dtype=torch.float64, device="cuda")

        def epe_fn():
            k[0] = (k[0] + 1) % 3
            rc = lib.ofb_epe_reduce_f32(ofb200.ptr(preds[k[0]]), ofb200.ptr(tgts[k[0]]), ofb200.ptr(valid), ofb200.ptr(acc), n, 8 * h, 8 * w, ofb200.stream_ptr())
            assert rc == 0
        ms = timeit(epe_fn)
        recs.append(record("C4 K4c EPE reduce (valid map)", ms, nbytes=n * 8 * h * 8 * w * 20))
    return recs


def main():
    which = sys.argv[1:] or ["warp", "corr", "lookup", "upsample"]
    print(json.dumps({"peaks": {k: PEAKS[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained")}}))

    def emit(recs):
        for r in recs:
            print(json.dumps(r), flush=True)

    if "warp" in which:
        emit(bench_warp_c2(variants=(1, 2, 0), masks=(0, 1)))
    if "upsample" in which:
        emit(bench_upsample_c4())
    if "corr" in which or "lookup" in which:
        for name, shp in {"C3 B16 55x128": (16, 256, 55, 128), "C4 B16 47x156": (16, 256, 47, 156),
                          "C5 B4 136x240": (4, 256, 136, 240)}.items():
            recs, blk, gen = bench_corr(name, *shp, cta_groups=(1, 2))
            emit(recs)
            emit([bench_lookup(name, blk, gen, shp[0], shp[2], shp[3])])
            del blk
            torch.cuda.empty_cache()
    if "ondemand" in which:
        emit([bench_ondemand("C4 B16 47x156", 16, 256, 47, 156), bench_ondemand("C5 B8 136x240", 8, 256, 136, 240),
              bench_ondemand("C5 B8 136x240", 8, 256, 136, 240, sigma=0.25)])


if __name__ == "__main__":
    main()
