"""world_size-2 gloo tests (CPU) of the multi-GPU host logic: contiguous pair sharding and the
(sum_epe, total) all-reduce behind AverageEndPointError.sync() / compute() -- the dist_reduce_fx="sum" semantics
of the reference's optical_flow/metrics/epe.py:22-23.  The per-rank metric state is what the K4c
kernel would have accumulated on that rank's shard; here the CPU oracle produces it."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, total_pairs, q):
    for p in (os.path.join(ROOT, "torch-optical-flow_b200"), ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    # CPU states on every rank: hide any GPU so an empty shard's state is not created on cuda:0
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      CUDA_VISIBLE_DEVICES="")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import oracle
        from ofb200.runner import shard_range
        from optical_flow.metrics.epe import AverageEndPointError

        r = np.random.default_rng(5)                       # same data on every rank, sharded below
        pred = r.standard_normal((total_pairs, 2, 12, 20)).astype(np.float32)
        target = r.standard_normal((total_pairs, 2, 12, 20)).astype(np.float32)
        valid = (r.random((total_pairs, 12, 20)) > 0.3).astype(np.float32)
        lo, hi = shard_range(total_pairs, rank, world)
        s, n = oracle.epe_sum_count(pred[lo:hi], target[lo:hi], valid[lo:hi]) if hi > lo else (0.0, 0)
        m = AverageEndPointError()
        if hi > lo:                                                    # a rank with an empty shard never calls update():
            m._acc = torch.tensor([s, float(n)], dtype=torch.float64)  # it must still take part in the collective
        g1 = m.sync()
        g2 = m.sync()                                                  # idempotent: the local state is not modified
        assert torch.equal(g1, g2)
        local = m._state().clone()
        assert float(local[0]) == s and int(local[1]) == n
        gs, gn = oracle.epe_sum_count(pred, target, valid)
        first = float(m.compute())
        # update -> sync -> update -> sync: a second batch (the same shard again) doubles both states exactly
        m._state().add_(torch.tensor([s, float(n)], dtype=torch.float64))
        g3 = m.sync()
        assert float(g3[1]) == 2 * gn and abs(float(g3[0]) - 2 * gs) <= 1e-9 * max(1.0, gs)
        q.put((rank, lo, hi, first, gs / gn, int(g1[1]), gn))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("total_pairs", [5, 8, 1])
def test_epe_sync_and_sharding_world2(total_pairs):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, total_pairs, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    res.sort()
    # shards are contiguous, disjoint and cover the batch
    assert res[0][1] == 0 and res[0][2] == res[1][1] and res[1][2] == total_pairs
    for _, _, _, got, ref, total, gn in res:
        assert total == gn
        assert abs(got - ref) <= 1e-6 * max(1.0, abs(ref))


def test_shard_range_properties():
    sys.path.insert(0, os.path.join(ROOT, "torch-optical-flow_b200"))
    from ofb200.runner import shard_range

    for total in (0, 1, 7, 64):
        for world in (1, 2, 4, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)
