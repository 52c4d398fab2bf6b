"""bench.py --dump-outputs: what the last timed step computed, written as .npy files that are the same from run to run
(the inputs are seeded), so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = ["corr.npy", "epe_state.npy", "flow_up.npy", "mask.npy", "warped.npy"]


def run_bench(out_dir, cwd):
    # two micro-batches of one pair: the second reuses the first one's lookup buffer
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--pairs", "2", "--micro", "1",
           "--e2e-steps", "1", "--no-named", "--no-cpu", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=cwd)
    assert res.returncode == 0, res.stdout[-2000:] + "\n" + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dump_outputs_are_reproducible(tmp_path):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    dumps = []
    for run in range(2):
        out_dir = tmp_path / f"run{run}"
        line = run_bench(out_dir, tmp_path)
        assert line["steps"] == 2
        assert sorted(os.listdir(out_dir)) == FILES
        assert sum(os.path.getsize(out_dir / f) for f in FILES) <= 64_000_000
        dumps.append({f[:-4]: np.load(out_dir / f) for f in FILES})
        state = dumps[-1]["epe_state"]
        assert state.dtype == np.float64 and state.shape == (2,)
        assert state[0] / state[1] == pytest.approx(line["epe"]["device"], rel=1e-6)   # the timed steps' metric state
    a, b = dumps
    for name in ("corr", "flow_up", "warped", "mask"):
        assert a[name].dtype == np.float32 and a[name].shape[0] == 2, name
        assert np.isfinite(a[name]).all(), name
        assert np.array_equal(a[name], b[name]), name
    assert not np.array_equal(a["corr"][0], a["corr"][1])       # pair 0 was sampled before pair 1 overwrote the buffer
    assert set(np.unique(a["mask"])) <= {0.0, 1.0}
    assert a["epe_state"][1] == b["epe_state"][1]
    assert a["epe_state"][0] == pytest.approx(b["epe_state"][0], rel=1e-12)     # per-CTA float64 atomics: order may vary

    # every dumped value is the output at its documented position: rerun the pass pair by pair on the same seeded
    # inputs and index each full output with positions drawn from the rule bench.py states
    sys.path.insert(0, ROOT)
    import bench
    from ofb200.runner import FIELDS, hot_path
    from optical_flow.metrics.epe import AverageEndPointError

    batch = bench.make_batch(2, torch.device("cuda", 0), 1234, torch)
    n = 60_000_000 // (16 * 2)
    for p in range(2):
        v = {k: (batch[k][:, p:p + 1] if k == "coords" else batch[k][p:p + 1]).contiguous() for k in FIELDS}
        out = hot_path(v, AverageEndPointError())
        for i, name in enumerate(("corr", "flow_up", "warped", "mask")):
            full = out[name][0].float().cpu().numpy().reshape(-1)
            pos = np.sort(np.random.default_rng(i).choice(full.size, n, replace=False))
            assert np.array_equal(a[name][p], full[pos]), (name, p)
