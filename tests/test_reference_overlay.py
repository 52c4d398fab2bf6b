"""The drop-in boundary next to a real reference checkout (SURVEY.md section 8b and 8f row 1).

CPU part (`-m "not gpu"`): in fresh interpreters, (1) with `torch-optical-flow_b200/` ahead of the reference on
sys.path and (2) with the reference imported first and `ofb200.patch_reference()` applied, the hot-path names are this
repository's while `read`, `write`, `flow2rgb`, `colorwheel` (reference optical_flow/__init__.py:1,3), the encoders,
the update block and the RAFT LightningModule itself keep coming from the reference.  No kernel runs.

GPU part: the UNMODIFIED reference `RAFT` (methods/raft/model/raft.py:87-147; random weights, fixed seed, Lightning
stubbed) runs 12 refinement iterations on a Sintel-size pair once on its stock ATen ops and once per overlay mode;
the final flows must agree.  Tolerances: fp32 pyramid <= 1e-4 * |ref|_inf on the full-resolution flow; bf16 pyramid
(the reference's `precision: 16` storage) <= 2e-2 * |ref|_inf -- twelve recurrent GRU iterations on a volume with
4e-3 relative rounding.

The reference is an unmodified checkout of the upstream torch-optical-flow project, which this repository does not
contain: the one OFB200_REFERENCE names, else one staged under the git-ignored oracle/_ref/ (`__graft_entry__.build()`
stages it there when OFB200_REFERENCE is set, tools/stage_reference.py).  Without either these tests skip.
"""
import hashlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE = os.path.join(ROOT, "tests", "overlay_probe.py")
NO_REFERENCE = ("no checkout of the upstream torch-optical-flow project: set OFB200_REFERENCE to one, or stage it "
                "under oracle/_ref/ (tools/stage_reference.py)")
sys.path.insert(0, os.path.join(ROOT, "tools"))
from stage_reference import find_reference as reference_root  # noqa: E402


def run_probe(*args, env=None, timeout=900):
    e = dict(os.environ)
    e.pop("PYTHONPATH", None)
    e.update(env or {})
    res = subprocess.run([sys.executable, PROBE, *args], capture_output=True, text=True, timeout=timeout, env=e)
    assert res.returncode == 0, res.stdout[-2000:] + "\n" + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


HOT = ["optical_flow.warp", "operator.warp", "operator.warp_grid", "optical_flow.resize", "RAFT.upsample_flow",
       "raft.CorrBlock", "model.corr.CorrBlock", "model.utils.bilinear_sampler", "model.utils.upflow8",
       "raft.sequence_loss", "epe.update"]
KEPT = ["optical_flow.flow2rgb", "optical_flow.read", "optical_flow.write", "optical_flow.colorwheel", "model.RAFT",
        "model.RAFT.forward", "model.update.BasicUpdateBlock", "model.extractor.BasicEncoder"]


@pytest.mark.parametrize("mode", ["path", "patch"])
def test_overlay_keeps_the_reference_working(mode):
    ref = reference_root()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    r = run_probe("names", mode, ref)
    assert all(r[k] == "ours" for k in HOT), {k: r[k] for k in HOT}
    assert all(r[k] == "reference" for k in KEPT), {k: r[k] for k in KEPT}
    assert r["metric_is_torchmetrics"]                  # the Metric subclass (states, sync, logging) is the reference's
    assert r["flow2rgb_shape"] == [3, 4, 5]             # the fall-through visualisation really runs
    if mode == "patch":
        assert r["unpatched"] == len(r["patched"]) == 24 and r["after_unpatch.warp"] == "reference"


def test_stock_reference_is_untouched_without_overlay():
    ref = reference_root()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    r = run_probe("names", "stock", ref)
    assert all(r[k] == "reference" for k in HOT + KEPT)


def test_vendored_reference_test_is_verbatim():
    """tests/golden/reference_tests/test_operator.py is the reference's file, byte for byte."""
    path = os.path.join(ROOT, "tests", "golden", "reference_tests", "test_operator.py")
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()
    assert digest == "7df2879fbf3f720c389385a8915a20102c7c996545a562accfe66eb1746de193"
    ref = reference_root()
    if ref is not None:
        upstream = os.path.join(ref, "tests", "operator", "test_operator.py")
        assert hashlib.sha256(open(upstream, "rb").read()).hexdigest() == digest


def test_drop_in_without_a_reference_says_what_is_missing():
    """Without a reference on the path the hot-path names work and the fall-through names raise ImportError."""
    code = ("import sys; sys.path.insert(0, %r); import optical_flow, model\n"
            "assert optical_flow.warp.__module__ == 'ofb200.ops.operator' and model.RAFT.__module__ == 'ofb200.ops.raft_ops'\n"
            "try:\n    from optical_flow import flow2rgb\nexcept ImportError as e:\n    print('OK', 'reference checkout' in str(e))\n"
            % os.path.join(ROOT, "torch-optical-flow_b200"))
    e = dict(os.environ)
    e.pop("PYTHONPATH", None)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=e, cwd="/")
    assert res.returncode == 0 and res.stdout.strip() == "OK True", res.stdout + res.stderr


# ------------------------------------------------------------------------------------------- GPU: live RAFT.forward
def _flows(path):
    import torch

    d = torch.load(path)
    return d["flow_lo"].double(), d["flow_up"].double()


@pytest.mark.gpu
def test_live_raft_forward_matches_stock_reference(tmp_path):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    ref = reference_root()
    if ref is None:
        pytest.skip(NO_REFERENCE)
    report = {"stock": run_probe("raft", "stock", ref, str(tmp_path / "stock.pt"))}
    lo0, up0 = _flows(tmp_path / "stock.pt")
    scale = float(up0.abs().max())
    assert scale > 0
    cases = [("patch", "fp32", 1e-4), ("path", "fp32", 1e-4), ("patch", "bf16", 2e-2), ("path", "bf16", 2e-2)]
    for mode, dt, rel in cases:
        out = tmp_path / f"{mode}_{dt}.pt"
        r = run_probe("raft", mode, ref, str(out), env={"OFB200_PYRAMID_DTYPE": dt})
        lo, up = _flows(out)
        err = float((up - up0).abs().max())
        r["max_abs_err_full_res"] = err
        r["rel_err"] = err / scale
        report[f"{mode}_{dt}"] = r
        assert r["ofb_launches"] >= 3 * (3 + 12 + 12), r          # the kernels really ran inside the live model
        assert err <= rel * scale, (mode, dt, err, scale)
        assert float((lo - lo0).abs().max()) <= rel * max(1.0, float(lo0.abs().max())), (mode, dt)
    print(json.dumps(report))
