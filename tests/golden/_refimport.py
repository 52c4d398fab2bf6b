"""Import an unmodified reference checkout (OFB200_REFERENCE, else one staged under oracle/_ref/) for golden-vector
generation.

Only used by tests/golden/make_golden.py. Nothing in tests/, bench.py or the
product imports this at run time: the stored vectors are all the tests need.

The reference needs pytorch_lightning / torchmetrics (not installed): they are
stubbed with the minimum surface the hot path touches (SURVEY.md section 8c).
"""
import os
import sys
import types

import torch
from torch import nn

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "tools"))
from stage_reference import find_reference  # noqa: E402

REF = find_reference() or ""


def _stub_third_party():
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")

        class LightningModule(nn.Module):
            def save_hyperparameters(self):
                import inspect

                frame = inspect.currentframe().f_back
                args = {k: v for k, v in frame.f_locals.items() if k not in ("self", "__class__")}
                self.hparams = types.SimpleNamespace(**args)

        pl.LightningModule = LightningModule
        pl.LightningDataModule = object
        loggers = types.ModuleType("pytorch_lightning.loggers")
        loggers.WandbLogger = object
        pl.loggers = loggers
        sys.modules["pytorch_lightning"] = pl
        sys.modules["pytorch_lightning.loggers"] = loggers
    if "torchmetrics" not in sys.modules:
        tm = types.ModuleType("torchmetrics")

        class Metric(nn.Module):
            def add_state(self, name, default, dist_reduce_fx=None):
                self.register_buffer(name, default.clone())

        tm.Metric = Metric
        sys.modules["torchmetrics"] = tm
    if "wandb" not in sys.modules:
        try:
            import wandb  # noqa: F401
        except Exception:
            wb = types.ModuleType("wandb")
            wb.Image = object
            sys.modules["wandb"] = wb


def load_reference():
    """Returns (optical_flow module, model.corr, model.utils, RAFT class)."""
    if not os.path.isdir(os.path.join(REF, "methods", "raft", "model")):
        raise RuntimeError("set OFB200_REFERENCE to a checkout of the upstream torch-optical-flow project, or stage "
                           "one under oracle/_ref/")
    _stub_third_party()
    for name in list(sys.modules):
        if name == "optical_flow" or name.startswith("optical_flow.") or name == "model" or name.startswith("model."):
            del sys.modules[name]
    sys.path.insert(0, REF)
    try:
        import optical_flow  # noqa
        import optical_flow.metrics.epe as epe  # noqa

        pkg = types.ModuleType("model")
        pkg.__path__ = [REF + "/methods/raft/model"]
        sys.modules["model"] = pkg
        import model.corr as corr
        import model.utils as utils
        import model.raft as raft
    finally:
        sys.path.remove(REF)
    return optical_flow, corr, utils, raft.RAFT
