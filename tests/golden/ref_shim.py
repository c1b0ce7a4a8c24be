"""Import shim for the upstream reference (test infrastructure only).

Loads the reference's hot-path modules from its source tree (BACS_REFERENCE_ROOT, else the
copy oracle/make_ref.py stages under oracle/_ref/) WITHOUT running its package __init__
files (they pull in pytorch_lightning / hydra / wandb, which are not installed), by
registering empty namespace packages and stubbing the three third-party imports the hot
path touches.  Nothing is copied from the reference; this only makes `import
loss.bacs_loss` etc. work so golden vectors can be generated and the oracle can be pinned.
Nothing in the product package, the GPU tests, bench.py's GPU path or smoke() imports it.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("BACS_REFERENCE_ROOT") or os.path.join(
    os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "oracle", "_ref")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "loss"))


def _ns(name: str, path: str) -> None:
    mod = types.ModuleType(name)
    mod.__path__ = [path]
    sys.modules[name] = mod


def _stub(name: str, **attrs) -> types.ModuleType:
    mod = sys.modules.get(name)
    if mod is None:
        mod = types.ModuleType(name)
        mod.__path__ = []
        sys.modules[name] = mod
    for key, val in attrs.items():
        setattr(mod, key, val)
    return mod


def install():
    """Registers namespace packages + stubs; returns a dict of reference modules."""
    if not reference_available():
        raise RuntimeError("reference tree not found at %s" % REFERENCE_ROOT)
    import torch
    import torch.nn.functional as F

    class FocalLoss(torch.nn.Module):
        """Restatement of segmentation_models_pytorch.losses.FocalLoss(mode='binary')
        (un-vendored third party; SURVEY.md §8c says parity for it is 'unpinned')."""

        def __init__(self, mode, alpha=None, gamma=2.0, ignore_index=None,
                     reduction="mean", normalized=False, reduced_threshold=None):
            super().__init__()
            assert mode == "binary" and reduction == "mean"
            assert not normalized and reduced_threshold is None
            self.alpha, self.gamma, self.ignore_index = alpha, gamma, ignore_index

        def forward(self, y_pred, y_true):
            y_true = y_true.view(-1)
            y_pred = y_pred.view(-1)
            if self.ignore_index is not None:
                keep = y_true != self.ignore_index
                y_pred, y_true = y_pred[keep], y_true[keep]
            y_true = y_true.type(y_pred.type())
            logpt = F.binary_cross_entropy_with_logits(y_pred, y_true, reduction="none")
            pt = torch.exp(-logpt)
            loss = (1.0 - pt).pow(self.gamma) * logpt
            if self.alpha is not None:
                loss = loss * (self.alpha * y_true + (1 - self.alpha) * (1 - y_true))
            return loss.mean()

    class CombinedLoader:  # batch plumbing only; never exercised by the oracle
        def __init__(self, loaders, mode="max_size_cycle"):
            self.loaders, self.mode = loaders, mode

    _stub("segmentation_models_pytorch")
    _stub("segmentation_models_pytorch.losses", FocalLoss=FocalLoss)
    _stub("pytorch_lightning")
    _stub("pytorch_lightning.trainer")
    _stub("pytorch_lightning.trainer.supporters", CombinedLoader=CombinedLoader)
    _stub("pytorch_lightning.utilities")
    _stub("pytorch_lightning.utilities.memory", garbage_collection_cuda=lambda: None)
    _stub("hydra")
    _stub("hydra.utils", get_original_cwd=lambda: os.environ.get("BACS_REF_CWD", os.getcwd()))
    for pkg in ("training", "loss", "networks"):
        if pkg not in sys.modules or not hasattr(sys.modules[pkg], "__path__") \
                or sys.modules[pkg].__path__ != [os.path.join(REFERENCE_ROOT, pkg)]:
            _ns(pkg, os.path.join(REFERENCE_ROOT, pkg))
    import importlib
    mods = {}
    for name in ("training.loss_utils", "networks.bg_detector", "loss.base_loss",
                 "loss.prototypes", "training.buffer", "loss.experience_replay",
                 "loss.bacs_loss"):
        mods[name] = importlib.import_module(name)
    return mods
