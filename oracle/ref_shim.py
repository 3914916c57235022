"""TEST INFRASTRUCTURE ONLY -- import shim for the *unmodified* reference tree.

Only usable in the build container, where ``/root/reference`` exists; nothing
under ``tests/ -m gpu``, ``smoke()`` or ``bench.py`` may import this module
(the GPU box has no reference tree).  It is used by ``oracle/make_golden.py``
to execute the reference's own torch code on the CPU and freeze the results
as fixtures under ``tests/golden/``, which pin the restatement in
``oracle/puzzle_oracle.py`` against the real thing.

Why a shim is needed (SURVEY.md D4): ``model5_b.py`` imports modules that are
not shipped with the reference (``pct``, ``pointtransformer_partseg``) or not
installed here (``pytorch_lightning``, ``open3d``, ``matplotlib``, ``pylab``,
``plyfile``, ``torchvision`` may or may not be present) and takes ``math`` /
``cm`` from ``from pylab import *`` (model5_b.py:57, used at :70).  We seed
``sys.modules`` with inert stand-ins *before* importing, never touching the
reference sources.
"""
from __future__ import annotations

import importlib
import math
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("PUZZLENET_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "model5_b.py"))


class _Anything:
    """Attribute sink: any attribute / call returns another sink."""

    def __init__(self, *a, **k):
        pass

    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return _Anything()

    def __call__(self, *a, **k):
        return _Anything()


def _stub(name: str, **attrs) -> types.ModuleType:
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    mod.__getattr__ = lambda attr: _Anything()  # type: ignore[attr-defined]
    mod.__path__ = []  # behave like a package so "import a.b" works
    sys.modules[name] = mod
    return mod


def _install_stubs() -> None:
    import torch.nn as nn

    def _have(name):
        try:
            importlib.import_module(name)
            return True
        except Exception:
            return False

    for name in ("open3d", "plyfile", "pct", "pointtransformer_partseg",
                 "emd_cuda"):
        if name not in sys.modules:
            _stub(name)
    if not _have("matplotlib"):
        _stub("matplotlib", use=lambda *a, **k: None, projections=_Anything())
        _stub("matplotlib.pyplot")
        _stub("mpl_toolkits")
        _stub("mpl_toolkits.mplot3d", Axes3D=_Anything)
        _stub("mpl_toolkits.mplot3d.art3d")
    if not _have("torchvision"):
        _stub("torchvision")
    if "pylab" not in sys.modules and not _have("pylab"):
        # model5_b.py:57 `from pylab import *` is where `math` comes from.
        mod = types.ModuleType("pylab")
        mod.math = math
        mod.cm = _Anything()
        mod.__all__ = ["math", "cm"]
        sys.modules["pylab"] = mod
    if not _have("pytorch_lightning"):
        class LightningModule(nn.Module):
            def save_hyperparameters(self, *a, **k):
                pass

            def log(self, *a, **k):
                pass

        pl = _stub("pytorch_lightning", LightningModule=LightningModule,
                   Trainer=_Anything, seed_everything=lambda *a, **k: None)
        cb = _stub("pytorch_lightning.callbacks", ModelCheckpoint=_Anything,
                   early_stopping=_Anything())
        pl.callbacks = cb


_loaded = {}


def load_reference():
    """Return a namespace with the reference modules (pointnet_util, model5_b, se3)."""
    if "ns" in _loaded:
        return _loaded["ns"]
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # make sure *our* same-named drop-in modules are not shadowing the reference
    for name in ("pointnet_util", "model5_b", "se_math", "PyTorchEMD"):
        mod = sys.modules.get(name)
        if mod is not None and not str(getattr(mod, "__file__", "")).startswith(REFERENCE_ROOT):
            del sys.modules[name]
    ns = types.SimpleNamespace()
    ns.pointnet_util = importlib.import_module("pointnet_util")
    ns.model5_b = importlib.import_module("model5_b")
    ns.se3 = importlib.import_module("se_math.se3")
    _loaded["ns"] = ns
    return ns


def reference_config():
    """The few fields TouchedRegraster.__init__/predict5 read (model5_b.py:601, :928)."""
    return types.SimpleNamespace(dataset="vase", pretrain_epochs=0, loss_sum=False,
                                 loss_mode=1, use_emd2=False, use_cd2=False,
                                 use_emd3=False, lr=0.9e-3, m=1, output_path="/tmp")
