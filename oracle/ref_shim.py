"""Imports the UNMODIFIED reference (DIAGNijmegen/bodyct-dram-emph-subtype) on CPU.  Test infrastructure.

The reference needs pytorch_lightning, hydra, omegaconf, SimpleITK, matplotlib and seaborn, none
of which is installed in this image; they are only used for orchestration, plotting and file I/O,
never for arithmetic on the hot path.  `load()` plants minimal stand-ins in sys.modules, puts the
reference checkout on sys.path, chdir()s into it (utils.py:84 opens ./conf/<name>.yaml relative to
the cwd) and imports its modules.  Works only where DRAM_REFERENCE_DIR names a checkout of the
upstream project; used by make_golden.py and by the parity-pinning tests that skip without one.
"""
import contextlib
import enum
import importlib
import os
import sys
import types

REF_DIR = os.environ.get("DRAM_REFERENCE_DIR", "")

_REF_MODULES = ["med3d", "models", "utils", "dataset", "base", "functional", "intensity_transforms",
                "spatial_transforms", "metrics", "sampler", "data_sampler", "confusion_matrix"]


def available():
    return bool(REF_DIR) and os.path.isfile(os.path.join(REF_DIR, "med3d.py"))


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def _plant_stubs():
    import torch
    import yaml

    class LightningModule(torch.nn.Module):
        def save_hyperparameters(self, *a, **k):
            pass

    class LightningDataModule:
        def __init__(self, *a, **k):
            pass

    class RunningStage(str, enum.Enum):
        TRAINING = "train"
        VALIDATING = "validate"
        TESTING = "test"
        PREDICTING = "predict"

    class _Anything:
        def __init__(self, *a, **k):
            pass

    pl = _module("pytorch_lightning", LightningModule=LightningModule, LightningDataModule=LightningDataModule)
    pl.loggers = _module("pytorch_lightning.loggers", TensorBoardLogger=_Anything)
    pl.trainer = _module("pytorch_lightning.trainer")
    pl.trainer.states = _module("pytorch_lightning.trainer.states", RunningStage=RunningStage)
    _module("SimpleITK")
    mpl = _module("matplotlib", use=lambda *a, **k: None)
    mpl.pyplot = _module("matplotlib.pyplot", Axes=_Anything)
    mpl.backends = _module("matplotlib.backends")
    mpl.backends.backend_agg = _module("matplotlib.backends.backend_agg", FigureCanvasAgg=_Anything)
    mpl.font_manager = _module("matplotlib.font_manager")
    mpl.collections = _module("matplotlib.collections", QuadMesh=_Anything)
    mpl.figure = _module("matplotlib.figure", Axes=_Anything, Figure=_Anything)
    mpl.text = _module("matplotlib.text", Text=_Anything)
    _module("seaborn")

    class OmegaConf:
        @staticmethod
        def load(path):
            with open(path) as f:
                return yaml.safe_load(f)

    _module("omegaconf", OmegaConf=OmegaConf)

    def instantiate(cfg):
        cfg = dict(cfg)
        mod, fn = cfg.pop("_target_").rsplit(".", 1)
        return getattr(importlib.import_module(mod), fn)(**cfg)

    hydra = _module("hydra")
    hydra.utils = _module("hydra.utils", instantiate=instantiate)


@contextlib.contextmanager
def reference_cwd():
    old = os.getcwd()
    os.chdir(REF_DIR)
    try:
        yield
    finally:
        os.chdir(old)


_loaded = None


def load():
    """Returns a namespace with the reference modules (`.med3d`, `.models`, ...)."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise FileNotFoundError(f"no reference checkout: set DRAM_REFERENCE_DIR (now {REF_DIR!r})")
    for name in _REF_MODULES:
        if name in sys.modules and not getattr(sys.modules[name], "__file__", "").startswith(REF_DIR):
            raise RuntimeError(f"module name clash: '{name}' is already imported from elsewhere")
    _plant_stubs()
    sys.path.insert(0, REF_DIR)
    ns = types.SimpleNamespace()
    with reference_cwd():
        for name in ["med3d", "functional", "base", "intensity_transforms", "utils", "spatial_transforms",
                     "dataset", "models"]:
            setattr(ns, name, importlib.import_module(name))
    _loaded = ns
    return ns


def model(arch):
    """The reference nn.Module for a conf/<arch>.yaml key (utils.py:83-85)."""
    ref = load()
    with reference_cwd():
        return ref.utils.get_model_by_name(arch).eval()
