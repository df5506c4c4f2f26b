"""Import the UNMODIFIED reference (test infrastructure / bench.py's reference arm only).

Where it is found, in this order:
  1. ``$CDR_REFERENCE_ROOT``;
  2. ``/root/reference`` — the read-only mount of the build container;
  3. ``baseline/_ref/`` — a verbatim, git-ignored copy of the reference's Python files that
     ``__graft_entry__.build()`` makes while (2) exists, so that the reference can ride to the
     GPU box next to the built ``.so`` (nothing under it is tracked or edited);
  4. ``oracle/_ref/`` — a git-ignored copy of the reference project placed there by hand.
``tests/golden/make_golden.py`` / ``make_driver_golden.py``, ``tests/test_reference_drivers.py``,
``tests/test_oracle_golden.py`` and ``bench.py --impl reference`` use this; the product package
never does.

Two third-party modules the reference imports are absent from this image and are stubbed before
the import — neither holds arithmetic of the hot path: ``matplotlib`` (plotting only,
tools/utils.py:3-4,10) and ``easydict`` (attribute access on the yaml config, inference.py:11).
"""
from __future__ import annotations

import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASELINE_REF = os.path.join(_REPO, "baseline", "_ref")
ORACLE_REF = os.path.join(_REPO, "oracle", "_ref")          # a git-ignored copy of the reference checkout, if one is placed there


def _candidates():
    env = os.environ.get("CDR_REFERENCE_ROOT")
    return ([env] if env else []) + ["/root/reference", BASELINE_REF, ORACLE_REF]


def root():
    """Directory holding the reference's models/cdrnet.py, or None."""
    for r in _candidates():
        if r and os.path.isfile(os.path.join(r, "models", "cdrnet.py")):
            return r
    return None


REF_ROOT = root() or "/root/reference"


def available() -> bool:
    return root() is not None


class EasyDict(dict):
    """Minimal stand-in for easydict.EasyDict (nested dict with attribute access)."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    def __setitem__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, EasyDict):
            v = EasyDict(v)
        super().__setitem__(k, v)

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    __setattr__ = __setitem__


def _stub_missing_modules():
    try:
        import matplotlib  # noqa: F401
    except ImportError:
        m = types.ModuleType("matplotlib")
        m.use = lambda *a, **k: None
        p = types.ModuleType("matplotlib.pyplot")
        m.pyplot = p
        sys.modules["matplotlib"] = m
        sys.modules["matplotlib.pyplot"] = p
    try:
        import easydict  # noqa: F401
    except ImportError:
        e = types.ModuleType("easydict")
        e.EasyDict = EasyDict
        sys.modules["easydict"] = e


def _import(names):
    r = root()
    if r is None:
        raise RuntimeError("reference not found (looked in " + ", ".join(_candidates()) + ")")
    _stub_missing_modules()
    # the reference's top-level packages are called `models` / `tools` / `dataset`; import them with
    # its root first on the path and restore the path afterwards
    saved = list(sys.path)
    sys.path.insert(0, r)
    try:
        import importlib
        return [importlib.import_module(n) for n in names]
    finally:
        sys.path[:] = saved


def load():
    """Returns a namespace with the reference's CDRNet, PoseResNet, calc_mpjpe,
    get_max_preds, triangulation, get_projection_matrix, project_3d_to_2d."""
    cdrnet, poseresnet, metrics, utils, common = _import(
        ["models.cdrnet", "models.poseresnet", "models.metrics", "tools.utils", "tools.common"])
    return types.SimpleNamespace(
        CDRNet=cdrnet.CDRNet, PoseResNet=poseresnet.PoseResNet, calc_mpjpe=metrics.calc_mpjpe,
        get_max_preds=utils.get_max_preds, triangulation=common.triangulation,
        get_projection_matrix=common.get_projection_matrix, project_3d_to_2d=common.project_3d_to_2d)


def load_drivers():
    """The reference's two inference drivers as modules: (inference, baseline) — inference.py:23-114
    (CDRNetInferencer) and baseline.py:22-103 (BaseLine).  Their module-level names CDRNet /
    PoseResNet / calc_mpjpe / get_max_preds / triangulation are what a drop-in replaces."""
    inference, baseline = _import(["inference", "baseline"])
    return inference, baseline


def load_config(name="mads_3d.yaml"):
    """configs/<name> of the reference as the EasyDict its drivers build (inference.py:127-128)."""
    import yaml
    with open(os.path.join(root(), "configs", name)) as f:
        return EasyDict(yaml.safe_load(f))


def sync_to_baseline_ref(src="/root/reference"):
    """Copy the reference's Python sources and configs verbatim into baseline/_ref/ (git-ignored, travels
    with gpurun).  No-op when `src` is absent (the GPU box).  Returns the number of files copied."""
    import shutil
    if not os.path.isfile(os.path.join(src, "models", "cdrnet.py")):
        return 0
    n = 0
    for dirpath, dirnames, filenames in os.walk(src):
        dirnames[:] = [d for d in dirnames if not d.startswith(".") and d != "__pycache__"]
        rel = os.path.relpath(dirpath, src)
        for f in filenames:
            if not f.endswith((".py", ".yaml", ".txt")):
                continue
            dst_dir = os.path.join(BASELINE_REF, rel) if rel != "." else BASELINE_REF
            os.makedirs(dst_dir, exist_ok=True)
            shutil.copyfile(os.path.join(dirpath, f), os.path.join(dst_dir, f))
            n += 1
    return n


def feature_stub(feats):
    """Stands in for ``model.encoder`` so the reference's own ``CDRNet.forward`` runs its
    post-encoder path (models/cdrnet.py:236-268) on given latents: returns the queued
    features in call order (left, right) while the image tensors still set img_size."""
    import torch

    class FeatureStub(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.feats = list(feats)
            self.i = 0

        def forward(self, x):
            f = self.feats[self.i % len(self.feats)]
            self.i += 1
            return f

    return FeatureStub()
