"""The reference's hot-path modules (``merv/util/nn_utils.py``) for tests and the CPU baseline.

TEST INFRASTRUCTURE ONLY.  ``load_reference_nn_utils()`` returns

* the UNMODIFIED reference file, exec'd as a module, when ``MERV_REFERENCE_ROOT`` names a checkout of the reference (or a
  byte-for-byte copy was staged into git-ignored ``oracle/_ref/nn_utils.py`` by ``stage_reference()``).  ``import merv`` needs
  draccus/timm/decord/..., but the hot-path classes only need torch + einops; ``timm`` is imported at nn_utils.py:15-16 for
  out-of-scope classes, so a stub package is placed in ``sys.modules`` first;
* otherwise ``oracle/reference_nn.py``, the in-repository restatement of those classes, pinned to the reference's recorded
  outputs under ``tests/golden/``.
"""

from __future__ import annotations

import importlib.util
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("MERV_REFERENCE_ROOT", "")
_SOURCE = os.path.join(REFERENCE_ROOT, "merv", "util", "nn_utils.py") if REFERENCE_ROOT else ""
_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "nn_utils.py")
_NN_UTILS = _SOURCE if _SOURCE and os.path.isfile(_SOURCE) else _STAGED
_cached = None


def reference_available() -> bool:
    """True when the reference's own file is reachable (not the restatement)."""
    return os.path.isfile(_NN_UTILS)


def reference_origin() -> str:
    """Where the loaded file comes from (recorded in bench.py's cpu_baseline)."""
    return "MERV_REFERENCE_ROOT" if _NN_UTILS == _SOURCE else "oracle/_ref (staged copy of merv/util/nn_utils.py)"


def stage_reference() -> bool:
    """Copy the reference file into git-ignored ``oracle/_ref/`` (only where ``MERV_REFERENCE_ROOT`` names one).  Returns True if
    the staged copy exists afterwards."""
    if _SOURCE and os.path.isfile(_SOURCE):
        import shutil

        os.makedirs(os.path.dirname(_STAGED), exist_ok=True)
        if not os.path.isfile(_STAGED) or open(_STAGED, "rb").read() != open(_SOURCE, "rb").read():
            shutil.copyfile(_SOURCE, _STAGED)
    return os.path.isfile(_STAGED)


def load_reference_nn_utils():
    """Returns the reference module (``ref.AveragePooling3DProjector``, ``ref.CrossAttentionAdapterLearnableQuery`` ...)."""
    global _cached
    if _cached is not None:
        return _cached
    if not reference_available():
        from oracle import reference_nn

        _cached = reference_nn
        return _cached
    import torch

    if "timm" not in sys.modules:
        timm, layers, models, regnet = (
            types.ModuleType(n) for n in ("timm", "timm.layers", "timm.models", "timm.models.regnet")
        )
        layers.LayerNorm2d, layers.trunc_normal_, regnet.RegStage = torch.nn.LayerNorm, torch.nn.init.trunc_normal_, object
        timm.layers, timm.models, models.regnet = layers, models, regnet
        sys.modules.update(
            {"timm": timm, "timm.layers": layers, "timm.models": models, "timm.models.regnet": regnet}
        )
    spec = importlib.util.spec_from_file_location("ref_nn_utils", _NN_UTILS)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    _cached = ref
    return ref
