"""B200-native (sm_100a) robust two-view / pose estimation hot path of bioengstrom/tsbb15-3d-reconstruction-project.

Import as ``import tsbb15_b200`` (alias module at the repo root) — the directory name contains hyphens.
Sub-modules mirror the reference's flat modules: ``lab3``, ``fun``, ``ransac``, ``pnp``; ``batched`` / ``parallel``
are the multi-pair and multi-GPU entry points; ``runtime`` is the numpy-level view of the C ABI.
"""
from . import _cabi, runtime, sampling  # noqa: F401
from ._cabi import (MODE_EPI_MAX, MODE_SAMPSON, RGError, SCORE_FP32_GUARDED, SCORE_FP64, SOLVER_JACOBI, SOLVER_QR,  # noqa: F401
                    TIE_FIRST, TIE_REFERENCE, TRI_LINEAR, TRI_OPTIMAL)

from ._cabi import FLAG_BOUNDED, FLAG_REUSE_POINTS  # noqa: F401

__all__ = ["runtime", "sampling", "lab3", "fun", "ransac", "pnp", "tables", "help_classes", "correspondences", "batched",
           "parallel", "synth", "philox", "device"]


def __getattr__(name):
    if name in ("lab3", "fun", "ransac", "pnp", "tables", "help_classes", "correspondences", "batched", "parallel", "synth",
                "philox", "device"):
        import importlib
        return importlib.import_module(f"{__name__}.{name}")
    raise AttributeError(name)
