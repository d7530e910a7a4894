"""septfa_b200 - B200-native (sm_100a) Sep-TFAnet-VAD inference forward pass.

Drop-in for ``model/model.py::SeparationModel`` and the sliding-window online drivers of the
reference (BaekMS/Sep-TFAnet-VAD); the arithmetic runs in hand-written CUDA kernels behind the
C ABI declared in ``include/septfa.h``. Submodules are imported lazily so that the CPU-only
utilities (``synth``) work without torch or the CUDA library.
"""
import importlib as _importlib

__all__ = ["SeparationModel", "OnlineSaving", "OnlineSavingKnownTargets", "LiveSession", "PITLossWrapper",
           "reorder_source_mse", "calc_sisdr", "synth"]

_LAZY = {
    "SeparationModel": "model", "OnlineSaving": "online", "OnlineSavingKnownTargets": "online", "LiveSession": "live",
    "PITLossWrapper": "pit", "reorder_source_mse": "pit", "calc_sisdr": "pit",
}


def __getattr__(name):
    if name in _LAZY:
        return getattr(_importlib.import_module(f"{__name__}.{_LAZY[name]}"), name)
    if name in ("synth", "model", "online", "live", "pit", "lib", "shard", "inference", "evaluate"):
        return _importlib.import_module(f"{__name__}.{name}")
    raise AttributeError(name)
