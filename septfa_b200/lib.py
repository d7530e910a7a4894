"""ctypes binding of libseptfa.so (the C ABI in include/septfa.h).

There is no fallback: if the shared library is missing or cannot be loaded, importing this
module's :func:`load` raises. Build it with ``python -m septfa_b200.build`` (or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libseptfa.so")

ENGINE_TCGEN05_F16 = 0
FMT_F32, FMT_PCM16, FMT_F16 = 0, 1, 2   # host sample formats of septfa_forward_host_submit_fmt
ENGINE_FP32_SIMT = 7  # bit mask: 1 conv1d, 2 dconv+res_out, 4 output conv on fp32 CUDA cores


class SeptfaError(RuntimeError):
    pass


class Config(C.Structure):
    """septfa_config: arch.args of config_*.json (config_with_vad.json:7-28)."""
    _fields_ = [(n, C.c_int32) for n in (
        "n_fft_bins", "bn_dim", "h_dim", "layer", "stack", "num_spk", "skip", "dilated", "causal",
        "weight_norm", "final_vad", "final_vad_masked_speakers", "noisy_phase", "activity_input_bool",
        "tf_attention", "apply_recursive_ln", "apply_residual_ln")]

    @classmethod
    def from_args(cls, a):
        return cls(int(a["n_fftBins"]), int(a["BN_dim"]), int(a["H_dim"]), int(a["layer"]), int(a["stack"]),
                   int(a["num_spk"]), int(bool(a["skip"])), int(bool(a["dilated"])), int(bool(a["casual"])),
                   int(bool(a["weight_norm"])), int(bool(a["final_vad"])), int(bool(a["final_vad_masked_speakers"])),
                   int(bool(a["noisy_phase"])), int(bool(a["activity_input_bool"])), int(bool(a["tf_attention"])),
                   int(bool(a["apply_recursive_ln"])), int(bool(a["apply_residual_ln"])))


class InferKw(C.Structure):
    """septfa_infer_kw: inference_kw of forward (model/model.py:444-457)."""
    _fields_ = [("length_smoothing_filter", C.c_int32), ("threshold_activated_vad", C.c_float),
                ("filter_signals_by_smo_vad", C.c_int32), ("filter_signals_by_unsmo_vad", C.c_int32),
                ("return_smoothed_vad", C.c_int32)]

    KEYS = ("length_smoothing_filter", "threshold_activated_vad", "filter_signals_by_smo_vad",
            "filter_signals_by_unsmo_vad", "return_smoothed_vad")

    @classmethod
    def from_dict(cls, kw):
        """Empty dict -> None (the reference's ``if inference_kw``); otherwise all five keys are
        required, a missing one raises KeyError exactly like model/model.py:445-456."""
        if not kw:
            return None
        return cls(int(kw["length_smoothing_filter"]), float(kw["threshold_activated_vad"]),
                   int(bool(kw["filter_signals_by_smo_vad"])), int(bool(kw["filter_signals_by_unsmo_vad"])),
                   int(bool(kw["return_smoothed_vad"])))


_lib = None

_PROTOS = {
    "septfa_version": (C.c_char_p, []),
    "septfa_last_error": (C.c_char_p, [C.c_void_p]),
    "septfa_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Config), C.c_int]),
    "septfa_destroy": (None, [C.c_void_p]),
    "septfa_set_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "septfa_commit_weights": (C.c_int, [C.c_void_p]),
    "septfa_num_keys": (C.c_int, [C.c_void_p]),
    "septfa_key_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "septfa_key_numel": (C.c_int64, [C.c_void_p, C.c_int]),
    "septfa_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "septfa_get_option": (C.c_int, [C.c_void_p, C.c_char_p]),
    "septfa_num_frames": (C.c_int64, [C.c_int64]),
    "septfa_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int64]),
    "septfa_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.POINTER(InferKw), C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                 C.c_void_p]),
    "septfa_forward_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.POINTER(InferKw), C.c_void_p,
                                      C.c_void_p]),
    "septfa_forward_host_submit": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int64, C.POINTER(InferKw),
                                             C.c_void_p, C.c_void_p]),
    "septfa_forward_host_wait": (C.c_int, [C.c_void_p, C.c_int]),
    "septfa_forward_host_submit_fmt": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64,
                                                 C.POINTER(InferKw), C.c_void_p, C.c_int, C.c_void_p]),
    "septfa_last_launch_count": (C.c_int, [C.c_void_p]),
    "septfa_graph_capture": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.POINTER(InferKw), C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "septfa_graph_launch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "septfa_graph_num_nodes": (C.c_int, [C.c_void_p]),
    "septfa_graph_destroy": (None, [C.c_void_p]),
    "septfa_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_int, C.c_int]),
    "septfa_online_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "septfa_online_create_win": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "septfa_online_destroy": (None, [C.c_void_p]),
    "septfa_online_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "septfa_online_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "septfa_online_step": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(InferKw), C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "septfa_online_hops_done": (C.c_int, [C.c_void_p]),
    "septfa_live_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "septfa_live_create_win": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "septfa_live_create_rate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "septfa_live_create_rates": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "septfa_live_input_hop": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "septfa_live_output_hop": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "septfa_live_destroy": (None, [C.c_void_p]),
    "septfa_live_vad_frames": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "septfa_live_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "septfa_live_release": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "septfa_live_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(InferKw), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "septfa_resample_geometry": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "septfa_resample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "septfa_resample_to_geometry": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "septfa_resample_to": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "septfa_minmax_normalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "septfa_sisdr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "septfa_pit_l1": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)


def load():
    """dlopen libseptfa.so and declare every prototype. Raises SeptfaError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SeptfaError(f"{LIB_PATH} not found: build it with `python -m septfa_b200.build` "
                          "(there is no CPU / PyTorch fallback for this path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(handle, rc):
    if rc != 0:
        msg = load().septfa_last_error(handle)
        raise SeptfaError(f"septfa error {rc}: {msg.decode() if msg else ''}")


PROF_NAMES = ("frontend", "conv1", "dconv", "gate", "resid", "outconv", "vad", "istft", "export")


def num_frames(L):
    return 1 + int(L) // 256


RESAMPLE_MIN_RATE, RESAMPLE_MAX_RATE = 8000, 192000   # rates septfa_resample and septfa_resample_to accept


def resample_geometry(rate):
    """``(delay, hop_multiple)`` of ``rate`` from septfa_resample_geometry (no device needed): the delay D in 16 kHz
    samples of a streaming resampler, and the number a live hop at that rate must be a multiple of. Raises SeptfaError
    for a rate the library refuses."""
    lib = load()
    d, m = C.c_int(), C.c_int()
    rc = lib.septfa_resample_geometry(int(rate), C.byref(d), C.byref(m))
    check(None, rc)
    return d.value, m.value


def resample_to_geometry(rate):
    """``(delay, hop_multiple)`` of the output ``rate`` from septfa_resample_to_geometry (no device needed): the delay
    D_out in output samples of a streaming 16000 -> ``rate`` resampler, and the number a live hop (16 kHz samples) must
    be a multiple of for that output rate. Raises SeptfaError for a rate the library refuses."""
    lib = load()
    d, m = C.c_int(), C.c_int()
    rc = lib.septfa_resample_to_geometry(int(rate), C.byref(d), C.byref(m))
    check(None, rc)
    return d.value, m.value
