"""Live streaming sessions: one hop per stream slot per push, streams that start and end independently, VAD per hop.

``OnlineSaving.calc_online`` drives S streams in lockstep over whole recordings the caller already holds. A
:class:`LiveSession` serves streams as they arrive: each slot hosts one stream at a time, every push carries one new
hop for any subset of the slots, and the session keeps each stream's last ``window - hop`` input samples and emitted
samples on the device (``septfa_live_*`` in ``include/septfa.h``). With a window of W and a hop of H samples (default
48000 / 16000), push k of a stream returns the stream's separated samples ``[H k, H (k + 1))``: the concatenated output
of a stream of N pushes equals ``OnlineSaving.calc_online(F.pad(x, (W - H, 0)))`` with ``max_len = W / 16000`` and
``save_sec = H / 16000`` on that stream alone (the windowing of ``model/online_class_known_targets.py:92-93``, the
stitch of ``model/online_class_unknown_targets.py:84-94``). The oldest sample of a hop comes back about H samples after
it was taken, plus the push time: the hop sets the latency.

A session at another input ``rate`` (8 .. 192 kHz) takes ``input_hop = hop * rate / 16000`` native samples per push and
resamples each stream on the device (``septfa_live_create_rate``), carrying the resampler's history from push to push.
It then serves the 16 kHz stream ``u = concat(delay zeros, resample(x))``: the output lags the input by ``delay``
samples (6 .. 12, see ``septfa_resample_geometry``) on top of the hop.

A session with another ``out_rate`` (8 .. 192 kHz, independent of ``rate``) returns ``output_hop = hop * out_rate /
16000`` samples per channel and push: the 16 kHz output resampled on the device (``septfa_live_create_rates``), i.e.
``concat(out_delay zeros, model.resample_to(y))`` of the 16 kHz output stream y, cut into hops. ``out_delay`` (0 at
16000, 18 at 48 kHz, see ``septfa_resample_to_geometry``) is in output samples. VAD and permutations are unchanged.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import lib as _lib

RATE = 16000             # the model's rate, and the default input rate
WINDOW = 48000
HOP = 16000              # the default hop
FRAMES_PER_HOP = 63      # VAD frames per push at the default geometry
MAX_WINDOW = 160000      # 10 s


def check_geometry(window, hop, rate=RATE, out_rate=RATE):
    """``(window, hop)`` as ints if the library accepts them: 256 <= hop, 2 hop <= window <= 160000, both multiples of 16
    samples (1 ms); ``rate`` and ``out_rate`` integers in 8000 .. 192000 Hz, and the hop a multiple of
    ``16000 / gcd(r, 16000)`` for both, so that a push carries a whole number of native samples and returns a whole
    number of output samples (160 at 44.1 kHz, any hop at 48 kHz). ``ValueError`` otherwise."""
    if not all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in (window, hop, rate, out_rate)):
        raise ValueError(f"window, hop, rate and out_rate are integers, got {window!r}, {hop!r}, {rate!r}, {out_rate!r}")
    window, hop, rate, out_rate = int(window), int(hop), int(rate), int(out_rate)
    for name, r in (("rate", rate), ("out_rate", out_rate)):
        if not _lib.RESAMPLE_MIN_RATE <= r <= _lib.RESAMPLE_MAX_RATE:
            raise ValueError(f"{name} = {r}: must lie in {_lib.RESAMPLE_MIN_RATE} .. {_lib.RESAMPLE_MAX_RATE} Hz")
        step = RATE // math.gcd(r, RATE)
        if hop % step:
            raise ValueError(f"{name} = {r}, hop = {hop}: the hop must be a multiple of {step} samples at this rate")
    if hop < 256:
        raise ValueError(f"hop = {hop}: must be >= 256 samples")
    if window < 2 * hop:
        raise ValueError(f"window = {window}, hop = {hop}: the window must be >= 2 hops")
    if window > MAX_WINDOW:
        raise ValueError(f"window = {window}: must be <= {MAX_WINDOW} samples (10 s)")
    if window % 16 or hop % 16:
        raise ValueError(f"window = {window}, hop = {hop}: both must be multiples of 16 samples (1 ms)")
    return window, hop


def check_slots(slots, capacity):
    """``slots`` as a contiguous int32 array of distinct slots in ``0 .. capacity - 1``, 1 <= len <= capacity;
    ``ValueError`` otherwise."""
    a = np.asarray(slots.cpu() if isinstance(slots, torch.Tensor) else slots)
    if a.ndim != 1 or not (1 <= a.size <= capacity):
        raise ValueError(f"a slot list is a 1-D list of 1 .. {capacity} slots, got shape {a.shape}")
    if not np.issubdtype(a.dtype, np.integer):
        raise ValueError(f"slots must be integers, got {a.dtype}")
    if a.min() < 0 or a.max() >= capacity:
        raise ValueError(f"slots must lie in 0 .. {capacity - 1}, got {a.min()} .. {a.max()}")
    if np.unique(a).size != a.size:
        raise ValueError("a slot may appear only once per call")
    return np.ascontiguousarray(a, dtype=np.int32)


class LiveSession:
    """``capacity`` stream slots on one device, for a :class:`~septfa_b200.model.SeparationModel`.

    Every stream has a window of ``window`` and a hop of ``hop`` samples at 16 kHz and arrives at ``rate`` Hz (see
    :func:`check_geometry`). ``push(slots, hops)`` takes one hop (``input_hop`` float32 samples at ``rate``, already
    normalised) for each listed slot and returns
    ``(out [n, 2, hop], vad [n, 2, frames_per_hop] or None, perm [n, 2] int32)`` on the device, stream-ordered on the
    current stream. ``vad`` holds the window frames ``first_frame .. first_frame + frames_per_hop - 1`` of the window's
    VAD output, those centred on the new hop (frame j centred on window sample ``256 j``; 125 .. 187 at the default),
    speakers in the emitted order; it is None for a model without a VAD head or with ``vad=False``. ``release(slots)``
    ends the streams in those slots: the next push into one starts a new stream. ``inference_kw`` is the forward's
    (gating, smoothed VAD), fixed for the session. At a rate other than 16000 the outputs are those of a 16 kHz session
    fed ``concat(delay zeros, model.resample(stream))``; ``delay`` is 0 at 16000. At an ``out_rate`` other than 16000,
    ``out`` is ``[n, 2, output_hop]``: hop k of ``concat(out_delay zeros, model.resample_to(y, out_rate))`` per channel,
    y the channel's 16 kHz output stream; ``out_delay`` is 0 at 16000.
    """

    def __init__(self, model, capacity, inference_kw=None, device=None, window=WINDOW, hop=HOP, rate=RATE,
                 out_rate=RATE):
        self.model = model
        self.capacity = int(capacity)
        if not 1 <= self.capacity <= 32767:
            raise ValueError("capacity must lie in 1 .. 32767")
        self.window, self.hop = check_geometry(window, hop, rate, out_rate)
        self.rate, self.out_rate = int(rate), int(out_rate)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("septfa_b200.LiveSession runs on CUDA only (no CPU fallback)")
        self._kw = _lib.InferKw.from_dict(inference_kw) if (inference_kw and model.final_vad) else None
        self._lv = C.c_void_p()
        with torch.cuda.device(self.device):
            self._h = model._handle(self.device)
            _lib.check(self._h.ptr, self._h.lib.septfa_live_create_rates(self._h.ptr, self.capacity, self.window, self.hop,
                                                                         self.rate, self.out_rate, C.byref(self._lv)))
            delay = C.c_int()
            self.input_hop = self._h.lib.septfa_live_input_hop(self._lv, C.byref(delay))
            self.delay = delay.value
            self.output_hop = self._h.lib.septfa_live_output_hop(self._lv, C.byref(delay))
            self.out_delay = delay.value
            j0 = C.c_int()
            self.frames_per_hop = self._h.lib.septfa_live_vad_frames(self._lv, C.byref(j0))
            self.first_frame = j0.value
            need = self._h.lib.septfa_live_workspace_bytes(self._lv, self.capacity)
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        self.last_launch_count = 0

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def push(self, slots, hops, vad=True):
        ids = check_slots(slots, self.capacity)
        n = ids.size
        if not (isinstance(hops, torch.Tensor) and hops.is_cuda and hops.dtype == torch.float32):
            raise ValueError("hops must be a CUDA float32 tensor")
        if tuple(hops.shape) != (n, self.input_hop):
            raise ValueError(f"hops must have shape ({n}, {self.input_hop}), got {tuple(hops.shape)}")
        if hops.device != self.device:
            raise ValueError(f"hops are on {hops.device}, the session on {self.device}")
        hops = hops.contiguous()
        with torch.cuda.device(self.device):
            h = self.model._handle(self.device)
            out = torch.empty((n, 2, self.output_hop), dtype=torch.float32, device=self.device)
            v = torch.empty((n, 2, self.frames_per_hop), dtype=torch.float32, device=self.device) \
                if (vad and self.model.final_vad) else None
            perm = torch.empty((n, 2), dtype=torch.int32, device=self.device)
            rc = h.lib.septfa_live_push(self._lv, ids.ctypes.data_as(C.c_void_p), n, C.c_void_p(hops.data_ptr()),
                                        C.byref(self._kw) if self._kw is not None else None, C.c_void_p(out.data_ptr()),
                                        C.c_void_p(v.data_ptr()) if v is not None else None, C.c_void_p(perm.data_ptr()),
                                        C.c_void_p(self._ws.data_ptr()), self._ws.numel(), self._stream())
            _lib.check(h.ptr, rc)
            self.last_launch_count = h.lib.septfa_last_launch_count(h.ptr)
        return out, v, perm

    def release(self, slots):
        ids = check_slots(slots, self.capacity)
        with torch.cuda.device(self.device):
            _lib.check(self._h.ptr, self._h.lib.septfa_live_release(self._lv, ids.ctypes.data_as(C.c_void_p), ids.size,
                                                                    self._stream()))

    def close(self):
        if self._lv:
            self._h.lib.septfa_live_destroy(self._lv)
            self._lv = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
