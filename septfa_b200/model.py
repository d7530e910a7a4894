"""Drop-in ``SeparationModel`` (reference: model/model.py:360-461) backed by libseptfa.so.

Same constructor (``SeparationModel(**config["arch"]["args"])``), same ``state_dict`` keys and
shapes (so the reference ``.pth`` checkpoints load with ``strict=True``), same
``forward(x, inference_kw={})`` return tuple and the same side-effect attributes
(``mask_per_speaker``, ``spectrum``, ``masks_b``, ``estimated_stfts``). The arithmetic runs in
the hand-written CUDA kernels behind the C ABI of ``include/septfa.h``; this class only owns
torch tensors (parameters, inputs, outputs, workspace) and passes raw device pointers plus the
current CUDA stream. There is no CPU path: inputs must live on a CUDA device.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import lib as _lib
from . import synth as _synth

_DEFAULTS = {  # model/model.py:362-366
    'n_fftBins': 512, 'BN_dim': 256, 'H_dim': 512, 'layer': 8, 'stack': 3, 'kernel': 3,
    'num_spk': 2, 'skip': False, 'dilated': True, 'casual': False, 'bool_drop': True,
    'drop_value': 0.1, 'weight_norm': False, 'final_vad': True, 'noisy_phase': False,
    'activity_input_bool': False, 'tf_attention': False, 'apply_recursive_ln': False,
    'apply_residual_ln': False, 'final_vad_masked_speakers': False}


def _attach(root: nn.Module, dotted: str, tensor: torch.Tensor, buffer: bool):
    """Register ``tensor`` under a dotted state_dict key, creating bare container modules."""
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, nn.Module())
        mod = mod._modules[p]
    if buffer:
        mod.register_buffer(parts[-1], tensor)
    else:
        mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


class _Handle:
    """One septfa_handle per CUDA device, with its weights committed."""

    def __init__(self, cfg: "_lib.Config", device_index: int):
        self.lib = _lib.load()
        self.ptr = C.c_void_p()
        rc = self.lib.septfa_create(C.byref(self.ptr), C.byref(cfg), device_index)
        if rc != 0:
            msg = self.lib.septfa_last_error(None)
            raise _lib.SeptfaError(f"septfa_create failed ({rc}): {msg.decode() if msg else ''}")
        self.version = -1
        self.workspace = None
        self.device_index = device_index

    def keys(self):
        n = self.lib.septfa_num_keys(self.ptr)
        return [(self.lib.septfa_key_name(self.ptr, i).decode(), self.lib.septfa_key_numel(self.ptr, i)) for i in range(n)]

    def __del__(self):
        try:
            if self.ptr:
                self.lib.septfa_destroy(self.ptr)
                self.ptr = None
        except Exception:
            pass


class SeparationModel(nn.Module):
    def __init__(self, **config):
        super().__init__()
        defaults = dict(_DEFAULTS)
        defaults.update(config)
        print(defaults)  # the reference prints the merged dict (model/model.py:371)
        for key, value in defaults.items():
            setattr(self, key, value)
        self._args = defaults
        self.n_fftBins_h = self.n_fftBins // 2 + 1
        # unsupported-at-these-configs branches fail loudly (SURVEY.md section 8a)
        if not self.weight_norm or self.skip or self.casual or not self.dilated or self.final_vad_masked_speakers:
            raise NotImplementedError(
                "septfa_b200 implements the shipped configurations only: weight_norm=True, skip=False, "
                "casual=False, dilated=True, final_vad_masked_speakers=False")
        if (self.n_fftBins, self.BN_dim, self.H_dim, self.num_spk) != (512, 256, 512, 2):
            raise NotImplementedError("septfa_b200 needs n_fftBins=512, BN_dim=256, H_dim=512, num_spk=2")
        # parameters / buffers with the reference's names and shapes (random init like a fresh reference module)
        seed = int(torch.initial_seed()) & 0x7FFFFFFF
        for k, v in _synth.make_state_dict(defaults, seed).items():
            _attach(self, k, v.clone(), buffer=k.endswith("window"))
        self._handles = {}
        self._weights_version = 0
        #: which optional outputs forward() materialises (all on = the reference's behaviour)
        self.materialize = {"estimated_stfts": True, "mask_per_speaker": True, "spectrum": True, "masks_b": True}
        self.engine = _lib.ENGINE_TCGEN05_F16
        self.last_launch_count = 0
        # Opt-in guard (costs a device reduction and a host sync per forward): raise if a forward returns non-finite
        # samples. In the fast mode p and racc travel between the block kernels as fp16 (|x| <= 65504): a checkpoint with
        # extreme weight_g could overflow there; set_option("precision", 2) keeps them in fp32.
        self.check_finite = False

    # -- weights ---------------------------------------------------------------------------
    def load_state_dict(self, state_dict, strict=True, **kw):
        out = super().load_state_dict(state_dict, strict=strict, **kw)
        self._weights_version += 1
        return out

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._weights_version += 1
        return out

    def refresh_weights(self):
        """Call after mutating parameters in place (the CUDA side keeps packed copies)."""
        self._weights_version += 1

    def set_engine(self, engine):
        self.engine = int(engine)

    def set_option(self, name, value):
        """Forwarded to septfa_set_option (e.g. "precision", "host_chunks", "dconv_mma"; include/septfa.h lists them).
        A name or value the library refuses raises SeptfaError (at once, or at the first call on a device without a
        handle yet) and is not kept, so the model stays usable."""
        for h in self._handles.values():
            _lib.check(h.ptr, h.lib.septfa_set_option(h.ptr, name.encode(), int(value)))
        if not hasattr(self, "_options"):
            self._options = {}
        self._options[name] = int(value)

    def set_profile(self, on: bool):
        """Per-kernel-class CUDA-event timing inside forward (septfa_set_option "profile")."""
        self._profile = bool(on)

    def read_profile(self, device=None, reset=True):
        """{class name: (milliseconds, intervals)} accumulated since the last reset."""
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        h = self._handle(dev)
        ms = (C.c_double * 16)()
        cnt = (C.c_int * 16)()
        _lib.check(h.ptr, h.lib.septfa_profile_read(h.ptr, ms, cnt, 16, int(reset)))
        return {n: (ms[i], cnt[i]) for i, n in enumerate(_lib.PROF_NAMES)}

    def _handle(self, device: torch.device) -> _Handle:
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._handles.get(idx)
        if h is None:
            h = _Handle(_lib.Config.from_args(self._args), idx)
            self._handles[idx] = h
        if h.version != self._weights_version:
            sd = super().state_dict()
            for name, numel in h.keys():
                t = sd[name].detach().to("cpu", torch.float32).contiguous()
                if t.numel() != numel:
                    raise _lib.SeptfaError(f"size mismatch for {name}")
                _lib.check(h.ptr, h.lib.septfa_set_tensor(h.ptr, name.encode(), C.c_void_p(t.data_ptr()), numel))
            _lib.check(h.ptr, h.lib.septfa_commit_weights(h.ptr))
            h.version = self._weights_version
        _lib.check(h.ptr, h.lib.septfa_set_option(h.ptr, b"engine", self.engine))
        _lib.check(h.ptr, h.lib.septfa_set_option(h.ptr, b"profile", int(getattr(self, "_profile", False))))
        for name, value in list(getattr(self, "_options", {}).items()):
            rc = h.lib.septfa_set_option(h.ptr, name.encode(), int(value))
            if rc != 0:
                del self._options[name]
                _lib.check(h.ptr, rc)
        return h

    # -- forward ---------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, inference_kw={}):
        """x - 2-speaker mixed signal, shape = [B, T]  (model/model.py:402-461)"""
        assert x.ndim == 2, "input tensor must be 2 dimensions (B, T), but got dimensions of {}".format(x.ndim)
        if not x.is_cuda:
            raise RuntimeError("septfa_b200.SeparationModel runs on CUDA (sm_100a) only: move the input to a B200 "
                               "(there is no CPU fallback)")
        kw = _lib.InferKw.from_dict(inference_kw) if (inference_kw and self.final_vad) else None
        x = x.detach().to(torch.float32).contiguous()
        B, L = x.shape
        T = _lib.num_frames(L)
        dev = x.device
        with torch.cuda.device(dev):
            h = self._handle(dev)
            need = h.lib.septfa_workspace_bytes(h.ptr, B, L)
            if need == 0:
                raise _lib.SeptfaError(f"unsupported input shape B={B}, L={L} (need L >= 257)")
            if h.workspace is None or h.workspace.numel() < need:
                h.workspace = None
                h.workspace = torch.empty(need, dtype=torch.uint8, device=dev)
            out = torch.empty((B, self.num_spk, L), dtype=torch.float32, device=dev)
            vad = torch.empty((B, self.num_spk, T), dtype=torch.float32, device=dev) if self.final_vad else None
            m = self.materialize
            est = torch.empty((B, self.num_spk, self.n_fftBins_h, T, 2), dtype=torch.float32, device=dev) \
                if m["estimated_stfts"] else None
            mask = torch.empty((B, self.num_spk, self.n_fftBins_h, T), dtype=torch.float32, device=dev) \
                if m["mask_per_speaker"] else None
            spec = torch.empty((B, self.n_fftBins_h, T), dtype=torch.float32, device=dev) if m["spectrum"] else None
            logits = torch.empty((B, self.n_fftBins_h * self.num_spk, T), dtype=torch.float32, device=dev) \
                if m["masks_b"] else None
            p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            rc = h.lib.septfa_forward(h.ptr, p(x), B, L, C.byref(kw) if kw is not None else None, p(out), p(vad),
                                      p(est), p(mask), p(spec), p(logits), p(h.workspace), h.workspace.numel(), stream)
            _lib.check(h.ptr, rc)
            self.last_launch_count = h.lib.septfa_last_launch_count(h.ptr)
            if self.check_finite and not bool(torch.isfinite(out).all()):
                raise RuntimeError("septfa_b200: the forward returned non-finite samples - a non-finite or constant input, or "
                                   "half-precision overflow of the tensors between the block kernels (extreme weight_g): "
                                   "try model.set_option('precision', 2)")
        self.spectrum = spec
        self.masks_b = logits
        self.mask_per_speaker = mask
        self.estimated_stfts = torch.view_as_complex(est) if est is not None else None
        if not self.final_vad:
            output_vad = 0                                    # model/model.py:426-427
        elif kw is not None and kw.return_smoothed_vad:
            output_vad = vad.unsqueeze(2)                     # [B, 2, 1, T], model/model.py:449-457
        else:
            output_vad = vad
        return out, output_vad, self.estimated_stfts

    def graphed(self, B, L, inference_kw={}, device=None):
        """The forward for one (B, L, inference_kw) as a replayable CUDA graph (septfa_graph_capture): for serving many
        small requests, where ~80 kernel launches of a few microseconds each dominate (launch-bound). Returns a
        :class:`GraphedForward`; ``g(x)`` copies ``x [B, L]`` into the graph's static input, replays the graph on the
        current stream and returns ``(out_separation, output_vad)`` - static tensors, overwritten by the next call."""
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        return GraphedForward(self, int(B), int(L), inference_kw, dev)

    def forward_host(self, x_host: torch.Tensor, inference_kw={}, device=0, pin_outputs=True):
        """End-to-end call with HOST tensors: septfa_forward_host does the H2D copy, the forward and
        the D2H copy of (out_separation, output_vad) through pinned staging buffers."""
        assert x_host.ndim == 2 and not x_host.is_cuda
        kw = _lib.InferKw.from_dict(inference_kw) if (inference_kw and self.final_vad) else None
        x_host = x_host.detach().to(torch.float32).contiguous()
        B, L = x_host.shape
        T = _lib.num_frames(L)
        dev = torch.device("cuda", device)
        with torch.cuda.device(dev):
            h = self._handle(dev)
            # page-locked result buffers (copied into directly by the library); pass pin_outputs=False for pageable
            pin = bool(pin_outputs)
            out = torch.empty((B, self.num_spk, L), dtype=torch.float32, pin_memory=pin)
            vad = torch.empty((B, self.num_spk, T), dtype=torch.float32, pin_memory=pin) if self.final_vad else None
            rc = h.lib.septfa_forward_host(h.ptr, C.c_void_p(x_host.data_ptr()), B, L,
                                           C.byref(kw) if kw is not None else None, C.c_void_p(out.data_ptr()),
                                           C.c_void_p(vad.data_ptr()) if vad is not None else None)
            _lib.check(h.ptr, rc)
            self.last_launch_count = h.lib.septfa_last_launch_count(h.ptr)
        return self._host_result(out, vad, kw)

    def _host_result(self, out, vad, kw):
        if not self.final_vad:
            return out, 0
        if kw is not None and kw.return_smoothed_vad:
            return out, vad.unsqueeze(2)
        return out, vad

    def minmax_normalize(self, x: torch.Tensor, lengths=None):
        """only_inference.py:81 on the device, batched: ``1.8 * (x - x.min()) / (x.max() - x.min()) - 0.9`` per
        utterance of ``x [B, L]`` (float32 CUDA), bit-identical to the reference's numpy expression. ``lengths``
        (optional int64 ``[B]``): valid samples per utterance of a zero-padded ragged batch."""
        assert x.ndim == 2 and x.is_cuda and x.dtype == torch.float32
        x = x.contiguous()
        out = torch.empty_like(x)
        if lengths is not None:
            lengths = torch.as_tensor(lengths, dtype=torch.int64, device=x.device).contiguous()
            assert lengths.numel() == x.shape[0]
        with torch.cuda.device(x.device):
            h = self._handle(x.device)
            rc = h.lib.septfa_minmax_normalize(h.ptr, C.c_void_p(x.data_ptr()), x.shape[0], x.shape[1],
                                               C.c_void_p(lengths.data_ptr()) if lengths is not None else None,
                                               C.c_void_p(out.data_ptr()),
                                               C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
            _lib.check(h.ptr, rc)
        return out

    def resample(self, x: torch.Tensor, rate):
        """torchaudio.functional.resample(x, rate, 16000) on the device (septfa_resample), batched: ``x [B, L]`` is a CUDA
        float32 tensor, or int16 PCM converted as ``astype(float32)`` (no scaling); returns float32
        ``[B, ceil(16000 L / rate)]``. ``rate``: an integer in 8000 .. 192000 Hz; 16000 returns the input values."""
        assert x.ndim == 2 and x.is_cuda and x.dtype in (torch.float32, torch.int16)
        if isinstance(rate, bool) or int(rate) != rate:
            raise ValueError(f"rate must be an integer number of Hz, got {rate!r}")
        rate = int(rate)
        x = x.contiguous()
        B, L = x.shape
        x_fmt = _lib.FMT_PCM16 if x.dtype == torch.int16 else _lib.FMT_F32
        out = torch.empty((B, max(-(-16000 * L // rate), 0) if rate > 0 else 0), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            h = self._handle(x.device)
            rc = h.lib.septfa_resample(h.ptr, C.c_void_p(x.data_ptr()), x_fmt, B, L, rate, C.c_void_p(out.data_ptr()),
                                       C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))
            _lib.check(h.ptr, rc)
            self.last_launch_count = h.lib.septfa_last_launch_count(h.ptr)
        return out

    def resample_to(self, y: torch.Tensor, rate):
        """torchaudio.functional.resample(y, 16000, rate) on the device (septfa_resample_to): the model's 16 kHz output
        back at ``rate``. ``y [..., L]`` is a CUDA float32 tensor whose leading dimensions are resampled as rows (a
        forward's ``[B, 2, L]`` goes in directly); returns float32 ``[..., ceil(rate L / 16000)]``. ``rate``: an integer
        in 8000 .. 192000 Hz; 16000 returns the input values."""
        assert y.ndim >= 1 and y.is_cuda and y.dtype == torch.float32
        if isinstance(rate, bool) or int(rate) != rate:
            raise ValueError(f"rate must be an integer number of Hz, got {rate!r}")
        rate = int(rate)
        y = y.contiguous()
        L = y.shape[-1]
        rows = y.numel() // L if L else 0
        out = torch.empty((*y.shape[:-1], max(-(-rate * L // 16000), 0) if rate > 0 else 0), dtype=torch.float32,
                          device=y.device)
        with torch.cuda.device(y.device):
            h = self._handle(y.device)
            rc = h.lib.septfa_resample_to(h.ptr, C.c_void_p(y.data_ptr()), rows, L, rate, C.c_void_p(out.data_ptr()),
                                          C.c_void_p(torch.cuda.current_stream(y.device).cuda_stream))
            _lib.check(h.ptr, rc)
            self.last_launch_count = h.lib.septfa_last_launch_count(h.ptr)
        return out

    def forward_host_submit(self, x_host: torch.Tensor, inference_kw={}, device=0, slot=0, out=None, vad=None,
                            out_dtype=torch.float32):
        """Asynchronous half of :meth:`forward_host` (septfa_forward_host_submit_fmt): enqueue copy-in, forward and
        copy-out of one batch on a pipeline slot (0 .. 3) and return a :class:`HostBatch` whose ``result()`` waits for
        it. Slots in rotation (three keep the pipeline full) let successive batches overlap their PCIe copies with each
        other's kernels. ``x_host`` is
        pinned if it is not already; ``out`` / ``vad`` may be caller-provided pinned result tensors (reused across
        batches), otherwise fresh pinned tensors are allocated.

        16-bit host formats halve the PCIe bytes: an ``int16`` ``x_host`` is PCM as ``scipy.io.wavfile.read`` returns
        it - the device then does only_inference.py:69,81 (``astype(float32)``, min-max normalise to +-0.9) before the
        forward; ``out_dtype=torch.float16`` returns the waveforms as the ``-ps 16`` format of ``save_audio``
        (Our_utils/utlis_inference.py:30-32)."""
        assert x_host.ndim == 2 and not x_host.is_cuda
        kw = _lib.InferKw.from_dict(inference_kw) if (inference_kw and self.final_vad) else None
        if x_host.dtype == torch.int16:
            x_fmt = _lib.FMT_PCM16
            x_host = x_host.detach().contiguous()
        else:
            x_fmt = _lib.FMT_F32
            x_host = x_host.detach().to(torch.float32).contiguous()
        if out_dtype not in (torch.float32, torch.float16):
            raise ValueError("out_dtype must be torch.float32 or torch.float16")
        out_fmt = _lib.FMT_F16 if out_dtype == torch.float16 else _lib.FMT_F32
        if not x_host.is_pinned():
            x_host = x_host.pin_memory()
        B, L = x_host.shape
        T = _lib.num_frames(L)
        dev = torch.device("cuda", device)
        with torch.cuda.device(dev):
            h = self._handle(dev)
            if out is None:
                out = torch.empty((B, self.num_spk, L), dtype=out_dtype, pin_memory=True)
            if vad is None and self.final_vad:
                vad = torch.empty((B, self.num_spk, T), dtype=torch.float32, pin_memory=True)
            assert tuple(out.shape) == (B, self.num_spk, L) and out.is_pinned() and out.is_contiguous() and out.dtype == out_dtype
            rc = h.lib.septfa_forward_host_submit_fmt(h.ptr, int(slot), C.c_void_p(x_host.data_ptr()), x_fmt, B, L,
                                                      C.byref(kw) if kw is not None else None, C.c_void_p(out.data_ptr()),
                                                      out_fmt, C.c_void_p(vad.data_ptr()) if vad is not None else None)
            _lib.check(h.ptr, rc)
            self.last_launch_count = h.lib.septfa_last_launch_count(h.ptr)
        return HostBatch(self, h, dev, int(slot), x_host, out, vad if self.final_vad else None, kw)

    def forward_host_stream(self, batches, inference_kw={}, device=0, out_dtype=torch.float32, reuse_outputs=False):
        """Generator over an iterable of host batches ``[B, L]`` (the loop of only_inference.py:80-100 over a data
        loader): yields ``(out_separation, output_vad)`` per batch, in order, keeping three batches in flight. Batches
        may be float32 (normalised) or int16 PCM; ``out_dtype`` as in :meth:`forward_host_submit`.
        ``reuse_outputs=True`` recycles five sets of pinned result buffers instead of page-locking fresh memory for
        every batch (cudaHostAlloc of 130 MB costs more than the batch's forward): a yielded result then stays valid
        until TWO further results have been yielded - enough for a loop that writes each result out before asking for
        the next."""
        pending = []
        # pinned result sets are kept on the module between calls (page-locking 130 MB costs ~15 ms: more than four forwards)
        pool = self.__dict__.setdefault("_host_result_pool", {})
        depth = 3   # batches in flight (pipeline slots in rotation): see include/septfa.h

        def buffers(i, xb):
            if not reuse_outputs:
                return None, None
            B, L = xb.shape
            key = (B, L, str(out_dtype), i % (depth + 2))
            if key not in pool:
                pool[key] = (torch.empty((B, self.num_spk, L), dtype=out_dtype, pin_memory=True),
                             torch.empty((B, self.num_spk, _lib.num_frames(L)), dtype=torch.float32, pin_memory=True)
                             if self.final_vad else None)
            return pool[key]

        for i, xb in enumerate(batches):
            if len(pending) == depth:
                yield pending.pop(0).result()
            o, v = buffers(i, xb)
            pending.append(self.forward_host_submit(xb, inference_kw, device, slot=i % depth, out=o, vad=v, out_dtype=out_dtype))
        while pending:
            yield pending.pop(0).result()


class GraphedForward:
    """A captured forward (see :meth:`SeparationModel.graphed`). Owns its static device buffers."""

    def __init__(self, model, B, L, inference_kw, dev):
        self._m, self.B, self.L, self._dev = model, B, L, dev
        self._kw = _lib.InferKw.from_dict(inference_kw) if (inference_kw and model.final_vad) else None
        T = _lib.num_frames(L)
        with torch.cuda.device(dev):
            h = model._handle(dev)
            self._h = h
            need = h.lib.septfa_workspace_bytes(h.ptr, B, L)
            if need == 0:
                raise _lib.SeptfaError(f"unsupported input shape B={B}, L={L} (need L >= 257)")
            self.x = torch.zeros((B, L), dtype=torch.float32, device=dev)
            self.out = torch.empty((B, model.num_spk, L), dtype=torch.float32, device=dev)
            self.vad = torch.empty((B, model.num_spk, T), dtype=torch.float32, device=dev)
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
            self._g = C.c_void_p()
            torch.cuda.synchronize(dev)
            rc = h.lib.septfa_graph_capture(h.ptr, C.c_void_p(self.x.data_ptr()), B, L,
                                            C.byref(self._kw) if self._kw is not None else None,
                                            C.c_void_p(self.out.data_ptr()), C.c_void_p(self.vad.data_ptr()),
                                            C.c_void_p(self._ws.data_ptr()), self._ws.numel(), C.byref(self._g))
            _lib.check(h.ptr, rc)
            self.num_nodes = h.lib.septfa_graph_num_nodes(self._g)

    def replay(self):
        """Replay on the current stream with whatever ``self.x`` holds."""
        with torch.cuda.device(self._dev):
            _lib.check(self._h.ptr, self._h.lib.septfa_graph_launch(self._g, C.c_void_p(torch.cuda.current_stream(self._dev).cuda_stream)))
        return self._m._host_result(self.out, self.vad, self._kw)

    def __call__(self, x):
        assert tuple(x.shape) == (self.B, self.L)
        self.x.copy_(x, non_blocking=True)
        return self.replay()

    def __del__(self):
        try:
            if self._g:
                self._h.lib.septfa_graph_destroy(self._g)
                self._g = None
        except Exception:
            pass


class HostBatch:
    """A batch in flight on one pipeline slot (returned by :meth:`SeparationModel.forward_host_submit`)."""

    def __init__(self, model, handle, dev, slot, x_host, out, vad, kw):
        self._m, self._h, self._dev, self.slot = model, handle, dev, slot
        self._x, self._out, self._vad, self._kw = x_host, out, vad, kw   # keeps the pinned buffers alive
        self._done = False

    def result(self):
        if not self._done:
            with torch.cuda.device(self._dev):
                _lib.check(self._h.ptr, self._h.lib.septfa_forward_host_wait(self._h.ptr, self.slot))
            self._done = True
        return self._m._host_result(self._out, self._vad, self._kw)
