"""Sliding-window "online" drivers (3 s window, 1 s hop by default) on top of the CUDA forward.

Reference: ``model/online_class_unknown_targets.py:9-105`` (``OnlineSaving``) and
``model/online_class_known_targets.py:9-154``. The reference re-runs the full non-causal model
on every window, keeps the last second, and fixes the speaker permutation against the
already-emitted signal with an L1 PIT (SURVEY.md section 0, D2). Here one hop of S independent
streams is one ``septfa_online_step`` call: batched forward + per-stream L1-PIT + reorder +
append, with the emitted tail kept on the device.

Deviation (documented, SURVEY.md section 3.3): the reference's ``nn.L1Loss`` reduces over the
batch too, so with B > 1 it would pick one permutation for the whole batch; it is only ever
called with B = 1. This driver decides per stream, i.e. it equals S independent reference runs.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np
import torch

from . import lib as _lib
from .live import check_geometry
from .pit import PITLossWrapper, calc_sisdr, reorder_source_mse


class OnlineSaving:
    """Drop-in for ``OnlineSaving`` (unknown targets), model/online_class_unknown_targets.py:9-105."""

    def __init__(self, model, save_path, criterion_similarity=None) -> None:
        self.indx = 0
        self.fs = 16000
        self.max_len = 3
        self.save_sec = 1
        self.model = model
        self.save_path = save_path
        self.online_sisdr = []
        self.reference_sisdr = []
        self.num_save_samples = 30
        self.similarity = False
        if criterion_similarity is not None:
            self.similarity = True
            self.criterion_similarity = criterion_similarity
            self._check_similarity_criterion(criterion_similarity)
        self.last_perms = None

    @staticmethod
    def _check_similarity_criterion(crit):
        """The stitch runs on the device as PITLossWrapper(nn.L1Loss(), pit_from='pw_pt') - the only criterion
        only_inference.py:85-86 ever passes. Anything else would silently be replaced by it, so it is refused."""
        lf = getattr(crit, "loss_func", None)
        if getattr(crit, "pit_from", None) != "pw_pt" or not isinstance(lf, torch.nn.L1Loss):
            raise NotImplementedError("septfa_b200.OnlineSaving stitches windows with PITLossWrapper(nn.L1Loss(), "
                                      "pit_from='pw_pt') on the device; other similarity criteria are not supported")

    def reset(self):
        self.indx = 0

    def get_indx(self):
        return self.indx

    def increase_indx(self):
        self.indx += 1

    def get_truncated_signal(self, full_signal_mix):
        s = int(np.floor(self.fs * self.indx * self.save_sec))
        return full_signal_mix[:, s: s + self.geometry()[0]]  # :39-41

    def geometry(self):
        """(W, H) = (fs * max_len, fs * save_sec) in samples. The device stitch takes integer windows and hops that
        ``live.check_geometry`` accepts (256 <= H, 2 H <= W <= 160000, multiples of 16); anything else raises
        ``NotImplementedError``."""
        wh = []
        for name, sec in (("max_len", self.max_len), ("save_sec", self.save_sec)):
            v = self.fs * sec
            if abs(v - round(v)) > 1e-6:
                raise NotImplementedError(f"septfa_b200.OnlineSaving: fs * {name} = {v} is not a whole number of samples")
            wh.append(int(round(v)))
        try:
            return check_geometry(*wh)
        except ValueError as e:
            raise NotImplementedError(f"septfa_b200.OnlineSaving: max_len = {self.max_len}, save_sec = {self.save_sec}: "
                                      f"{e}") from None

    # -- wav dumps (host I/O, batch item 0 like the reference) ------------------------------
    def save_audio(self, name_folder, separated_signals, mix):
        from scipy.io.wavfile import write
        d = Path(f"{self.save_path}/{name_folder}/indx_{self.indx}")
        d.mkdir(parents=True, exist_ok=True)
        write(str(d / "mixed.wav"), self.fs, mix[0].detach().cpu().numpy().astype(np.float32))
        write(str(d / "output_0.wav"), self.fs, separated_signals[0, 0].detach().cpu().numpy().astype(np.float32))
        write(str(d / "output_1.wav"), self.fs, separated_signals[0, 1].detach().cpu().numpy().astype(np.float32))

    def save_last_online_audio(self, name_folder, online_signal, mixed_signal_t):
        from scipy.io.wavfile import write
        d = Path(f"{self.save_path}/{name_folder}")
        d.mkdir(parents=True, exist_ok=True)
        sig = online_signal[0].detach().cpu().numpy()
        write(str(d / "online_signal0.wav"), self.fs, sig[0].astype(np.float32))
        write(str(d / "online_signal1.wav"), self.fs, sig[1].astype(np.float32))
        write(str(d / "ref_mix.wav"), self.fs, mixed_signal_t[0].detach().cpu().numpy().astype(np.float32))

    # -- the driver --------------------------------------------------------------------------
    def calc_online(self, full_signal_mix, name_folder, sample_indx, inference_kw):
        """model/online_class_unknown_targets.py:72-105. ``full_signal_mix`` [S, L] on a CUDA device."""
        if not full_signal_mix.is_cuda:
            raise RuntimeError("septfa_b200.OnlineSaving runs on CUDA only (no CPU fallback)")
        win_len, hop = self.geometry()
        x = full_signal_mix.detach().float()
        if x.shape[-1] < win_len:                                                             # :73-74
            x = torch.nn.functional.pad(x, (0, win_len - x.shape[-1]))
        max_indx = np.floor((x.shape[-1] - self.fs * self.max_len) / (self.fs * self.save_sec))  # :77
        S = x.shape[0]
        dev = x.device
        kw = _lib.InferKw.from_dict(inference_kw) if (inference_kw and self.model.final_vad) else None
        with torch.cuda.device(dev):
            h = self.model._handle(dev)
            st = C.c_void_p()
            _lib.check(h.ptr, h.lib.septfa_online_create_win(h.ptr, S, win_len, hop, C.byref(st)))
            try:
                need = h.lib.septfa_online_workspace_bytes(st)
                ws = torch.empty(need, dtype=torch.uint8, device=dev)
                n_hops = int(max_indx) + 1
                online = torch.empty((S, 2, hop * n_hops), dtype=torch.float32, device=dev)
                perms = torch.empty((n_hops, S, 2), dtype=torch.int32, device=dev)
                stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                while self.indx <= max_indx:                                                  # :80
                    win = self.get_truncated_signal(x).contiguous()
                    emitted = torch.empty((S, 2, hop), dtype=torch.float32, device=dev)
                    rc = h.lib.septfa_online_step(st, C.c_void_p(win.data_ptr()), C.byref(kw) if kw is not None else None,
                                                  C.c_void_p(emitted.data_ptr()), C.c_void_p(perms[self.indx].data_ptr()),
                                                  C.c_void_p(ws.data_ptr()), ws.numel(), stream)
                    _lib.check(h.ptr, rc)
                    online[:, :, self.indx * hop:(self.indx + 1) * hop] = emitted              # :94 (cat)
                    if sample_indx < self.num_save_samples:                                   # :95-96
                        # per-window dumps of batch item 0: the model's window output (first tensor of the online
                        # workspace, [S, 2, W]) reordered by this hop's permutation, and the window of the mixture
                        base = (ws.data_ptr() + 255) // 256 * 256 - ws.data_ptr()
                        pred0 = ws[base: base + 2 * win_len * 4].view(torch.float32).view(1, 2, -1)
                        pred0 = pred0[:, perms[self.indx][0].long()]
                        self.save_audio(name_folder, pred0, win)
                    self.increase_indx()
                torch.cuda.current_stream(dev).synchronize()
            finally:
                h.lib.septfa_online_destroy(st)
        self.online_signal = online
        self.last_perms = perms
        a = int(np.floor(self.fs * (self.max_len - self.save_sec)))
        b = int(np.floor(self.fs * (self.max_len + (self.indx - 1) * self.save_sec)))
        mixed_signal_t = x[:, a:b]                                                            # :100
        if sample_indx < self.num_save_samples:
            self.save_last_online_audio(name_folder, self.online_signal, mixed_signal_t)      # :102-103
        self.reset()                                                                          # :105
        return self.online_signal


class OnlineSavingKnownTargets(OnlineSaving):
    """``OnlineSaving`` of model/online_class_known_targets.py:9-154 (ground-truth targets available).

    The reference file is stale (it unpacks six return values from a forward that returns three,
    :105,126); this class implements its *intended* behaviour against the current 3-tuple forward:
    left-pad 2 s (:92-93), tail-pad to whole hops (:94-97), per-window PIT against the true
    sources when no similarity criterion is given, SI-SDR of the stitched signal vs the full-length
    ("reference") pass (:126-145).
    """

    def __init__(self, criterion_separation, model, save_path, device=None, criterion_similarity=None) -> None:
        # argument order of the reference's constructor (model/online_class_known_targets.py:10); `device` is accepted
        # and ignored there too (the tensors decide)
        super().__init__(model, save_path, criterion_similarity)
        self.criterion_separation = criterion_separation
        self.num_save_samples = 2000000                                                       # :20

    def calc_online(self, full_signal_mix, target_signal, name_folder, sample_indx, inference_kw=None):
        """model/online_class_known_targets.py:85-154 (which calls the model without inference_kw: the default here)."""
        inference_kw = inference_kw or {}
        x = full_signal_mix.detach().float()
        tgt = target_signal.detach().float()
        fs, ml, ss = self.fs, self.max_len, self.save_sec
        if x.shape[-1] < fs * ml:                                                             # :86-88
            x = torch.nn.functional.pad(x, (0, fs * ml - x.shape[-1]))
            tgt = torch.nn.functional.pad(tgt, (0, fs * ml - tgt.shape[-1]))
        x = torch.nn.functional.pad(x, (int(fs * (ml - ss)), 0))                              # :92
        tgt = torch.nn.functional.pad(tgt, (int(fs * (ml - ss)), 0))                          # :93
        pad_zero = (x.shape[-1] - fs * ml) % (fs * ss)                                        # :94
        if pad_zero:
            x = torch.nn.functional.pad(x, (0, pad_zero))
            tgt = torch.nn.functional.pad(tgt, (0, pad_zero))
        if self.similarity:
            # same stitching as the unknown-target driver (:110-119)
            saved = self.num_save_samples
            self.num_save_samples = 0
            online = OnlineSaving.calc_online(self, x, name_folder, sample_indx, inference_kw)
            self.num_save_samples = saved
            n_hops = online.shape[-1] // int(fs * ss)
        else:
            # per-window PIT against the true sources (:106-107,120-121)
            max_indx = int(np.floor((x.shape[-1] - fs * ml) / (fs * ss)))
            chunks = []
            for indx in range(max_indx + 1):
                s = int(fs * indx * ss)
                with torch.no_grad():
                    pred, _, _ = self.model(x[:, s:s + ml * fs].contiguous(), inference_kw)
                _, idx = self.criterion_separation(pred, tgt[:, :, s:s + ml * fs], return_incides=True)
                pred = reorder_source_mse(pred, idx)
                chunks.append(pred[:, :, pred.shape[-1] - int(fs * ss):])
            online = torch.cat(chunks, dim=-1)
            n_hops = max_indx + 1
        a = int(np.floor(fs * (ml - ss)))
        b = int(np.floor(fs * (ml + (n_hops - 1) * ss)))
        # reference score: full-length pass (:126-134)
        with torch.no_grad():
            pred_full, _, _ = self.model(x, inference_kw)
        _, idx = self.criterion_separation(pred_full, tgt, return_incides=True)
        pred_full = reorder_source_mse(pred_full, idx)
        self.reference_sisdr.append(torch.mean(calc_sisdr(pred_full[:, :, a:b], tgt[:, :, a:b])).item())
        # online score (:137-145)
        true_t = tgt[:, :, a:b]
        _, idx = self.criterion_separation(online, true_t, return_incides=True)
        self.online_signal = reorder_source_mse(online, idx)
        self.online_sisdr.append(torch.mean(calc_sisdr(self.online_signal, true_t)).item())
        self.reset()
        return self.online_signal
