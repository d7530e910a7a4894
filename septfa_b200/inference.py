"""``only_inference.py`` with the CUDA model: same flags, same pre/post-processing.

Reference: ``only_inference.py:27-137`` and ``Our_utils/utlis_inference.py:9-46``.

    python -m septfa_b200.inference -c config_with_vad.json -r model_with_vad.pth -pm mix.wav \
        -sp results -ikw '{"filter_signals_by_smo_vad": true}'

Differences, all host-side: the model and the audio are moved to the CUDA device selected by
``-d`` (the reference script never leaves the CPU); ``-ps 16`` writes 16-bit PCM (the reference
hands float16 to scipy, which raises); mask PNGs are written only if matplotlib is importable.
The run-directory / logging side effects of ``parse_config.ConfigParser`` are not reproduced.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
from pathlib import Path

import numpy as np
import torch

from .model import SeparationModel
from .online import OnlineSaving
from .pit import PITLossWrapper
from .synth import DEFAULT_INFERENCE_KW


def parse_dictionary(dictionary_string):
    """only_inference.py:17-23."""
    try:
        return json.loads(dictionary_string)
    except json.JSONDecodeError as e:
        raise argparse.ArgumentTypeError(f"Invalid dictionary provided: {dictionary_string}. Error: {e}")


def load_checkpoint_state_dict(path):
    """only_inference.py:57-58: ``torch.load(resume, map_location='cpu')['state_dict']``. Checkpoints
    written by base/base_trainer.py:164-171 may hold numpy scalars (``monitor_best``), which
    torch >= 2.6 refuses under weights_only=True - fall back like the reference's torch did."""
    try:
        ckpt = torch.load(path, map_location="cpu")
    except Exception:
        ckpt = torch.load(path, map_location="cpu", weights_only=False)
    return ckpt["state_dict"]


def read_mixture(path_audio):
    """only_inference.py:68-83: wav -> float32 mono @16 kHz -> min-max normalised to [-0.9, 0.9], shape [1, L]."""
    from scipy.io.wavfile import read
    samplerate, audio = read(path_audio)
    audio = np.array(audio, dtype=np.float32)
    if audio.ndim > 1:
        print("The audio is not mono, the first channel was chosen")
        audio = audio[0] if audio.shape[1] > audio.shape[0] else audio[:, 0]
    if samplerate != 16000:
        print("The audio is not 16KHz, resmapling to 16KHz..")
        try:
            import torchaudio.transforms as T
            audio = T.Resample(samplerate, 16000, dtype=torch.float32)(torch.tensor(audio)).numpy()
        except ImportError:
            from math import gcd
            from scipy.signal import resample_poly
            g = gcd(int(samplerate), 16000)
            audio = resample_poly(audio, 16000 // g, int(samplerate) // g).astype(np.float32)
    normalized = 1.8 * (audio - audio.min()) / (audio.max() - audio.min()) - 0.9             # :81
    return torch.from_numpy(np.asarray(normalized, dtype=np.float32)).unsqueeze(0)


def save_audio(mix_waves, separated_signals, save_path, bit16):
    """Our_utils/utlis_inference.py:24-37 (batch item 0)."""
    from scipy.io.wavfile import write
    Path(save_path).mkdir(parents=True, exist_ok=True)
    sigs = {"Mixed_0.wav": mix_waves[0], "Speaker_0.wav": separated_signals[0, 0], "Speaker_1.wav": separated_signals[0, 1]}
    for name, t in sigs.items():
        a = t.detach().cpu().numpy().astype(np.float32)
        if bit16 == 16:
            a = np.clip(np.round(a * 32767.0), -32768, 32767).astype(np.int16)
        write(os.path.join(save_path, name), 16000, a)


def _pyplot():
    """matplotlib.pyplot with the Agg backend, or None when matplotlib is absent (or only a stub module is importable)."""
    try:
        import matplotlib
        matplotlib.use("Agg")
        import matplotlib.pyplot as plt
        return plt if hasattr(plt, "subplots") else None
    except (ImportError, AttributeError):
        return None


def plot_spectrogram(masks, title, save_path):
    """Our_utils/utlis_inference.py:9-22; skipped (with a note) when matplotlib is unavailable."""
    plt = _pyplot()
    if plt is None:
        print("matplotlib not available: mask PNGs not written")
        return
    masks = masks.cpu()
    for i in range(masks.shape[1]):
        fig, axs = plt.subplots(1, 1)
        axs.set_title(f"Spectrogram (db) - {title}")
        axs.set_ylabel("freq_bin")
        axs.set_xlabel("frame")
        im = axs.imshow(masks[0, i].detach().numpy(), origin="lower", aspect="auto")
        fig.colorbar(im, ax=axs)
        Path(save_path).mkdir(parents=True, exist_ok=True)
        plt.savefig(Path(save_path).joinpath(f"Mask_Speaker_{i}"))
        plt.close("all")


def save_vad(vad_output, save_path):
    """Our_utils/utlis_inference.py:39-46: the decisions ``p >= 0.5`` of batch item 0, one figure per speaker
    (``estimated_vad_{spk}.png``). Without matplotlib the decisions are written as ``estimated_vad_{spk}.npy``."""
    Path(save_path).mkdir(parents=True, exist_ok=True)
    vad_output = vad_output.detach().cpu()
    if vad_output.ndim == 4:            # [B, 2, 1, T] when return_smoothed_vad
        vad_output = vad_output[:, :, 0]
    plt = _pyplot()
    for spk in range(vad_output.shape[1]):
        est_vad = torch.where(vad_output[0, spk] >= 0.5, 1, 0)
        if plt is None:
            np.save(os.path.join(save_path, f"estimated_vad_{spk}.npy"), est_vad.numpy())
        else:
            plt.plot(est_vad)
            plt.savefig(os.path.join(save_path, f"estimated_vad_{spk}.png"))
            plt.close()


def _first_channel(audio):
    """read_mixture's channel choice (only_inference.py:70-72)."""
    return audio[0] if audio.shape[1] > audio.shape[0] else audio[:, 0]


def separate_files(model, paths, save_dir, inference_kw=None, precision_save=32, device=0, batch=64, out_rate=None):
    """The file loop either side of the forward (SURVEY.md section 8(f) rank 1), batched: 16-bit wav files of EQUAL
    length and rate are grouped into batches. 16 kHz mono batches travel to the device as int16 PCM, are converted and
    min-max normalised there (only_inference.py:69,81, bit-identical to numpy), separated, and come back as float32 or -
    for ``precision_save=16`` - float16, three batches in flight (forward_host_stream). 16-bit files at another rate in
    8 .. 192 kHz, and 16-bit stereo files at 16 kHz, are batched on the device in the reference's order: astype, resample
    to 16 kHz (SeparationModel.resample; the identity at 16 kHz), normalise, forward. Stereo files are reduced to the first
    channel as read_mixture does. These files do not go through read_mixture, so its notes on stereo and resampled input
    are not printed for them. Other files (float wav, rates outside that range) take the single-file path of
    :func:`read_mixture`. Writes ``<stem>_Speaker_{0,1}.wav`` into ``save_dir`` (float32 wav, or 16-bit PCM for precision
    16) and returns ``{path: vad [2, T]}``.

    ``out_rate`` sets the rate of the written files. ``None`` writes the model's 16 kHz output. ``"input"`` writes each
    file at its own rate with exactly its input length: ``SeparationModel.resample_to(out, rate)[..., :L]`` on the device
    (the round trip is zero-phase, so the output stays aligned with the input); every file's rate must then lie in
    8 .. 192 kHz, or ``ValueError`` is raised before any file is written. An integer in 8 .. 192 kHz writes every file at
    that rate, ``ceil(out_rate L16 / 16000)`` samples for a 16 kHz output of L16 samples. When a group's output rate is not
    16 kHz, 16 kHz mono files take the batched device path of the other rates."""
    from .lib import RESAMPLE_MAX_RATE, RESAMPLE_MIN_RATE
    from scipy.io.wavfile import read, write
    if out_rate is not None and out_rate != "input" and (
            isinstance(out_rate, bool) or not isinstance(out_rate, (int, np.integer))
            or not RESAMPLE_MIN_RATE <= out_rate <= RESAMPLE_MAX_RATE):
        raise ValueError(f"out_rate must be None, 'input' or an integer in {RESAMPLE_MIN_RATE} .. {RESAMPLE_MAX_RATE} Hz, "
                         f"got {out_rate!r}")

    def target(sr):   # the rate a file at sr is written at
        return 16000 if out_rate is None else int(sr) if out_rate == "input" else int(out_rate)

    Path(save_dir).mkdir(parents=True, exist_ok=True)
    kw = copy.deepcopy(DEFAULT_INFERENCE_KW)
    kw.update(inference_kw or {})
    groups, rate_groups, singles = {}, {}, []
    for pth in paths:
        sr, audio = read(pth)
        if out_rate == "input" and not RESAMPLE_MIN_RATE <= sr <= RESAMPLE_MAX_RATE:
            raise ValueError(f"{pth}: out_rate='input' needs a rate in {RESAMPLE_MIN_RATE} .. {RESAMPLE_MAX_RATE} Hz, "
                             f"the file is at {sr} Hz")
        if (sr == 16000 and audio.ndim == 1 and audio.dtype == np.int16 and len(audio) >= 257
                and target(sr) == 16000):
            groups.setdefault(len(audio), []).append((pth, audio))
        elif (RESAMPLE_MIN_RATE <= sr <= RESAMPLE_MAX_RATE and audio.dtype == np.int16 and audio.ndim in (1, 2)
              and audio.size):
            a = np.ascontiguousarray(audio if audio.ndim == 1 else _first_channel(audio))
            if -(-16000 * len(a) // sr) >= 257:
                rate_groups.setdefault((sr, len(a)), []).append((pth, a))
            else:
                singles.append((pth, sr, len(a)))
        else:
            singles.append((pth, sr, len(audio) if audio.ndim == 1 or not audio.size else len(_first_channel(audio))))
    out_dtype = torch.float16 if precision_save == 16 else torch.float32
    vads = {}

    def to_rate(out, sr, n):
        """The 16 kHz outputs [..., L16] (device) at the file's output rate; n: the file's input length."""
        r = target(sr)
        if r == 16000:
            return out
        out = model.resample_to(out, r)
        return out[..., :n] if out_rate == "input" else out

    def emit(pth, out, vad, rate=16000):
        stem = Path(pth).stem
        for s in range(2):
            a = out[s].float().numpy()
            if precision_save == 16:
                a = np.clip(np.round(a * 32767.0), -32768, 32767).astype(np.int16)
            write(os.path.join(save_dir, f"{stem}_Speaker_{s}.wav"), rate, a)
        vads[pth] = vad

    for _, items in sorted(groups.items()):
        chunks = [items[i:i + batch] for i in range(0, len(items), batch)]
        batches = (torch.from_numpy(np.stack([a for _, a in ch])) for ch in chunks)
        for ch, (out, vad) in zip(chunks, model.forward_host_stream(batches, kw, device=device, out_dtype=out_dtype, reuse_outputs=True)):
            for i, (pth, _) in enumerate(ch):
                emit(pth, out[i], vad[i].clone() if torch.is_tensor(vad) else None)
    dev = torch.device("cuda", device)
    for (sr, n), items in sorted(rate_groups.items()):
        for i in range(0, len(items), batch):
            ch = items[i:i + batch]
            x = torch.from_numpy(np.stack([a for _, a in ch])).to(dev)
            with torch.no_grad():
                out, vad, _ = model(model.minmax_normalize(model.resample(x, sr)), kw)
            out = to_rate(out, sr, n).to(out_dtype).cpu()
            vad = vad.cpu() if torch.is_tensor(vad) else None
            for j, (pth, _) in enumerate(ch):
                emit(pth, out[j], vad[j].clone() if vad is not None else None, target(sr))
    for pth, sr, n in singles:
        x = read_mixture(pth).to(torch.device("cuda", device))
        with torch.no_grad():
            out, vad, _ = model(x, kw)
        if RESAMPLE_MIN_RATE <= sr <= RESAMPLE_MAX_RATE:
            out, rate = to_rate(out, sr, n), target(sr)
        else:
            rate = 16000
        emit(pth, out[0].cpu(), vad[0].cpu() if torch.is_tensor(vad) else None, rate)
    return vads


def main(argv=None):
    args = argparse.ArgumentParser(description="septfa_b200 inference (flags of only_inference.py:110-134)")
    args.add_argument("-c", "--config", default="config_without_vad.json", type=str)
    args.add_argument("-r", "--resume", default="model_without_vad.pth", type=str)
    args.add_argument("-d", "--device", default="0", type=str, help="index of the GPU to use")
    args.add_argument("-sp", "--save_test_path", default="results_withoutvad", type=str)
    args.add_argument("-o", "--online", default=True, type=bool)  # bool-of-string, like the reference (:122)
    args.add_argument("-ps", "--precision_save", default=32, choices=[16, 32], type=int)
    args.add_argument("-pm", "--path_mix", type=str, required=True)
    args.add_argument("-ikw", "--inference_kw", type=parse_dictionary, default={})
    a = args.parse_args(argv)

    with open(a.config) as f:
        config = json.load(f)
    if config["arch"]["type"] != "SeparationModel":
        raise ValueError(f"unknown arch type {config['arch']['type']}")
    device = torch.device("cuda", int(a.device.split(",")[0]))
    model = SeparationModel(**config["arch"]["args"])                                          # :31
    model.load_state_dict(load_checkpoint_state_dict(a.resume), strict=True)                  # :57-60
    model.eval().to(device)
    inference_kw = copy.deepcopy(DEFAULT_INFERENCE_KW)                                        # :64-66
    inference_kw.update(a.inference_kw)
    x = read_mixture(a.path_mix).to(device)
    if a.online:                                                                              # :84-89
        crit = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt")
        OnlineSaving(model, a.save_test_path, crit).calc_online(x, "online_results", 0, inference_kw)
    with torch.no_grad():
        out_separation, output_vad, _ = model(x, inference_kw)                                # :90-91
    plot_spectrogram(model.mask_per_speaker, "Mask in fft domain", a.save_test_path)          # :92-94
    save_audio(x, out_separation, a.save_test_path, a.precision_save)                         # :95
    # :96-97: `config.resume == "model_without_vad.pth"` compares a pathlib.Path with a str in the reference and is
    # therefore never true there; the comparison is kept on the plain string the user typed
    if a.resume == "model_without_vad.pth":
        save_vad(output_vad, a.save_test_path)
    return out_separation, output_vad


if __name__ == "__main__":
    main()
