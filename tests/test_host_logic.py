"""CPU: host-side logic - the C ABI library loads and exports every symbol include/septfa.h
declares, the drop-in module keeps the reference's state_dict layout, PIT / reorder / SI-SDR
helpers, seeded synthetic inputs, the batch sharding plan (incl. a 2-rank gloo run)."""
import contextlib
import ctypes
import io
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from septfa_b200 import lib as L
from septfa_b200 import synth


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "septfa.h")).read()
    declared = set(re.findall(r"\b(septfa_[a-z0-9_]+)\s*\(", header))
    assert declared, "no prototypes found"
    assert os.path.exists(L.LIB_PATH), "libseptfa.so not built (python -m septfa_b200.build)"
    so = ctypes.CDLL(L.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(so, name), f"{name} declared in septfa.h but not exported"
    assert declared == set(L.EXPORTED_SYMBOLS), "ctypes prototypes out of sync with the header"
    lib = L.load()
    assert b"sm_100a" in lib.septfa_version()
    assert lib.septfa_num_frames(64000) == 251 and lib.septfa_num_frames(48000) == 188


def test_no_cpu_fallback_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from septfa_b200.model import SeparationModel
    with contextlib.redirect_stdout(io.StringIO()):
        m = SeparationModel(**synth.CONFIG_WITH_VAD)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 4000))
    # the C ABI refuses too: no device -> error code, never a silent CPU path
    lib = L.load()
    h = ctypes.c_void_p()
    cfg = L.Config.from_args(synth.CONFIG_WITH_VAD)
    assert lib.septfa_create(ctypes.byref(h), ctypes.byref(cfg), 0) != 0
    assert b"CUDA" in lib.septfa_last_error(None)


@pytest.mark.parametrize("name,cfg", [("with_vad", synth.CONFIG_WITH_VAD), ("without_vad", synth.CONFIG_WITHOUT_VAD)])
def test_state_dict_layout_equals_reference(name, cfg):
    """Keys, order and shapes recorded from the reference's own SeparationModel (make_golden env)."""
    from septfa_b200.model import SeparationModel
    ref = json.load(open(os.path.join(GOLDEN, "state_dict_keys.json")))[name]
    with contextlib.redirect_stdout(io.StringIO()) as out:
        m = SeparationModel(**cfg)
    assert "n_fftBins" in out.getvalue()  # the reference prints the merged config (model/model.py:371)
    mine = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert list(mine.keys()) == list(ref.keys())
    assert mine == ref
    m.load_state_dict(synth.make_state_dict(cfg, 11), strict=True)
    bad = synth.make_state_dict(cfg, 11)
    bad.pop("TCN.LN.weight")
    with pytest.raises(RuntimeError):
        m.load_state_dict(bad, strict=True)


def test_unsupported_configs_fail_loudly():
    from septfa_b200.model import SeparationModel
    for bad in ({"casual": True}, {"skip": True}, {"weight_norm": False}, {"dilated": False}, {"BN_dim": 128}):
        with contextlib.redirect_stdout(io.StringIO()), pytest.raises(NotImplementedError):
            SeparationModel(**dict(synth.CONFIG_WITH_VAD, **bad))


def test_infer_kw_semantics():
    assert L.InferKw.from_dict({}) is None
    with pytest.raises(KeyError):  # missing keys raise like model/model.py:445-456
        L.InferKw.from_dict({"filter_signals_by_smo_vad": True})
    kw = L.InferKw.from_dict(dict(synth.DEFAULT_INFERENCE_KW, threshold_activated_vad=0.3))
    assert abs(kw.threshold_activated_vad - 0.3) < 1e-7 and kw.length_smoothing_filter == 3


def test_pit_host_helpers_match_reference_semantics():
    from septfa_b200.pit import PITLossWrapper, calc_sisdr, reorder_source_mse
    torch.manual_seed(0)
    tgt = torch.randn(3, 2, 500)
    est = tgt[:, [1, 0]] + 0.01 * torch.randn(3, 2, 500)
    w = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt", per_stream=True)
    loss, idx = w(est, tgt, return_incides=True)
    assert idx.tolist() == [[1, 0]] * 3
    assert torch.allclose(reorder_source_mse(est, idx), est[:, [1, 0]])
    # reference quirk: nn.L1Loss reduces over the batch -> one joint decision (model/pit_wrapper.py:173-176)
    mixed_est = torch.cat([tgt[:1], tgt[1:, [1, 0]]])
    _, joint = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt")(mixed_est, tgt, return_incides=True)
    assert joint.tolist() == [[1, 0]] * 3
    _, per = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt", per_stream=True)(mixed_est, tgt, return_incides=True)
    assert per.tolist() == [[0, 1], [1, 0], [1, 0]]
    # ties -> identity
    z = torch.zeros(1, 2, 10)
    assert PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt")(z, z, return_incides=True)[1].tolist() == [[0, 1]]
    v = calc_sisdr(torch.tensor([2.5, 0.0, 2.0, 8.0]), torch.tensor([3.0, -0.5, 2.0, 7.0]), zero_mean=False)
    assert abs(v.item() - 18.4030) < 1e-3


def test_synth_is_deterministic_and_normalised():
    a = synth.make_mixtures(2, 5000, 77)
    b = synth.make_mixtures(2, 5000, 77)
    assert np.array_equal(a, b) and a.dtype == np.float32
    assert abs(a.max() - 0.9) < 1e-6 and abs(a.min() + 0.9) < 1e-6  # only_inference.py:81
    sd = synth.make_state_dict_numpy(synth.CONFIG_WITH_VAD, 5)
    assert len(sd) == 719 and sum(v.size for k, v in sd.items() if "window" not in k) == 5005347


def test_shard_plan():
    from septfa_b200.shard import shard_range
    for n, w in ((8192, 8), (10, 4), (3, 8), (256, 1)):
        parts = [shard_range(n, r, w) for r in range(w)]
        assert parts[0][0] == 0 and parts[-1][1] == n
        assert all(parts[i][1] == parts[i + 1][0] for i in range(w - 1))
        assert max(b - a for a, b in parts) - min(b - a for a, b in parts) <= 1


@pytest.mark.timeout(300)
def test_two_rank_gloo_sharding_and_metric_gather(tmp_path):
    """world_size-2 gloo run of the sharding/gather host logic (the data path has no collective)."""
    script = tmp_path / "w.py"
    script.write_text(
        "import os, sys, torch, torch.distributed as dist\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "from septfa_b200.shard import shard_range, gather_max_time, gather_counts\n"
        "dist.init_process_group('gloo')\n"
        "r, w = dist.get_rank(), dist.get_world_size()\n"
        "a, b = shard_range(11, r, w)\n"
        "tot = gather_counts(b - a)\n"
        "t = gather_max_time(0.5 + r)\n"
        "assert tot == 11 and abs(t - 1.5) < 1e-9, (tot, t)\n"
        "if r == 0: print('OK', tot, t)\n"
        "dist.destroy_process_group()\n")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731", str(script)],
                       capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "OK 11 1.5" in r.stdout


def test_pit_helpers_equal_reference_functions():
    """The re-written pairwise-loss / exhaustive-permutation helpers against the reference's, 2 and 3 sources, including
    exact ties (-> identity, torch.min's first index). The expected values are stored in tests/golden/reference_helpers.npz:
    computed by the reference's own functions where it can be imported, otherwise by tests/golden/make_helper_golden.py's
    restatement of their code, which shares nothing with septfa_b200 (``meta["source"]`` says which)."""
    from conftest import load_golden
    from septfa_b200.pit import PITLossWrapper
    g, _ = load_golden("reference_helpers")
    for n_src in (2, 3):
        pw = torch.from_numpy(g[f"pit_pw{n_src}"])       # rows of all-equal entries and rows with partial ties
        loss, idx = PITLossWrapper.find_best_perm_factorial(pw)
        assert np.array_equal(idx.numpy(), g[f"pit_idx{n_src}"]) and np.allclose(loss.numpy(), g[f"pit_loss{n_src}"],
                                                                                 rtol=0, atol=1e-7)
    est, tgt = torch.from_numpy(g["pit_est"]), torch.from_numpy(g["pit_tgt"])
    l1 = torch.nn.L1Loss()
    assert np.array_equal(PITLossWrapper.get_pw_losses(l1, est, tgt).numpy(), g["pit_pw_l1"])
    loss, idx = PITLossWrapper(l1, pit_from="pw_pt")(est, tgt, return_incides=True)
    assert np.array_equal(idx.numpy(), g["pit_wrapper_idx"]) and abs(loss.item() - g["pit_wrapper_loss"].item()) < 1e-7


def test_reference_bytecode_build_matches_source(tmp_path):
    """oracle/ref_loader.py: the byte-compiled reference under oracle/_ref (what the GPU box imports) is the same program
    as /root/reference (what this container imports): same forward result for the same weights and input."""
    from oracle import ref_loader
    if not os.path.isdir(ref_loader.REF_SRC):
        pytest.skip("reference sources not present")
    assert ref_loader.build_ref()
    code = (
        "import sys, io, contextlib, warnings; warnings.filterwarnings('ignore'); sys.path.insert(0, %r)\n"
        "import numpy as np, torch\n"
        "from oracle import ref_loader\n"
        "from septfa_b200 import synth\n"
        "ns = ref_loader.load()\n"
        "with contextlib.redirect_stdout(io.StringIO()):\n"
        "    m = ns.model.SeparationModel(**synth.CONFIG_WITH_VAD)\n"
        "m.load_state_dict(synth.make_state_dict(synth.CONFIG_WITH_VAD, 3)); m.eval()\n"
        "with torch.no_grad():\n"
        "    out, vad, _ = m(torch.from_numpy(synth.make_mixtures(1, 9000, 77)), {})\n"
        "np.save(sys.argv[1], np.concatenate([out.numpy().ravel(), vad.numpy().ravel()]))\n"
        "print(ns.kind)\n" % ROOT)
    res = {}
    for kind, env_ref in (("source", ref_loader.REF_SRC), ("bytecode", "/nonexistent")):
        out = tmp_path / f"{kind}.npy"
        r = subprocess.run([sys.executable, "-c", code, str(out)], capture_output=True, text=True,
                           env=dict(os.environ, SEPTFA_REFERENCE=env_ref, PYTHONDONTWRITEBYTECODE="1"))
        assert r.returncode == 0, r.stderr[-2000:]
        assert r.stdout.strip().endswith(kind)
        res[kind] = np.load(out)
    assert np.array_equal(res["source"], res["bytecode"])


def test_cli_host_preprocessing_and_writers_match_reference_golden(tmp_path):
    """The host side of ``only_inference.py`` either side of the forward, without a GPU: ``read_mixture`` (stereo int16
    wav -> channel 0 -> float32 -> min-max normalise, only_inference.py:68-83) must reproduce the ``Mixed_0.wav`` the
    UNMODIFIED reference script wrote for the same file (tests/golden/cli_with_vad_ps32.npz); ``save_audio``
    (Our_utils/utlis_inference.py:24-37) round-trips float32 and writes 16-bit PCM for ``-ps 16``; ``save_vad``
    (:39-46) writes the 0.5-thresholded decisions of batch item 0; ``parse_dictionary`` (only_inference.py:17-23)."""
    import argparse
    from scipy.io.wavfile import read, write
    from conftest import load_golden
    from septfa_b200 import inference
    g, meta = load_golden("cli_with_vad_ps32")
    wav = tmp_path / "mix.wav"
    write(str(wav), 16000, synth.make_cli_wav(meta["weight_seed"], fs=16000))
    with contextlib.redirect_stdout(io.StringIO()) as said:
        x = inference.read_mixture(str(wav))
    assert "not mono" in said.getvalue()
    assert x.dtype == torch.float32 and tuple(x.shape) == (1, 48000)
    assert np.abs(x[0].numpy() - g["Mixed_0"]).max() <= 1e-6
    assert abs(x.max().item() - 0.9) < 1e-6 and abs(x.min().item() + 0.9) < 1e-6
    # writers
    sep = torch.stack([torch.from_numpy(g["Speaker_0"]), torch.from_numpy(g["Speaker_1"])])[None]
    inference.save_audio(x, sep, str(tmp_path / "o32"), 32)
    for name in ("Speaker_0", "Speaker_1"):
        sr, a = read(str(tmp_path / "o32" / f"{name}.wav"))
        assert sr == 16000 and a.dtype == np.float32 and np.array_equal(a, g[name])
    sr, m = read(str(tmp_path / "o32" / "Mixed_0.wav"))
    assert np.array_equal(m, x[0].numpy())
    inference.save_audio(x, sep, str(tmp_path / "o16"), 16)
    sr, a16 = read(str(tmp_path / "o16" / "Speaker_1.wav"))
    assert sr == 16000 and a16.dtype == np.int16 and np.abs(a16 / 32767.0 - g["Speaker_1"]).max() <= 0.5 / 32767 + 1e-7
    vad = torch.tensor([[[0.2, 0.5, 0.7, 0.49], [0.9, 0.1, 0.5, 0.0]]])
    inference.save_vad(vad, str(tmp_path / "vad"))
    inference.save_vad(vad[:, :, None], str(tmp_path / "vad4"))            # [B, 2, 1, T] of return_smoothed_vad
    for d in ("vad", "vad4"):
        files = sorted(p.name for p in (tmp_path / d).iterdir())
        assert [f.rsplit(".", 1)[0] for f in files] == ["estimated_vad_0", "estimated_vad_1"]
        if files[0].endswith(".npy"):
            assert np.array_equal(np.load(str(tmp_path / d / files[0])), [0, 1, 1, 0])
            assert np.array_equal(np.load(str(tmp_path / d / files[1])), [1, 0, 1, 0])
    assert inference.parse_dictionary('{"filter_signals_by_smo_vad": true}') == {"filter_signals_by_smo_vad": True}
    with pytest.raises(argparse.ArgumentTypeError):
        inference.parse_dictionary("{not json")


def test_integration_doc_lists_every_entry_point():
    """INTEGRATION.md's entry-point table names every symbol include/septfa.h declares (and nothing the header lacks)."""
    header = open(os.path.join(ROOT, "include", "septfa.h")).read()
    declared = set(re.findall(r"\b(septfa_[a-z0-9_]+)\s*\(", header))
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    table = doc.split("### Entry points and the reference interface each one stands for")[1].split("## 3. Build")[0]
    listed = set(re.findall(r"`(septfa_[a-z0-9_]+)`", "\n".join(l.split("|")[1] for l in table.splitlines() if l.startswith("| `"))))
    assert listed == declared, (sorted(declared - listed), sorted(listed - declared))
