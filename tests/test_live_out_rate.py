"""Live sessions at an output rate (septfa_live_create_rates) and separate_files(out_rate=...), on the GPU.

Let y be the 16 kHz stream of one emitted channel: what a 16 kHz-output session returns for that stream. A session with
output rate R returns, per push k, z[k Ho, (k + 1) Ho) of z = concat(D_out zeros, resample(y, 16000, R)),
Ho = H R / 16000. The live kernel and the batch kernel compute each output sample with the same function from the same
16 kHz samples, so the stream must equal, to the bit, SeparationModel.resample_to of the 16 kHz session's output.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from septfa_b200 import synth
from septfa_b200.live import LiveSession

pytestmark = pytest.mark.gpu

INVALID = -1   # SEPTFA_E_INVALID
KW_GATE = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
# (input rate, output rate, W, H)
CASES = [(16000, 48000, 48000, 16000), (48000, 48000, 48000, 16000), (44100, 44100, 48000, 16000),
         (8000, 8000, 48000, 16000), (16000, 8000, 48000, 16000), (48000, 44100, 48000, 8000)]


def cid(c):
    return f"in{c[0]}_out{c[1]}_W{c[2]}_H{c[3]}"


def n_pushes(W, H):
    return -(-(W - H) // H) + 2


def native(n_streams, n_samples, seed):
    x = synth.make_mixtures(n_streams, n_samples, seed)
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def run_alone(m, x1, kw, W, H, rate, out_rate):
    """One stream x1 pushed hop by hop into a fresh one-slot session -> (out [2, N Ho], vad [N, 2, F], perm [N, 2])."""
    sess = LiveSession(m, 1, kw, window=W, hop=H, rate=rate, out_rate=out_rate)
    Hn = sess.input_hop
    outs, vads, perms = [], [], []
    for k in range(x1.shape[-1] // Hn):
        o, v, p = sess.push([0], x1[None, k * Hn:(k + 1) * Hn])
        outs.append(o[0]); vads.append(v[0]); perms.append(p[0])
    return torch.cat(outs, -1), torch.stack(vads), torch.stack(perms)


def at_out_rate(m, y16, out_rate, delay, n):
    """concat(delay zeros, model.resample_to(y16))[..., :n] for y16 [..., N H]."""
    return F.pad(m.resample_to(y16.contiguous(), out_rate), (delay, 0))[..., :n]


@pytest.mark.parametrize("gate", [False, True])
@pytest.mark.parametrize("case", CASES, ids=cid)
def test_live_out_rate_equals_resample_to_of_the_16k_output(cuda_models, case, gate):
    from septfa_b200 import lib as L
    rate, out_rate, W, H = case
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    kw = KW_GATE if gate else {}
    sess = LiveSession(m, 1, kw, window=W, hop=H, rate=rate, out_rate=out_rate)
    assert sess.out_rate == out_rate and sess.output_hop * 16000 == H * out_rate
    assert sess.out_delay == L.resample_to_geometry(out_rate)[0]
    N = n_pushes(W, H)
    x = native(1, N * sess.input_hop, 930)
    out, vad, perm = run_alone(m, x[0], kw, W, H, rate, out_rate)
    y16, r_vad, r_perm = run_alone(m, x[0], kw, W, H, rate, 16000)
    ref = at_out_rate(m, y16, out_rate, sess.out_delay, N * sess.output_hop)
    assert out.shape == ref.shape == (2, N * sess.output_hop)
    assert torch.equal(out.view(torch.int32), ref.view(torch.int32))
    assert torch.equal(vad, r_vad)
    assert torch.equal(perm, r_perm)


def test_live_out_rate_matches_the_oracle(cuda_models):
    """Float64 torchaudio applied to the oracle's live output (a 48 kHz stream in and out)."""
    import torchaudio.functional as AF
    from oracle import septfa_oracle as O
    rate = out_rate = 48000
    H = 16000
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 41, 0)
    sess = LiveSession(m, 2, KW_GATE, rate=rate, out_rate=out_rate)
    N, Hn, D, Ho, Do = 4, sess.input_hop, sess.delay, sess.output_hop, sess.out_delay
    x = native(2, N * Hn, 1530)
    outs, perms = [], []
    for k in range(N):
        o, _, p = sess.push([0, 1], x[:, k * Hn:(k + 1) * Hn])
        outs.append(o); perms.append(p)
    out, perm = torch.cat(outs, -1).cpu().numpy(), torch.stack(perms).cpu().numpy()
    u64 = AF.resample(x.cpu().double(), rate, 16000).numpy()
    u = np.pad(u64, ((0, 0), (D, 0)))[:, :N * H].astype(np.float32)
    Wo = O.OracleWeights(synth.make_state_dict_numpy(args, 41), args, np.float32)
    ref_sig, ref_perms = O.calc_online(np.pad(u, ((0, 0), (2 * H, 0))), Wo, dict(KW_GATE))
    assert np.array_equal(ref_perms, perm)
    z64 = AF.resample(torch.from_numpy(np.asarray(ref_sig, dtype=np.float64)), 16000, out_rate).numpy()
    ref = np.pad(z64, ((0, 0), (0, 0), (Do, 0)))[..., :N * Ho]
    assert out.shape == ref.shape
    assert np.abs(out - ref).max() < 1e-3, np.abs(out - ref).max()


def make_schedule(capacity, n_streams, steps, seed, max_hops):
    """Streams of 1 .. max_hops hops that start at random steps in random free slots, push at most once per step, and
    release their slot after their last hop -> [(released slots, [(stream, slot, k), ...])] per step."""
    rng = np.random.default_rng(seed)
    lengths = [int(v) for v in rng.integers(1, max_hops + 1, n_streams)]
    pending, active, free, sched = list(range(n_streams)), {}, list(range(capacity)), []
    for _ in range(steps):
        ended = [i for i, (_, k) in active.items() if k == lengths[i]]
        released = [active.pop(i)[0] for i in ended]
        free += released
        while pending and free and rng.random() < 0.75:
            active[pending.pop(0)] = [free.pop(int(rng.integers(len(free)))), 0]
        pushers = [i for i in active if rng.random() < 0.85]
        rng.shuffle(pushers)
        push = []
        for i in pushers:
            push.append((i, active[i][0], active[i][1]))
            active[i][1] += 1
        sched.append((released, push))
    return sched


def run_schedule(sess, x, sched):
    Hn = sess.input_hop
    res = {}
    for released, push in sched:
        if released:
            sess.release(released)
        if not push:
            continue
        out, v, perm = sess.push([sl for _, sl, _ in push], torch.stack([x[i, k * Hn:(k + 1) * Hn] for i, _, k in push]))
        for j, (i, _, k) in enumerate(push):
            r = res.setdefault(i, ([], [], []))
            assert len(r[0]) == k
            r[0].append(out[j]); r[1].append(v[j]); r[2].append(perm[j])
    return {i: (torch.cat(o, -1), torch.stack(v), torch.stack(p)) for i, (o, v, p) in res.items()}


def test_live_out_rate_staggered_streams_with_slot_reuse(cuda_models):
    """Slot reuse and release: each stream of a staggered schedule equals, to the bit, the same schedule through a
    16 kHz-output session resampled with resample_to, and matches its one-stream run."""
    rate, out_rate, W, H = 44100, 48000, 48000, 16000
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sched = make_schedule(8, 12, 10, 5, 4)
    assert any(rel for rel, _ in sched)
    sess = LiveSession(m, 8, KW_GATE, rate=rate, out_rate=out_rate)
    ref_sess = LiveSession(m, 8, KW_GATE, rate=rate)
    Hn, Ho, Do = sess.input_hop, sess.output_hop, sess.out_delay
    x = native(12, 4 * Hn, 1130)
    got, ref = run_schedule(sess, x, sched), run_schedule(ref_sess, x, sched)
    assert len(got) == 12
    for i, (o, v, p) in got.items():
        y16, r_v, r_p = ref[i]
        K = p.shape[0]
        assert torch.equal(o.view(torch.int32), at_out_rate(m, y16, out_rate, Do, K * Ho).view(torch.int32)), i
        assert torch.equal(v, r_v) and torch.equal(p, r_p), i
        a_out, a_vad, a_perm = run_alone(m, x[i, :K * Hn], KW_GATE, W, H, rate, out_rate)
        assert torch.equal(p, a_perm), i
        assert (o - a_out).abs().max().item() <= 5e-4, i
        assert (v - a_vad).abs().max().item() < 1e-3, i


def test_live_out_rate_released_slot_starts_from_zero_history(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sess = LiveSession(m, 1, KW_GATE, out_rate=44100)
    x = native(2, 3 * 16000, 1730)
    for k in range(3):
        sess.push([0], x[0:1, k * 16000:(k + 1) * 16000])
    sess.release([0])
    got = [sess.push([0], x[1:2, k * 16000:(k + 1) * 16000]) for k in range(3)]
    fresh = LiveSession(m, 1, KW_GATE, out_rate=44100)
    ref = [fresh.push([0], x[1:2, k * 16000:(k + 1) * 16000]) for k in range(3)]
    for a, b in zip(got, ref):
        for u, v in zip(a, b):
            assert torch.equal(u, v)


def test_live_out_rate_launches_and_workspace(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    n = 3
    plain = LiveSession(m, n, KW_GATE)
    same = LiveSession(m, n, KW_GATE, out_rate=16000)
    up = LiveSession(m, n, KW_GATE, out_rate=48000)
    both = LiveSession(m, n, KW_GATE, rate=48000)
    both_up = LiveSession(m, n, KW_GATE, rate=48000, out_rate=48000)
    lib = plain._h.lib
    assert (same.output_hop, same.out_delay) == (16000, 0)
    assert (up.output_hop, up.out_delay) == (48000, 18)
    for k in (1, n):
        assert lib.septfa_live_workspace_bytes(same._lv, k) == lib.septfa_live_workspace_bytes(plain._lv, k)
        extra = lib.septfa_live_workspace_bytes(up._lv, k) - lib.septfa_live_workspace_bytes(plain._lv, k)
        assert extra == -(-k * 2 * 16000 * 4 // 256) * 256   # the emitted 16 kHz hops
        assert (lib.septfa_live_workspace_bytes(both_up._lv, k) - lib.septfa_live_workspace_bytes(both._lv, k)) == extra
    x = native(n, 3 * 16000, 1930)
    x48 = native(n, 3 * 48000, 1931)
    for k in range(3):
        hop = x[:, k * 16000:(k + 1) * 16000]
        a, b = plain.push([2, 0, 1], hop), same.push([2, 0, 1], hop)
        for u, v in zip(a, b):
            assert torch.equal(u, v)
        assert same.last_launch_count == plain.last_launch_count > 70
        o, _, _ = up.push([2, 0, 1], hop)
        assert o.shape == (n, 2, 48000)
        assert up.last_launch_count == plain.last_launch_count + 1   # the output resampling kernel
        both.push([0, 1, 2], x48[:, k * 48000:(k + 1) * 48000])
        both_up.push([0, 1, 2], x48[:, k * 48000:(k + 1) * 48000])
        assert both_up.last_launch_count == both.last_launch_count + 1 == plain.last_launch_count + 2


def test_live_out_rate_refused(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sess = LiveSession(m, 2, KW_GATE, out_rate=44100)
    h, lib = sess._h, sess._h.lib
    x = native(2, 3 * 16000, 2130)
    sess.push([0, 1], x[:, :16000])
    assert lib.septfa_last_launch_count(h.ptr) > 70
    # (W, H, input rate, output rate, the rate the message names)
    for W, H, r, o, named in ((48000, 4080, 16000, 44100, "out rate 44100"), (48000, 8000, 16000, 11025, "out rate 11025"),
                              (48000, 4000, 16000, 22050, "out rate 22050"), (48000, 16000, 16000, 7999, "out rate 7999"),
                              (48000, 16000, 16000, 192001, "out rate 192001"), (48000, 16000, 48000, 0, "out rate 0"),
                              (48000, 4080, 44100, 48000, "rate 44100")):
        with pytest.raises(ValueError):
            LiveSession(m, 2, KW_GATE, window=W, hop=H, rate=r, out_rate=o)
        lv = C.c_void_p()
        assert lib.septfa_live_create_rates(h.ptr, 2, W, H, r, o, C.byref(lv)) == INVALID, (W, H, r, o)
        msg = lib.septfa_last_error(h.ptr).decode()
        assert named in msg, msg
        assert not lv.value
        assert lib.septfa_last_launch_count(h.ptr) == 0
    ref = LiveSession(m, 2, KW_GATE, out_rate=44100)
    ref.push([0, 1], x[:, :16000])
    for k in (1, 2):   # the session is unaffected by the refused creates
        a = sess.push([0, 1], x[:, k * 16000:(k + 1) * 16000])
        b = ref.push([0, 1], x[:, k * 16000:(k + 1) * 16000])
        for u, v in zip(a, b):
            assert torch.equal(u, v)


def write_files(tmp_path, specs):
    from scipy.io.wavfile import write
    paths = []
    for rate, stereo, ns in specs:
        for i, n in enumerate(ns):
            pcm = np.round(synth.make_mixture(rate + i, n, 6000 + i) * 25000.0).astype(np.int16)
            if stereo:
                pcm = np.stack([pcm, np.roll(pcm, 17) // 2], 1)
            pth = tmp_path / f"r{rate}_{i}.wav"
            write(str(pth), rate, pcm)
            paths.append((str(pth), rate, n))
    return paths


def test_separate_files_writes_at_the_input_rate(cuda_models, tmp_path):
    """out_rate="input": every wav has its file's rate and input length, and equals resample_to of the 16 kHz output
    (out_rate=None) trimmed to that length."""
    from pathlib import Path

    from scipy.io.wavfile import read
    from septfa_b200 import inference
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    kw = {"filter_signals_by_smo_vad": True}
    files = write_files(tmp_path, ((44100, True, (30000, 30000, 41000)), (48000, False, (36000, 36000)),
                                   (8000, False, (9000, 9000)), (16000, False, (20000, 20000))))
    paths = [p for p, _, _ in files]
    v16 = inference.separate_files(m, paths, str(tmp_path / "s16"), kw, batch=4)
    vin = inference.separate_files(m, paths, str(tmp_path / "sin"), kw, batch=4, out_rate="input")
    assert set(vin) == set(paths)
    for pth, rate, n in files:
        for s_ in range(2):
            name = f"{Path(pth).stem}_Speaker_{s_}.wav"
            sr16, a16 = read(str(tmp_path / "s16" / name))
            sr, a = read(str(tmp_path / "sin" / name))
            assert sr16 == 16000 and sr == rate and a.dtype == np.float32 and a.shape == (n,), (pth, sr, a.shape)
            ref = m.resample_to(torch.from_numpy(a16).cuda()[None], rate)[0, :n].cpu().numpy()
            assert np.abs(a - ref).max() < 5e-4, pth
        assert (vin[pth] - v16[pth]).abs().max().item() < 1e-3, pth


def test_separate_files_at_a_fixed_out_rate(cuda_models, tmp_path):
    """An int out_rate on a 16 kHz mono group: written at that rate with torchaudio's length."""
    from pathlib import Path

    from scipy.io.wavfile import read
    from septfa_b200 import inference
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    files = write_files(tmp_path, ((16000, False, (20000, 20000)), (44100, False, (30000,))))
    paths = [p for p, _, _ in files]
    inference.separate_files(m, paths, str(tmp_path / "s16"), {}, batch=4)
    inference.separate_files(m, paths, str(tmp_path / "s48"), {}, batch=4, out_rate=48000)
    for pth, rate, n in files:
        for s_ in range(2):
            name = f"{Path(pth).stem}_Speaker_{s_}.wav"
            _, a16 = read(str(tmp_path / "s16" / name))
            sr, a = read(str(tmp_path / "s48" / name))
            assert sr == 48000 and a.shape == (3 * a16.shape[0],)
            ref = m.resample_to(torch.from_numpy(a16).cuda()[None], 48000)[0].cpu().numpy()
            assert np.abs(a - ref).max() < 5e-4, pth


def test_separate_files_input_rate_refuses_before_writing(cuda_models, tmp_path):
    from scipy.io.wavfile import write
    from septfa_b200 import inference
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    files = write_files(tmp_path, ((16000, False, (20000,)),))
    bad = tmp_path / "r4000.wav"
    write(str(bad), 4000, np.zeros(8000, np.int16))
    with pytest.raises(ValueError):
        inference.separate_files(m, [files[0][0], str(bad)], str(tmp_path / "out"), {}, out_rate="input")
    assert not list((tmp_path / "out").glob("*.wav"))
    for bad_rate in (7999, 16000.0, "native", True):
        with pytest.raises(ValueError):
            inference.separate_files(m, [files[0][0]], str(tmp_path / "out"), {}, out_rate=bad_rate)
