"""Live sessions at a native input rate (septfa_live_create_rate) and the batched device path of separate_files for
files at other rates, on the GPU.

A stream x at `rate` is served as the 16 kHz stream u = concat(D zeros, resample(x)). The live kernel and the batch
kernel compute each output sample with the same function from the same native samples, so a one-slot session at `rate`
must equal, to the bit, a one-slot 16 kHz session fed u computed by SeparationModel.resample.
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
CASES = [(48000, 48000, 16000), (44100, 48000, 16000), (8000, 48000, 16000), (48000, 48000, 8000)]


def cid(c):
    return f"r{c[0]}_W{c[1]}_H{c[2]}"


def n_pushes(W, H):
    return -(-(W - H) // H) + 2


def native(n_streams, n_samples, rate, seed):
    """Mixtures at `rate` in [-0.9, 0.9] (synth's 16 kHz mixtures stretched; the content does not matter here)."""
    x = synth.make_mixtures(n_streams, n_samples, seed)
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def run_alone(m, x1, kw, W, H, rate, vad=True):
    """One stream x1 pushed hop by hop into a fresh one-slot session at `rate` -> (out [2, N*H], vad [N, 2, F], perm)."""
    sess = LiveSession(m, 1, kw, window=W, hop=H, rate=rate)
    Hn = sess.input_hop
    outs, vads, perms = [], [], []
    for k in range(x1.shape[-1] // Hn):
        o, v, p = sess.push([0], x1[None, k * Hn:(k + 1) * Hn], vad=vad)
        outs.append(o[0]); vads.append(v[0] if v is not None else None); perms.append(p[0])
    return torch.cat(outs, -1), (torch.stack(vads) if vad else None), torch.stack(perms)


def delayed(m, x, rate, delay, n):
    """u = concat(delay zeros, model.resample(x))[:, :n] for x [S, L]."""
    return F.pad(m.resample(x, rate), (delay, 0))[:, :n].contiguous()


def make_schedule(capacity, n_streams, steps, seed, max_hops):
    """Streams of 1 .. max_hops hops that start at random steps in random free slots, push at most once per step (some
    skip a step), and release their slot after their last hop. -> [(released slots, [(stream, slot, k), ...])] per step,
    each step's push list in random slot order."""
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


@pytest.mark.parametrize("gate", [False, True])
@pytest.mark.parametrize("case", CASES, ids=cid)
def test_live_rate_one_stream_equals_16k_session_on_resampled_stream(cuda_models, case, gate):
    rate, W, H = case
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    kw = KW_GATE if gate else {}
    sess = LiveSession(m, 1, kw, window=W, hop=H, rate=rate)
    assert sess.rate == rate and sess.input_hop * 16000 == H * rate
    assert sess.delay == {8000: 12}.get(rate, 6)
    N = n_pushes(W, H)
    x = native(1, N * sess.input_hop, rate, 930)
    out, vad, perm = run_alone(m, x[0], kw, W, H, rate)
    u = delayed(m, x, rate, sess.delay, N * H)
    r_out, r_vad, r_perm = run_alone(m, u[0], kw, W, H, 16000)
    assert out.shape == (2, N * H)
    assert torch.equal(out.view(torch.int32), r_out.view(torch.int32))
    assert torch.equal(vad, r_vad)
    assert torch.equal(perm, r_perm)


def test_live_rate_matches_the_oracle(cuda_models):
    import torchaudio.functional as AF
    from oracle import septfa_oracle as O
    rate, H = 48000, 16000
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 41, 0)
    sess = LiveSession(m, 2, KW_GATE, rate=rate)
    N, Hn, D = 4, sess.input_hop, sess.delay
    x = native(2, N * Hn, rate, 1530)
    outs, vads, perms = [], [], []
    for k in range(N):
        o, v, p = sess.push([0, 1], x[:, k * Hn:(k + 1) * Hn])
        outs.append(o); vads.append(v); perms.append(p)
    out, perm = torch.cat(outs, -1).cpu().numpy(), torch.stack(perms).cpu().numpy()
    vad = torch.stack(vads).cpu().numpy()                    # [N, 2 streams, 2, F]
    u64 = AF.resample(x.cpu().double(), rate, 16000).numpy()
    u = np.pad(u64, ((0, 0), (D, 0)))[:, :N * H].astype(np.float32)
    Wo = O.OracleWeights(synth.make_state_dict_numpy(args, 41), args, np.float32)
    win_vads = []

    def fwd(w):   # the oracle's forward, keeping each window's VAD output
        o, v, _, _ = O.forward(w, Wo, dict(KW_GATE))
        win_vads.append(v)
        return o
    ref_sig, ref_perms = O.calc_online(np.pad(u, ((0, 0), (2 * H, 0))), Wo, dict(KW_GATE), forward_fn=fwd)
    assert np.array_equal(ref_perms, perm)
    assert np.abs(out - ref_sig).max() < 1e-3, np.abs(out - ref_sig).max()
    # the push's VAD frames: the window frames j0 .. j0 + F - 1, speakers in the emitted order
    j0, F_ = sess.first_frame, sess.frames_per_hop
    ref_vad = np.stack([np.stack([win_vads[k][s_, ref_perms[k][s_], j0:j0 + F_] for s_ in range(2)]) for k in range(N)])
    assert np.abs(vad - ref_vad).max() < 1e-3, np.abs(vad - ref_vad).max()


def test_live_rate_staggered_streams_with_slot_reuse(cuda_models):
    rate, W, H = 44100, 48000, 16000
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sess = LiveSession(m, 8, KW_GATE, rate=rate)
    Hn = sess.input_hop
    sched = make_schedule(8, 12, 10, 5, 4)
    assert any(rel for rel, _ in sched)
    x = native(12, 4 * Hn, rate, 1130)
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
    assert len(res) == 12
    for i, (o, v, p) in res.items():
        o, v, p = torch.cat(o, -1), torch.stack(v), torch.stack(p)
        K = p.shape[0]
        a_out, a_vad, a_perm = run_alone(m, x[i, :K * Hn], KW_GATE, W, H, rate)
        assert torch.equal(p, a_perm), i
        assert (o - a_out).abs().max().item() <= 5e-4, i
        assert (v - a_vad).abs().max().item() < 1e-3, i


def test_live_rate_released_slot_starts_from_zero_history(cuda_models):
    rate = 48000
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sess = LiveSession(m, 1, KW_GATE, rate=rate)
    Hn = sess.input_hop
    x = native(2, 3 * Hn, rate, 1730)
    for k in range(3):
        sess.push([0], x[0:1, k * Hn:(k + 1) * Hn])
    sess.release([0])
    got = [sess.push([0], x[1:2, k * Hn:(k + 1) * Hn]) for k in range(3)]
    fresh = LiveSession(m, 1, KW_GATE, rate=rate)
    ref = [fresh.push([0], x[1:2, k * Hn:(k + 1) * Hn]) for k in range(3)]
    for a, b in zip(got, ref):
        for u, v in zip(a, b):
            assert torch.equal(u, v)


def test_resampling_banks_survive_a_weight_commit(cuda_models):
    """A weight commit (load_state_dict, .to(), refresh_weights) re-uploads the weights; the resampling banks that
    septfa_resample and the live sessions at other rates hold must stay valid across it."""
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    x = native(3, 44100, 44100, 2330)
    before = m.resample(x, 44100)
    sess = LiveSession(m, 1, KW_GATE, rate=48000)
    Hn = sess.input_hop
    xs = native(1, 3 * Hn, 48000, 2331)
    sess.push([0], xs[:, :Hn])
    m.refresh_weights()
    m(native(2, 16000, 16000, 2332), {})             # the commit, and new allocations after it
    after = m.resample(x, 44100)
    assert torch.equal(before.view(torch.int32), after.view(torch.int32))
    got = [sess.push([0], xs[:, k * Hn:(k + 1) * Hn]) for k in (1, 2)]
    fresh = LiveSession(m, 1, KW_GATE, rate=48000)
    ref = [fresh.push([0], xs[:, k * Hn:(k + 1) * Hn]) for k in range(3)][1:]
    for a, b in zip(got, ref):
        for u_, v_ in zip(a, b):
            assert torch.equal(u_, v_)


def test_live_rate_16k_equals_plain_session(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    x = native(2, 3 * 16000, 16000, 1930)
    a, b = LiveSession(m, 2, KW_GATE, rate=16000), LiveSession(m, 2, KW_GATE)
    assert (a.input_hop, a.delay) == (16000, 0)
    c = LiveSession(m, 2, KW_GATE, rate=48000)
    xc = native(2, 3 * 48000, 48000, 1931)
    for k in range(3):
        ra = a.push([1, 0], x[[1, 0], k * 16000:(k + 1) * 16000])
        rb = b.push([1, 0], x[[1, 0], k * 16000:(k + 1) * 16000])
        for u, v in zip(ra, rb):
            assert torch.equal(u, v)
        assert a.last_launch_count == b.last_launch_count > 70
        c.push([1, 0], xc[[1, 0], k * 48000:(k + 1) * 48000])
        assert c.last_launch_count == b.last_launch_count + 1   # the resampling kernel


def test_live_rate_refused(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    rate = 44100
    sess = LiveSession(m, 2, KW_GATE, rate=rate)
    Hn = sess.input_hop
    x = native(2, 3 * Hn, rate, 2130)
    h, lib = sess._h, sess._h.lib
    ref = LiveSession(m, 2, KW_GATE, rate=rate)
    sess.push([0, 1], x[:, :Hn])
    ref.push([0, 1], x[:, :Hn])
    for W, H, r in ((48000, 4080, 44100), (48000, 8000, 11025), (48000, 16000, 7999), (48000, 16000, 192001)):
        with pytest.raises(ValueError):
            LiveSession(m, 2, KW_GATE, window=W, hop=H, rate=r)
        lv = C.c_void_p()
        assert lib.septfa_live_create_rate(h.ptr, 2, W, H, r, C.byref(lv)) == INVALID, (W, H, r)
        assert f"rate {r}" in lib.septfa_last_error(h.ptr).decode()
        assert not lv.value
        assert lib.septfa_last_launch_count(h.ptr) == 0
    with pytest.raises(ValueError):
        sess.push([0, 1], x[:, :16000])             # a 16 kHz hop into a 44.1 kHz session
    with pytest.raises(ValueError):
        sess.push([0, 1], x[:, :Hn + 1])
    with pytest.raises(ValueError):
        sess.push([0], x[:, Hn:2 * Hn])             # two hops for one slot
    out = torch.empty((2, 2, 16000), device="cuda")
    perm = torch.empty((2, 2), dtype=torch.int32, device="cuda")
    ids = np.array([0, 1], dtype=np.int32)
    rc = lib.septfa_live_push(sess._lv, ids.ctypes.data_as(C.c_void_p), 2, None, None, C.c_void_p(out.data_ptr()), None,
                              C.c_void_p(perm.data_ptr()), C.c_void_p(sess._ws.data_ptr()), sess._ws.numel(),
                              C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == INVALID and lib.septfa_last_launch_count(h.ptr) == 0
    for k in (1, 2):   # every slot is as it was: the session continues like one that saw no refused call
        a = sess.push([0, 1], x[:, k * Hn:(k + 1) * Hn])
        b = ref.push([0, 1], x[:, k * Hn:(k + 1) * Hn])
        for u, v in zip(a, b):
            assert torch.equal(u, v)


def test_separate_files_batches_other_rates_on_the_device(cuda_models, tmp_path, monkeypatch):
    """Files at 44.1 kHz stereo, 48 kHz mono, 8 kHz mono and 16 kHz stereo, two of equal length per rate (a real batch):
    each file's outputs equal read_mixture + forward of that file, and none of them takes the single-file path."""
    from pathlib import Path

    from scipy.io.wavfile import read, write
    from septfa_b200 import inference
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    kw = {"filter_signals_by_smo_vad": True}
    paths = []
    for rate, stereo, ns in ((44100, True, (30000, 30000, 41000)), (48000, False, (36000, 36000, 50000)),
                             (8000, False, (9000, 9000, 12000)), (16000, True, (20000, 20000))):
        for i, n in enumerate(ns):
            pcm = np.round(synth.make_mixture(rate + i, n, 6000 + i) * 25000.0).astype(np.int16)
            if stereo:
                pcm = np.stack([pcm, np.roll(pcm, 17) // 2], 1)
            pth = tmp_path / f"r{rate}_{i}.wav"
            write(str(pth), rate, pcm)
            paths.append(str(pth))
    read_mixture = inference.read_mixture

    def single_path(pth):
        raise AssertionError(f"{pth} took the single-file path")

    monkeypatch.setattr(inference, "read_mixture", single_path)
    vads = inference.separate_files(m, paths, str(tmp_path / "sep"), kw, precision_save=32, batch=4)
    assert set(vads) == set(paths)
    full_kw = dict(synth.DEFAULT_INFERENCE_KW, **kw)
    for pth in paths:
        x = read_mixture(pth).cuda()
        ref_out, ref_vad, _ = m(x, full_kw)
        for s_ in range(2):
            sr, a = read(str(tmp_path / "sep" / f"{Path(pth).stem}_Speaker_{s_}.wav"))
            assert sr == 16000 and a.dtype == np.float32 and a.shape == (ref_out.shape[-1],)
            assert np.abs(a - ref_out[0, s_].cpu().numpy()).max() < 5e-4, pth
        assert (vads[pth] - ref_vad[0].cpu()).abs().max().item() < 1e-3, pth
