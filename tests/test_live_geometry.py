"""Live sessions and the lockstep online driver with a configurable window W and hop H (septfa_live_create_win,
septfa_online_create_win) on the GPU.

The spec is the reference's OnlineSaving.calc_online with max_len = W / 16000 and save_sec = H / 16000; a live stream
is that applied to the stream left-padded with W - H zeros. As in test_live.py, one stream per push gives the forward
bit-identical windows, so everything must be equal; streams that share a push with others differ by the forward's fp16
batch-placement noise at most.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from septfa_b200 import synth
from septfa_b200.live import LiveSession
from septfa_b200.online import OnlineSaving

pytestmark = pytest.mark.gpu

INVALID = -1   # SEPTFA_E_INVALID
FS = 16000
GEOMETRIES = [(48000, 8000), (48000, 4000), (32000, 8000), (40000, 12000)]
KW_GATE = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
REFUSED = [(48000, 24016), (48000, 240), (48000, 4008), (48008, 4000), (160016, 16000)]


def gid(g):
    return f"W{g[0]}_H{g[1]}"


def n_pushes(W, H):
    """Enough pushes to reach the steady state: the overlap is the whole history from push ceil((W - H) / H) on."""
    return -(-(W - H) // H) + 2


def lockstep(m, x, kw, W, H):
    """OnlineSaving.calc_online with max_len = W / fs, save_sec = H / fs on x [S, L] -> (out [S, 2, N*H], perms [N, S, 2])."""
    o = OnlineSaving(m, "/tmp/septfa_live_geometry_test")
    o.num_save_samples = 0
    o.max_len, o.save_sec = W / FS, H / FS
    sig = o.calc_online(x, "n", 0, dict(kw))
    return sig, o.last_perms


def run_alone(m, x1, kw, W, H, vad=True):
    """One stream x1 [N*H] pushed hop by hop into a fresh one-slot session -> (out [2, N*H], vad [N, 2, F], perm [N, 2])."""
    sess = LiveSession(m, 1, kw, window=W, hop=H)
    outs, vads, perms = [], [], []
    for k in range(x1.shape[-1] // H):
        o, v, p = sess.push([0], x1[None, k * H:(k + 1) * H], vad=vad)
        outs.append(o[0]); vads.append(v[0] if v is not None else None); perms.append(p[0])
    return torch.cat(outs, -1), (torch.stack(vads) if vad else None), torch.stack(perms)


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


def run_schedule(sess, x, sched, H):
    """Drive the schedule; x [n_streams, >= max_hops*H]. -> {stream: (out [2, K*H], vad [K, 2, F], perm [K, 2])}."""
    res = {}
    for released, push in sched:
        if released:
            sess.release(released)
        if not push:
            continue
        hops = torch.stack([x[i, k * H:(k + 1) * H] for i, _, k in push])
        out, v, perm = sess.push([sl for _, sl, _ in push], hops)
        for j, (i, _, k) in enumerate(push):
            r = res.setdefault(i, ([], [], []))
            assert len(r[0]) == k
            r[0].append(out[j]); r[1].append(v[j]); r[2].append(perm[j])
    return {i: (torch.cat(o, -1), torch.stack(v), torch.stack(p)) for i, (o, v, p) in res.items()}


@pytest.mark.parametrize("gate", [False, True])
@pytest.mark.parametrize("geom", GEOMETRIES, ids=gid)
def test_live_geometry_one_stream_equals_lockstep(cuda_models, geom, gate):
    W, H = geom
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    kw = KW_GATE if gate else {}
    N = n_pushes(W, H)
    x = torch.from_numpy(synth.make_mixtures(1, N * H, 910)).cuda()
    ref, ref_perms = lockstep(m, F.pad(x, (W - H, 0)), kw, W, H)
    assert ref.shape == (1, 2, N * H)
    out, vad, perm = run_alone(m, x[0], kw, W, H)
    assert torch.equal(out, ref[0])
    assert torch.equal(perm, ref_perms[:, 0])
    assert torch.isfinite(vad).all()


@pytest.mark.parametrize("geom", [(48000, 4000), (40000, 12000)], ids=gid)
def test_live_geometry_and_lockstep_match_the_oracle(cuda_models, geom):
    from oracle import septfa_oracle as O
    W, H = geom
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 41, 0)
    N = n_pushes(W, H)
    xd = synth.make_mixtures(2, N * H, 1510)
    xp = np.pad(xd, ((0, 0), (W - H, 0)))
    Wo = O.OracleWeights(synth.make_state_dict_numpy(args, 41), args, np.float32)
    # calc_online slices with fs * indx * save_sec and fs * max_len, which numpy takes only as integers; the forward
    # does not depend on fs, so the same windows and hops are expressed in units of g = gcd(W, H) samples
    g = math.gcd(W, H)
    ref_sig, ref_perms = O.calc_online(xp, Wo, dict(KW_GATE), fs=g, max_len=W // g, save_sec=H // g)
    assert ref_sig.shape == (2, 2, N * H)
    x = torch.from_numpy(xd).cuda()
    sess = LiveSession(m, 2, KW_GATE, window=W, hop=H)
    outs, perms = [], []
    for k in range(N):
        o, _, p = sess.push([0, 1], x[:, k * H:(k + 1) * H])
        outs.append(o); perms.append(p)
    live_out, live_perm = torch.cat(outs, -1).cpu().numpy(), torch.stack(perms).cpu().numpy()
    ls_out, ls_perm = lockstep(m, torch.from_numpy(xp).cuda(), KW_GATE, W, H)
    for out, perm in ((live_out, live_perm), (ls_out.cpu().numpy(), ls_perm.cpu().numpy())):
        assert np.array_equal(ref_perms, perm)
        assert np.abs(out - ref_sig).max() < 1e-3, np.abs(out - ref_sig).max()


@pytest.mark.parametrize("smoothed", [False, True])
@pytest.mark.parametrize("geom", GEOMETRIES + [(49152, 4096)], ids=gid)
def test_live_geometry_vad_is_the_windows_vad_of_the_new_hop(cuda_models, geom, smoothed):
    W, H = geom
    R = W - H
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    kw = dict(KW_GATE, return_smoothed_vad=smoothed)
    sess = LiveSession(m, 2, kw, window=W, hop=H)
    j0, nf = sess.first_frame, sess.frames_per_hop
    assert (j0, nf) == (-(-R // 256), -(-W // 256) - -(-R // 256))
    if geom == (49152, 4096):
        assert (nf, j0) == (16, 176)
    N = n_pushes(W, H)
    x = torch.from_numpy(synth.make_mixtures(2, N * H, 1310)).cuda()
    xp = F.pad(x, (R, 0))
    for k in range(N):
        out, vad, perm = sess.push([1, 0], x[[1, 0], k * H:(k + 1) * H])
        assert vad.shape == (2, 2, nf)
        win = xp[[1, 0], k * H:k * H + W].contiguous()
        pred, wvad, _ = m(win, dict(kw))
        wvad = wvad.reshape(2, 2, -1)[..., j0:j0 + nf]
        if smoothed:
            assert set(torch.unique(wvad).tolist()) <= {0.0, 1.0}
        for j in range(2):
            assert torch.equal(vad[j], wvad[j, perm[j].long()])
            assert torch.equal(out[j], pred[j, perm[j].long(), R:])


def test_live_geometry_staggered_schedule(cuda_models):
    W, H = 48000, 4000
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sched = make_schedule(8, 12, 40, 7, 16)
    assert any(rel for rel, _ in sched)
    assert any([sl for _, sl, _ in p] != sorted(sl for _, sl, _ in p) for _, p in sched)
    assert max(k for _, p in sched for _, _, k in p) >= (W - H) // H + 1   # some stream reaches the steady state
    x = torch.from_numpy(synth.make_mixtures(12, 16 * H, 1110)).cuda()
    res = run_schedule(LiveSession(m, 8, KW_GATE, window=W, hop=H), x, sched, H)
    assert len(res) == 12
    for i, (out, vad, perm) in res.items():
        K = perm.shape[0]
        a_out, a_vad, a_perm = run_alone(m, x[i, :K * H], KW_GATE, W, H)
        assert torch.equal(perm, a_perm), i
        assert (out - a_out).abs().max().item() <= 5e-4, i
        assert (vad - a_vad).abs().max().item() < 1e-3, i
    res2 = run_schedule(LiveSession(m, 8, KW_GATE, window=W, hop=H), x, sched, H)
    assert res.keys() == res2.keys()
    for i in res:
        for u, v in zip(res[i], res2[i]):
            assert torch.equal(u, v)


def test_live_geometry_1024_slots_staggered_copies(cuda_models):
    """16 mixtures pushed together into a 16-slot session, and 1024 copies of them (slot s: mixture s % 16, starting at
    step (s // 16) % 3, slot lists in descending order) into a 1024-slot session. Without the VAD gate, as in
    test_live_1024_slots_staggered_copies."""
    W, H = 48000, 4000
    kw = dict(synth.DEFAULT_INFERENCE_KW)
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    N = n_pushes(W, H)
    x = torch.from_numpy(synth.make_mixtures(16, N * H, 710)).cuda().view(16, N, H)
    small = LiveSession(m, 16, kw, window=W, hop=H)
    s_res = [small.push(list(range(16)), x[:, k]) for k in range(N)]
    s_out = torch.stack([o for o, _, _ in s_res], 1)    # [16, N, 2, H]
    s_vad = torch.stack([v for _, v, _ in s_res], 1)
    s_perm = torch.stack([p for _, _, p in s_res], 1)
    big = LiveSession(m, 1024, kw, window=W, hop=H)
    start = (np.arange(1024) // 16) % 3
    b_out = torch.empty((1024, N, 2, H), device="cuda")
    b_vad = torch.empty((1024, N, 2, big.frames_per_hop), device="cuda")
    b_perm = torch.empty((1024, N, 2), dtype=torch.int32, device="cuda")
    for t in range(N + 2):
        slots = np.nonzero((start <= t) & (t - start < N))[0][::-1].copy()
        si = torch.from_numpy(slots).long().cuda()
        ks = torch.from_numpy(t - start[slots]).long().cuda()
        o, v, p = big.push(slots, x[si % 16, ks].contiguous())
        b_out[si, ks], b_vad[si, ks], b_perm[si, ks] = o, v, p
    idx = torch.arange(1024, device="cuda") % 16
    assert torch.equal(b_perm, s_perm[idx])
    assert (b_out - s_out[idx]).abs().max().item() < 5e-4
    assert (b_vad - s_vad[idx]).abs().max().item() < 1e-3


def test_live_create_win_default_equals_live_create(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    H = 16000
    sched = make_schedule(8, 12, 10, 5, 6)
    x = torch.from_numpy(synth.make_mixtures(12, 6 * H, 2110)).cuda()
    a = LiveSession(m, 8, KW_GATE, window=48000, hop=16000)
    b = LiveSession(m, 8, KW_GATE)
    b.close()   # the same session object, its state from the fixed-geometry entry point
    _lv = C.c_void_p()
    assert b._h.lib.septfa_live_create(b._h.ptr, 8, C.byref(_lv)) == 0
    b._lv = _lv
    ra, rb = run_schedule(a, x, sched, H), run_schedule(b, x, sched, H)
    assert ra.keys() == rb.keys() and len(ra) == 12
    for i in ra:
        for u, v in zip(ra[i], rb[i]):
            assert torch.equal(u, v)


def test_live_geometry_refused(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    sess = LiveSession(m, 2, KW_GATE, window=48000, hop=4000)
    x = torch.from_numpy(synth.make_mixtures(2, 48000 + 2 * 4800, 1910)).cuda()
    h = sess._h
    lib = h.lib
    for W, H in REFUSED:
        sess.push([0, 1], x[:, :4000])
        assert lib.septfa_last_launch_count(h.ptr) > 70
        lv = C.c_void_p()
        assert lib.septfa_live_create_win(h.ptr, 2, W, H, C.byref(lv)) == INVALID, (W, H)
        assert f"window {W}, hop {H}" in lib.septfa_last_error(h.ptr).decode()
        assert not lv.value
        assert lib.septfa_last_launch_count(h.ptr) == 0
        sess.push([0, 1], x[:, :4000])
        st = C.c_void_p()
        assert lib.septfa_online_create_win(h.ptr, 2, W, H, C.byref(st)) == INVALID, (W, H)
        assert f"window {W}, hop {H}" in lib.septfa_last_error(h.ptr).decode()
        assert not st.value
        assert lib.septfa_last_launch_count(h.ptr) == 0
        with pytest.raises(ValueError):
            LiveSession(m, 2, KW_GATE, window=W, hop=H)
    with pytest.raises(ValueError):
        sess.push([0, 1], x[:, :16000])   # a hop of the default length into a 4000-sample session
    # OnlineSaving: 0.3 s hops (4800 samples) run; 0.2001 s (3201.6 samples) is refused before anything is launched
    o = OnlineSaving(m, "/tmp/septfa_live_geometry_test")
    o.num_save_samples = 0
    o.save_sec = 0.3
    sig = o.calc_online(x, "n", 0, {})
    assert sig.shape == (2, 2, 3 * 4800) and o.last_perms.shape == (3, 2, 2) and torch.isfinite(sig).all()
    o.save_sec = 0.2001
    sess.push([0, 1], x[:, :4000])
    with pytest.raises(NotImplementedError):
        o.calc_online(x, "n", 0, {})
    assert o.indx == 0
