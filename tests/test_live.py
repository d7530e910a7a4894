"""Live streaming sessions (septfa_live_*, septfa_b200.LiveSession) on the GPU.

By definition a stream of N pushes in a live session emits what OnlineSaving.calc_online emits for that stream alone,
left-padded with 2 s of zeros. Where a push carries the stream in the same batch position as the reference run (one
stream per push), the forward sees bit-identical windows and everything must be equal; where streams share a push with
others, the forward's fp16 batch-placement noise is allowed, as in test_online_many_streams_equals_per_stream_runs.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from septfa_b200 import synth
from septfa_b200.live import FRAMES_PER_HOP, HOP, LiveSession
from septfa_b200.online import OnlineSaving

pytestmark = pytest.mark.gpu

INVALID, E_WORKSPACE = -1, -5   # SEPTFA_E_INVALID, SEPTFA_E_WORKSPACE

CONFIGS = {"with_vad": synth.CONFIG_WITH_VAD, "without_vad": synth.CONFIG_WITHOUT_VAD}
KW_GATE = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)


def calc_online(m, x, kw):
    """The reference semantics: OnlineSaving.calc_online(F.pad(x, (32000, 0))) -> (out [S, 2, N*HOP], perms [N, S, 2])."""
    o = OnlineSaving(m, "/tmp/septfa_live_test")
    o.num_save_samples = 0
    sig = o.calc_online(F.pad(x, (2 * HOP, 0)), "n", 0, dict(kw))
    return sig, o.last_perms


def run_alone(m, x1, kw, vad=True):
    """One stream x1 [N*HOP] pushed hop by hop into a fresh one-slot session -> (out [2, N*HOP], vad [N, 2, 63], perm [N, 2])."""
    sess = LiveSession(m, 1, kw)
    outs, vads, perms = [], [], []
    for k in range(x1.shape[-1] // HOP):
        o, v, p = sess.push([0], x1[None, k * HOP:(k + 1) * HOP], vad=vad)
        outs.append(o[0]); vads.append(v[0] if v is not None else None); perms.append(p[0])
    return torch.cat(outs, -1), (torch.stack(vads) if vad else None), torch.stack(perms)


def make_schedule(capacity, n_streams, steps, seed):
    """Streams of 1 .. 6 hops that start at random steps in random free slots, push at most once per step (some skip a
    step), and release their slot after their last hop. -> (lengths, [(released slots, [(stream, slot, k), ...])] per step),
    each step's push list in random slot order."""
    rng = np.random.default_rng(seed)
    lengths = [int(v) for v in rng.integers(1, 7, n_streams)]
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
    return lengths, sched


def run_schedule(sess, x, sched, vad=True):
    """Drive the schedule; x [n_streams, >= 6*HOP]. -> {stream: (out [2, K*HOP], vad [K, 2, 63], perm [K, 2])}."""
    res = {}
    for released, push in sched:
        if released:
            sess.release(released)
        if not push:
            continue
        hops = torch.stack([x[i, k * HOP:(k + 1) * HOP] for i, _, k in push])
        out, v, perm = sess.push([sl for _, sl, _ in push], hops, vad=vad)
        for j, (i, _, k) in enumerate(push):
            r = res.setdefault(i, ([], [], []))
            assert len(r[0]) == k
            r[0].append(out[j]); r[1].append(v[j] if v is not None else None); r[2].append(perm[j])
    return {i: (torch.cat(o, -1), torch.stack(v) if vad else None, torch.stack(p)) for i, (o, v, p) in res.items()}


@pytest.mark.parametrize("gate", [False, True])
@pytest.mark.parametrize("cfg", ["with_vad", "without_vad"])
def test_live_one_stream_equals_calc_online(cuda_models, cfg, gate):
    m = cuda_models(CONFIGS[cfg], 41, 0)
    kw = KW_GATE if gate else {}
    x = torch.from_numpy(synth.make_mixtures(1, 6 * HOP, 900)).cuda()
    ref, ref_perms = calc_online(m, x, kw)
    out, vad, perm = run_alone(m, x[0], kw)
    assert torch.equal(out, ref[0])
    assert torch.equal(perm, ref_perms[:, 0])
    assert vad.shape == (6, 2, FRAMES_PER_HOP) and torch.isfinite(vad).all()


def test_live_staggered_streams_with_slot_reuse(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    lengths, sched = make_schedule(8, 12, 10, 5)
    ns = [len(p) for _, p in sched]
    assert min(n for n in ns if n) == 1 and max(ns) == 8
    assert any(rel for rel, _ in sched)
    assert any([sl for _, sl, _ in p] != sorted(sl for _, sl, _ in p) for _, p in sched)
    x = torch.from_numpy(synth.make_mixtures(12, 6 * HOP, 1100)).cuda()
    sess = LiveSession(m, 8, KW_GATE)
    res = run_schedule(sess, x, sched)
    assert len(res) == 12
    for i, (out, vad, perm) in res.items():
        K = perm.shape[0]
        a_out, a_vad, a_perm = run_alone(m, x[i, :K * HOP], KW_GATE)
        assert torch.equal(perm, a_perm), i
        assert (out - a_out).abs().max().item() <= 5e-4, i
        assert (vad - a_vad).abs().max().item() < 1e-3, i


@pytest.mark.parametrize("smoothed", [False, True])
def test_live_vad_is_the_windows_vad_of_the_new_hop(cuda_models, smoothed):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    kw = dict(KW_GATE, return_smoothed_vad=smoothed)
    x = torch.from_numpy(synth.make_mixtures(2, 4 * HOP, 1300)).cuda()
    xp = F.pad(x, (2 * HOP, 0))
    sess, sess_novad = LiveSession(m, 2, kw), LiveSession(m, 2, kw)
    for k in range(4):
        out, vad, perm = sess.push([1, 0], x[[1, 0], k * HOP:(k + 1) * HOP])
        out2, vad2, perm2 = sess_novad.push([1, 0], x[[1, 0], k * HOP:(k + 1) * HOP], vad=False)
        assert vad2 is None and torch.equal(out, out2) and torch.equal(perm, perm2)
        win = xp[[1, 0], k * HOP:k * HOP + 3 * HOP].contiguous()
        pred, wvad, _ = m(win, dict(kw))
        wvad = wvad.reshape(2, 2, -1)[..., 125:188]
        if smoothed:
            assert set(torch.unique(wvad).tolist()) <= {0.0, 1.0}
        for j in range(2):
            assert torch.equal(vad[j], wvad[j, perm[j].long()])
            assert torch.equal(out[j], pred[j, perm[j].long(), 2 * HOP:])


def test_live_matches_the_oracle(cuda_models):
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 41, 0)
    xd = synth.make_mixtures(2, 4 * HOP, 1500)
    sess = LiveSession(m, 2, KW_GATE)
    x = torch.from_numpy(xd).cuda()
    outs, perms = [], []
    for k in range(4):
        o, _, p = sess.push([0, 1], x[:, k * HOP:(k + 1) * HOP])
        outs.append(o); perms.append(p)
    out, perm = torch.cat(outs, -1).cpu().numpy(), torch.stack(perms).cpu().numpy()
    W = O.OracleWeights(synth.make_state_dict_numpy(args, 41), args, np.float32)
    ref_sig, ref_perms = O.calc_online(np.pad(xd, ((0, 0), (2 * HOP, 0))), W, dict(KW_GATE))
    assert np.array_equal(ref_perms, perm)
    assert np.abs(out - ref_sig).max() < 1e-3, np.abs(out - ref_sig).max()


def run_1024_copies(m, kw, n_hops=4):
    """16 mixtures pushed together into a 16-slot session, and 1024 copies of them (slot s: mixture s % 16, starting at
    step (s // 16) % 3, slot lists in descending order) into a 1024-slot session -> (small, big) results, each
    (out [S, 2, n_hops*HOP], vad [S, n_hops, 2, 63], perm [S, n_hops, 2])."""
    x = torch.from_numpy(synth.make_mixtures(16, n_hops * HOP, 700)).cuda()
    small = LiveSession(m, 16, kw)
    s_res = [small.push(list(range(16)), x[:, k * HOP:(k + 1) * HOP]) for k in range(n_hops)]
    s_res = (torch.cat([o for o, _, _ in s_res], -1), torch.stack([v for _, v, _ in s_res], 1),
             torch.stack([p for _, _, p in s_res], 1))
    big = LiveSession(m, 1024, kw)
    start = (np.arange(1024) // 16) % 3
    b_out = torch.empty((1024, 2, n_hops * HOP), device="cuda")
    b_vad = torch.empty((1024, n_hops, 2, FRAMES_PER_HOP), device="cuda")
    b_perm = torch.empty((1024, n_hops, 2), dtype=torch.int32, device="cuda")
    for t in range(n_hops + 2):
        slots = np.nonzero((start <= t) & (t - start < n_hops))[0]
        ks = t - start[slots]
        hops = torch.stack([x[s % 16, k * HOP:(k + 1) * HOP] for s, k in zip(slots, ks)])
        o, v, p = (r.flip(0) for r in big.push(slots[::-1].copy(), hops.flip(0)))
        for j, (s, k) in enumerate(zip(slots, ks)):
            b_out[s, :, k * HOP:(k + 1) * HOP] = o[j]
            b_vad[s, k] = v[j]
            b_perm[s, k] = p[j]
    return s_res, (b_out, b_vad, b_perm)


def test_live_1024_slots_staggered_copies(cuda_models):
    """Without the VAD gate, so that the waveforms differ by the fp16 batch-placement noise alone (a gated frame whose
    probability lies within that noise of the threshold may be zeroed in one run and not in the other)."""
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    (s_out, s_vad, s_perm), (b_out, b_vad, b_perm) = run_1024_copies(m, dict(synth.DEFAULT_INFERENCE_KW))
    idx = torch.arange(1024, device="cuda") % 16
    assert torch.equal(b_perm, s_perm[idx])
    assert (b_out - s_out[idx]).abs().max().item() < 5e-4
    assert (b_vad - s_vad[idx]).abs().max().item() < 1e-3


def test_live_release_starts_a_new_stream(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    x = torch.from_numpy(synth.make_mixtures(2, 4 * HOP, 1700)).cuda()
    sess = LiveSession(m, 1, KW_GATE)
    for k in range(3):
        sess.push([0], x[0:1, k * HOP:(k + 1) * HOP])
    sess.release([0])
    b = [sess.push([0], x[1:2, k * HOP:(k + 1) * HOP]) for k in range(4)]
    f_out, f_vad, f_perm = run_alone(m, x[1], KW_GATE)
    assert torch.equal(torch.cat([o[0] for o, _, _ in b], -1), f_out)
    assert torch.equal(torch.stack([v[0] for _, v, _ in b]), f_vad)
    assert torch.equal(torch.stack([p[0] for _, _, p in b]), f_perm)


def test_live_refused_calls_change_nothing(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    x = torch.from_numpy(synth.make_mixtures(2, 3 * HOP, 1900)).cuda()
    sess, clean = LiveSession(m, 4, KW_GATE), LiveSession(m, 4, KW_GATE)
    for s in (sess, clean):
        s.push([2, 0], x[:, :HOP])
    h = sess._h
    lib = h.lib
    out = torch.empty((4, 2, HOP), device="cuda")
    vad = torch.empty((4, 2, FRAMES_PER_HOP), device="cuda")
    perm = torch.empty((4, 2), dtype=torch.int32, device="cuda")
    hops = x[[0, 1, 0, 1], HOP:2 * HOP].contiguous()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ws, ws_n = C.c_void_p(sess._ws.data_ptr()), sess._ws.numel()

    def push(slots, n=None, hops_p=hops.data_ptr(), out_p=out.data_ptr(), ws_bytes=ws_n):
        ids = np.asarray(slots, dtype=np.int32)
        return lib.septfa_live_push(sess._lv, ids.ctypes.data_as(C.c_void_p), len(slots) if n is None else n,
                                    C.c_void_p(hops_p) if hops_p else None, C.byref(sess._kw),
                                    C.c_void_p(out_p) if out_p else None, C.c_void_p(vad.data_ptr()),
                                    C.c_void_p(perm.data_ptr()), ws, ws_bytes, stream)

    too_small = lib.septfa_live_workspace_bytes(sess._lv, 2) - 1
    cases = [
        (dict(slots=[2, 4]), INVALID, "out of range"),
        (dict(slots=[-1]), INVALID, "out of range"),
        (dict(slots=[2, 0, 2]), INVALID, "twice"),
        (dict(slots=[0], n=0), INVALID, "capacity"),
        (dict(slots=[0, 1, 2, 3, 1], n=5), INVALID, "capacity"),
        (dict(slots=[2, 0], hops_p=0), INVALID, "null"),
        (dict(slots=[2, 0], out_p=0), INVALID, "null"),
        (dict(slots=[2, 0], ws_bytes=too_small), E_WORKSPACE, "workspace"),
    ]
    for kwargs, code, msg in cases:
        rc = push(**kwargs)
        assert rc == code, (kwargs, rc)
        assert msg in lib.septfa_last_error(h.ptr).decode(), (kwargs, lib.septfa_last_error(h.ptr))
        assert lib.septfa_last_launch_count(h.ptr) == 0
    ids = np.asarray([1, 1], dtype=np.int32)
    assert lib.septfa_live_release(sess._lv, ids.ctypes.data_as(C.c_void_p), 2, stream) == INVALID
    # the Python layer refuses the same lists before calling the library
    for bad in ([2, 4], [2, 2], [], [0, 1, 2, 3, 0]):
        with pytest.raises(ValueError):
            sess.push(bad, x[:len(bad) or 1, :HOP])
    with pytest.raises(ValueError):
        sess.release([5])
    a = sess.push([0, 2], x[[1, 0], HOP:2 * HOP])
    b = clean.push([0, 2], x[[1, 0], HOP:2 * HOP])
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert sess.last_launch_count > 70   # window assembly + the forward's ~78 kernels + PIT / emit


def test_live_is_deterministic(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 41, 0)
    _, sched = make_schedule(8, 12, 10, 5)
    x = torch.from_numpy(synth.make_mixtures(12, 6 * HOP, 2100)).cuda()
    r1 = run_schedule(LiveSession(m, 8, KW_GATE), x, sched)
    r2 = run_schedule(LiveSession(m, 8, KW_GATE), x, sched)
    assert r1.keys() == r2.keys()
    for i in r1:
        for u, v in zip(r1[i], r2[i]):
            assert torch.equal(u, v)
