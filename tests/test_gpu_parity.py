"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI
(ctypes -> libseptfa.so), against (a) the golden vectors produced by the unmodified reference,
(b) the numpy oracle on seeded inputs, (c) size-independent properties at full size.

Tolerances (north_star: waveform max-abs + SI-SDR delta < 0.05 dB vs the fp32 reference; VAD
decisions bit-exact except frames whose reference probability lies within 1e-3 of the threshold):
  * default engine (tcgen05, fp16 operands, fp32 accumulate): |wav - ref| <= 5e-4 abs on signals of
    RMS ~0.1, SI-SDR(ours, ref) >= 60 dB (an error 60 dB below the signal moves any SI-SDR against
    any target by < 0.01 dB), |p - p_ref| < 1e-3 on every frame, decisions as stated above;
  * fp32 CUDA-core engine: |wav - ref| <= 2e-5, SI-SDR >= 100 dB, |p - p_ref| < 5e-5.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, sisdr_db
from septfa_b200 import synth

pytestmark = pytest.mark.gpu

# est: |e - ref| <= 2e-3 * (1 + |ref|): 2e-3 absolute on small values, 2e-3 relative on the large ones (|S| reaches ~40)
TOL = {0: dict(wav=5e-4, sisdr=60.0, vad=1e-3, logits=1e-2, est=2e-3),
       7: dict(wav=2e-5, sisdr=100.0, vad=5e-5, logits=5e-4, est=1e-4)}


def check_decisions(p, p_ref, thr):
    """VAD frame decisions agree bit-exactly except where |p_ref - thr| < 1e-3."""
    d, d_ref = p >= np.float32(thr), p_ref >= np.float32(thr)
    bad = (d != d_ref) & (np.abs(p_ref - thr) >= 1e-3)
    assert not bad.any(), f"{bad.sum()} VAD decisions differ outside the 1e-3 band"


def smoothed_from(p, thr):
    d = (p >= np.float32(thr)).astype(np.float32)
    sm = d.copy()
    if p.shape[-1] >= 3:
        sm[..., 1:-1] = np.minimum(d[..., :-2] + d[..., 2:], 1.0)
    return sm


def gate_unsure(p_ref, thr):
    """Frames whose SMOOTHED decision may legitimately differ between two implementations that agree on every raw
    decision outside the 1e-3 band: s[t] depends on d[t-1] and d[t+1] (on d[t] at the two edges), model.py:449-451."""
    near = np.abs(p_ref - np.float32(thr)) < 1e-3
    unsure = near.copy()
    if near.shape[-1] >= 3:
        unsure[..., 1:-1] = near[..., :-2] | near[..., 2:]
    return unsure


def check_outputs(out, est, p, ref_out, ref_est, p_ref, kw, tol, stride=1, wav_scale=1.0):
    """Waveforms and estimated STFTs against the reference with the VAD gate in force. Where the smoothed gate of a
    frame differs - allowed only if a raw decision behind it lies inside the 1e-3 band - that frame (est) and the 512
    samples it overlaps (waveform) are left out; EVERYTHING else is compared. Nothing is skipped silently."""
    B, S, T = p.shape
    frame_ok = np.ones((B, S, T), dtype=bool)
    if kw and (kw.get("filter_signals_by_smo_vad") or kw.get("filter_signals_by_unsmo_vad")):
        thr = kw["threshold_activated_vad"]
        diff = smoothed_from(p, thr) != smoothed_from(p_ref, thr)
        assert not (diff & ~gate_unsure(p_ref, thr)).any(), "smoothed gate differs outside the 1e-3 band"
        frame_ok = ~diff
    if est is not None and ref_est is not None:
        err = np.abs(est - ref_est) / (1.0 + np.abs(ref_est))
        err = np.where(frame_ok[:, :, None, :], err, 0.0)
        assert err.max() <= tol["est"], ("est", err.max())
    L = out.shape[-1]
    samp_ok = np.ones(out.shape, dtype=bool)
    for b, s_, t in zip(*np.nonzero(~frame_ok)):     # frame t overlaps output samples [256 (t-1), 256 (t+1))
        samp_ok[b, s_, max(0, 256 * (t - 1)):min(L, 256 * (t + 1))] = False
    o, r, ok = out[..., ::stride], ref_out, samp_ok[..., ::stride]
    assert o.shape == r.shape
    d = np.where(ok, o - r, 0.0)
    assert np.abs(d).max() <= tol["wav"] * wav_scale, ("wav", np.abs(d).max())
    assert sisdr_db(np.where(ok, o, 0.0), np.where(ok, r, 0.0)) >= tol["sisdr"]
    return int((~frame_ok).sum())


def run_golden(cuda_models, name, engine):
    g, meta = load_golden(name)
    tol = TOL[engine]
    m = cuda_models(meta["args"], meta["weight_seed"], engine)
    x = torch.from_numpy(synth.make_mixtures(meta["n"], meta["length"], meta["base_seed"])).cuda()
    st = meta["stride"]
    # probabilities: ours from a plain forward, the reference's from the first case that returns them
    p_ours = m(x, {})[1].cpu().numpy() if meta["args"]["final_vad"] else None
    i_prob = next(i for i, kw in enumerate(meta["kws"]) if not (kw and kw.get("return_smoothed_vad")))
    p_ref = g[f"kw{i_prob}_vad"]
    if p_ours is not None:
        assert np.abs(p_ours - p_ref).max() < tol["vad"], np.abs(p_ours - p_ref).max()
    for i, kw in enumerate(meta["kws"]):
        out, vad, est = m(x, dict(kw) if kw else {})
        assert m.last_launch_count > 70  # our kernels ran (no library / CPU path exists)
        ref_vad = g[f"kw{i}_vad"]
        if ref_vad.size:
            v = vad.cpu().numpy()
            assert v.shape == ref_vad.shape
            thr = kw["threshold_activated_vad"] if kw else 0.5
            if kw and kw.get("return_smoothed_vad"):
                # the returned smoothed decisions [B,2,1,T]: exactly the smoothing of our own probabilities, and equal to
                # the REFERENCE's smoothed decisions on every frame no in-band raw decision can influence
                assert set(np.unique(v)) <= {0.0, 1.0}
                assert np.array_equal(v[:, :, 0], smoothed_from(p_ours, thr))
                assert not ((v[:, :, 0] != ref_vad[:, :, 0]) & ~gate_unsure(p_ref, thr)).any()
            else:
                assert np.abs(v - ref_vad).max() < tol["vad"], np.abs(v - ref_vad).max()
                check_decisions(v, ref_vad, thr)
        ref_est = g[f"kw{i}_est"] if f"kw{i}_est" in g else None
        e = est.cpu().numpy()
        if ref_est is not None:
            assert e.dtype == np.complex64 and e.shape == ref_est.shape
        check_outputs(out.cpu().numpy(), e if ref_est is not None else None, p_ours, g[f"kw{i}_out"], ref_est, p_ref, kw, tol, stride=st)
        if i == 0 and "logits" in g:
            assert np.abs(m.masks_b.cpu().numpy() - g["logits"]).max() < tol["logits"]
            sp = m.spectrum.cpu().numpy()
            assert np.abs(sp - g["spectrum"]).max() < 2e-5 * np.abs(g["spectrum"]).max()
            assert np.abs(m.mask_per_speaker.cpu().numpy() - g["mask"]).max() < tol["logits"]
    return m, x, g, meta


@pytest.mark.parametrize("engine", [0, 7])
@pytest.mark.parametrize("name", ["fwd_with_vad_small", "fwd_without_vad_small"])
def test_small_golden(cuda_models, name, engine):
    run_golden(cuda_models, name, engine)


@pytest.mark.parametrize("engine", [0, 7])
def test_cfg1_one_4s_mixture(cuda_models, engine):
    """BASELINE.json configs[0]: config_with_vad, one 4 s mixture, VAD gating on."""
    run_golden(cuda_models, "cfg1_with_vad_4s", engine)


def test_online_window_length_3s(cuda_models):
    run_golden(cuda_models, "fwd_with_vad_3s", 0)  # T = 188, ragged istft tail (L % 256 = 128)


def test_long_form_60s(cuda_models):
    run_golden(cuda_models, "cfg4_without_vad_60s", 0)  # T = 3751, separation-only config


def test_smoothed_vad_is_smoothing_of_own_decisions(cuda_models):
    g, meta = load_golden("fwd_with_vad_small")
    m = cuda_models(meta["args"], meta["weight_seed"], 0)
    x = torch.from_numpy(synth.make_mixtures(meta["n"], meta["length"], meta["base_seed"])).cuda()
    kw = dict(synth.DEFAULT_INFERENCE_KW, return_smoothed_vad=True, threshold_activated_vad=0.45,
              length_smoothing_filter=5)  # filter length is ignored by the reference (model.py:445-448)
    _, p, _ = m(x, {})
    _, sm, _ = m(x, kw)
    assert sm.shape == (meta["n"], 2, 1, p.shape[-1])  # [B,2,1,T], model/model.py:449-457
    assert np.array_equal(sm.cpu().numpy()[:, :, 0], smoothed_from(p.cpu().numpy(), 0.45))
    # gating zeroes exactly the frames whose smoothed decision is 0
    kw2 = dict(kw, filter_signals_by_smo_vad=True)
    _, sm2, est = m(x, kw2)
    e = est.cpu().numpy()
    gate = sm2.cpu().numpy()[:, :, 0][:, :, None, :]
    assert np.all(e[np.broadcast_to(gate == 0, e.shape)] == 0)


@pytest.mark.parametrize("cfg_name", ["with", "without"])
@pytest.mark.parametrize("B,L", [(1, 257), (3, 1000), (2, 4099), (1, 12800)])
def test_against_oracle_seeded(cuda_models, cfg_name, B, L):
    """Ragged / minimum lengths against the fp64 numpy oracle (the checker, never the product), VAD gate on."""
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITH_VAD if cfg_name == "with" else synth.CONFIG_WITHOUT_VAD
    seed = 21
    m = cuda_models(args, seed, 0)
    W = O.OracleWeights(synth.make_state_dict_numpy(args, seed), args, np.float64)
    x = synth.make_mixtures(B, L, 900 + L)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    ref_out, ref_vad, ref_est, _ = O.forward(x, W, dict(kw))
    out, vad, est = m(torch.from_numpy(x).cuda(), dict(kw))
    v = vad.cpu().numpy()
    p_ref = ref_vad.astype(np.float32)
    assert np.abs(v - ref_vad).max() < 1e-3
    check_decisions(v, p_ref, 0.5)
    # very short inputs end in the ragged istft tail (division by a small window envelope, SURVEY appendix A.10), so
    # the absolute waveform tolerance scales with the reference's peak there
    tol = dict(TOL[0], wav=1e-3)
    check_outputs(out.cpu().numpy(), est.cpu().numpy(), v, ref_out.astype(np.float32), ref_est.astype(np.complex64), p_ref, kw, tol,
                  wav_scale=max(1.0, float(np.abs(ref_out).max())))


SWEEP_SHAPES = [(1, 257), (1, 32768), (2, 32767), (3, 33000), (9, 64000), (33, 20000), (130, 4000), (2, 300000), (1, 131072),
                (5, 65536), (300, 16000)]


@pytest.mark.parametrize("seed", [9, 21])
@pytest.mark.parametrize("cfg_name", ["with", "without"])
def test_shape_sweep_against_oracle(cuda_models, cfg_name, seed):
    """The VAD parity gate on odd shapes (tiles straddling utterances, one tile per utterance, T below / above every
    kernel-selection threshold, ragged istft tails), two weight seeds, both configurations, default precision mode,
    against the fp64 oracle: |dp| < 1e-3 on every frame (north_star band) - measured worst case 4e-4 - and the decision
    rule. Batches repeat min(B, 8) distinct utterances; every copy is checked against its oracle result."""
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITH_VAD if cfg_name == "with" else synth.CONFIG_WITHOUT_VAD
    m = cuda_models(args, seed, 0)
    W = O.OracleWeights(synth.make_state_dict_numpy(args, seed), args, np.float64)
    worst = 0.0
    for B, L in SWEEP_SHAPES:
        nd = min(B, 8)
        xd = synth.make_mixtures(nd, L, 4242)
        ref_out, ref_vad, _, _ = O.forward(xd, W, {})
        x = torch.from_numpy(np.tile(xd, ((B + nd - 1) // nd, 1))[:B]).cuda()
        out, vad, _ = m(x, {})
        v, o = vad.cpu().numpy(), out.cpu().numpy()
        assert np.isfinite(o).all()
        idx = np.arange(B) % nd
        dv = np.abs(v - ref_vad[idx]).max()
        worst = max(worst, dv)
        assert dv < 1e-3, (cfg_name, seed, B, L, dv)
        check_decisions(v, ref_vad[idx].astype(np.float32), 0.5)
        tail = (L % 256) if (L % 256) > 200 else 0   # samples only the last frame covers: envelope -> ~1e-8 there
        assert np.abs(o[..., :L - tail] - ref_out[idx][..., :L - tail]).max() <= 5e-4, (cfg_name, seed, B, L)
        assert sisdr_db(o[:nd, :, :L - tail], ref_out[..., :L - tail]) >= 60.0
    assert worst < 7.5e-4, worst      # margin pin: the tolerance band is 1e-3


def test_engines_agree(cuda_models):
    """tcgen05 fp16 engine vs fp32 CUDA-core engine on the same device buffers."""
    args = synth.CONFIG_WITH_VAD
    x = torch.from_numpy(synth.make_mixtures(4, 16000, 4321)).cuda()
    m = cuda_models(args, 31, 7)
    o7, v7, _ = m(x, {})
    m = cuda_models(args, 31, 0)
    o0, v0, _ = m(x, {})
    assert (o7 - o0).abs().max().item() < 5e-4
    assert (v7 - v0).abs().max().item() < 1e-3
    assert sisdr_db(o0.cpu().numpy(), o7.cpu().numpy()) > 60


@pytest.mark.parametrize("cfg_name", ["with", "without"])
@pytest.mark.parametrize("B,L", [(3, 64000), (2, 30000), (5, 9000), (2, 100000), (1, 200000), (2, 400000), (1, 580000)])
def test_fused_residual_kernel_equals_streaming_kernels(cuda_models, cfg_name, B, L):
    """The cluster-resident gate + residual kernel (resid_fused.cu) against k_tf_gate + k_resid<0,1> on the
    same buffers: same arithmetic, different summation grouping of the GroupNorm statistics, so they agree
    to the fp16 operand noise level. Also bit-reproducible run to run (no atomics in the fused kernel)."""
    args = synth.CONFIG_WITH_VAD if cfg_name == "with" else synth.CONFIG_WITHOUT_VAD
    m = cuda_models(args, 33, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW) if cfg_name == "with" else {}
    x = torch.from_numpy(synth.make_mixtures(B, L, 777)).cuda()
    try:
        m.set_option("precision", 1)     # the fused kernel reads fp16 accumulators: the single-pass ("fast") mode
        m.set_option("fused_resid", 0)
        o0, v0, _ = m(x, kw)
        n0 = m.last_launch_count
        m.set_option("fused_resid", 1)
        o1, v1, _ = m(x, kw)
        n1 = m.last_launch_count
        o2, v2, _ = m(x, kw)
    finally:
        m.set_option("fused_resid", 1)
        m.set_option("precision", 0)
    assert n1 < n0, (n0, n1)            # the fused kernel really replaced three launches per block
    assert (o1 - o0).abs().max().item() < 5e-4
    assert sisdr_db(o1.cpu().numpy(), o0.cpu().numpy()) > 60
    if v0.numel():
        # two fp16-noisy evaluations of the same probabilities: each is within 1e-3 of the fp32 reference
        # (test_against_oracle_seeded), so their mutual distance is bounded by 2e-3
        assert (v1.float() - v0.float()).abs().max().item() < 2e-3
    if L >= 32768:
        assert torch.equal(o1, o2)


@pytest.mark.parametrize("B,L", [(3, 64000), (2, 40000), (1, 200000)])
def test_persistent_conv1_equals_one_tile_kernel(cuda_models, B, L):
    """The persistent warp-specialised conv1 kernel (gemm_conv1_persist.cu: double-buffered TMEM, TMA bulk stores)
    against the one-tile-per-CTA kernel (gemm_tc.cu MODE 0) on the same buffers: identical operands and accumulation,
    only the grouping of the statistics' partial sums differs -> agreement to the fp16 operand noise level; and the
    persistent kernel is bit-reproducible run to run."""
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 34, 0)
    x = torch.from_numpy(synth.make_mixtures(B, L, 778)).cuda()
    try:
        m.set_option("conv1_persist", 0)
        o0, v0, _ = m(x, {})
        m.set_option("conv1_persist", 1)
        o1, v1, _ = m(x, {})
        o2, v2, _ = m(x, {})
    finally:
        m.set_option("conv1_persist", 1)
    assert (o1 - o0).abs().max().item() < 5e-4
    assert sisdr_db(o1.cpu().numpy(), o0.cpu().numpy()) > 60
    assert (v1 - v0).abs().max().item() < 2e-3
    assert torch.equal(o1, o2) and torch.equal(v1, v2)


def test_batch_invariance_and_determinism(cuda_models):
    """Utterances are independent: item b of a batch equals the same item run alone up to the fp16
    operand noise (tiles straddle utterances differently, so the statistics' partial sums - and with
    them some fp16 roundings - differ). Repeated runs of the SAME call are bit-identical whenever an
    utterance spans at least one 128-frame tile (L >= 2 s): per-tile statistics are reduced in a fixed
    order and accumulated in double. Shorter inputs (several utterances per tile) use shared-memory
    float atomics for the 3rd+ utterance of a tile and reproduce only to the fp16 noise level."""
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 32, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW)
    x = torch.from_numpy(synth.make_mixtures(5, 40000, 555)).cuda()   # T = 157
    ob, vb, _ = m(x, kw)
    ob2, vb2, _ = m(x, kw)
    assert torch.equal(ob, ob2) and torch.equal(vb, vb2)
    for b in (0, 3, 4):
        o1, v1, _ = m(x[b:b + 1].contiguous(), kw)
        assert (o1[0] - ob[b]).abs().max().item() < 5e-4, (o1[0] - ob[b]).abs().max().item()
        assert (v1[0] - vb[b]).abs().max().item() < 1e-3, (v1[0] - vb[b]).abs().max().item()
    xs = torch.from_numpy(synth.make_mixtures(5, 9000, 556)).cuda()    # T = 36: five utterances share a tile
    os1, vs1, _ = m(xs, kw)
    os2, vs2, _ = m(xs, kw)
    assert (os1 - os2).abs().max().item() < 5e-4 and (vs1 - vs2).abs().max().item() < 1e-3


def test_reproducible_under_disturbed_timing(cuda_models):
    """Race check for the persistent / cluster kernels (mbarrier pipelines, single-buffer TMA refill, DSMEM exchange):
    the same forward repeated while a second stream hammers the memory system must stay bit-identical."""
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 35, 0)
    x = torch.from_numpy(np.tile(synth.make_mixtures(16, 48000, 321), (4, 1))).cuda()   # 64 x 3 s: T = 188, 6-CTA clusters
    side = torch.cuda.Stream()
    junk = torch.empty(128 << 20, dtype=torch.uint8, device="cuda")
    ref = None
    for i in range(6):
        if i % 2 == 1:
            with torch.cuda.stream(side):
                for _ in range(10):
                    junk.fill_(i)
        out, vad, _ = m(x, {})
        torch.cuda.synchronize()
        if ref is None:
            ref = (out.clone(), vad.clone())
        else:
            assert torch.equal(out, ref[0]) and torch.equal(vad, ref[1]), f"run {i} differs"


def test_forward_host_equals_forward(cuda_models):
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 33, 0)
    xh = torch.from_numpy(synth.make_mixtures(3, 8000, 77))
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    out_h, vad_h = m.forward_host(xh, kw)
    out_d, vad_d, _ = m(xh.cuda(), kw)
    assert not out_h.is_cuda
    assert (out_h - out_d.cpu()).abs().max().item() < 5e-4, (out_h - out_d.cpu()).abs().max().item()
    assert (vad_h - vad_d.cpu()).abs().max().item() < 1e-3


def test_forward_host_stream_equals_forward(cuda_models):
    """The asynchronous two-slot host pipeline (forward_host_submit / forward_host_stream) returns, per batch and in
    order, what the synchronous device forward returns - including ragged last batches and slot reuse."""
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 31, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    batches = [torch.from_numpy(synth.make_mixtures(n, 20000, 900 + i)) for i, n in enumerate((3, 2, 4, 1, 3))]
    got = list(m.forward_host_stream(batches, kw))
    assert len(got) == len(batches)
    for xb, (o, v) in zip(batches, got):
        od, vd, _ = m(xb.cuda(), kw)
        assert not o.is_cuda and o.is_pinned()
        assert (o - od.cpu()).abs().max().item() < 5e-4 and (v - vd.cpu()).abs().max().item() < 1e-3
    # slot protocol errors are reported, not swallowed
    f = m.forward_host_submit(batches[0], kw, slot=0)
    with pytest.raises(Exception):
        m.forward_host_submit(batches[1], kw, slot=0)
    f.result()


def test_minmax_normalize_bit_exact(cuda_models):
    """Device pre-processing (SURVEY 8(f) rank 1): the min-max normalisation of only_inference.py:81, batched,
    against the reference's own numpy expression - bit-exact, including ragged batches and the constant-signal NaN."""
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    rng = np.random.default_rng(7)
    B, L = 5, 50021
    x = (rng.standard_normal((B, L)) * rng.uniform(0.01, 30.0, (B, 1))).astype(np.float32)
    x[1] = -np.abs(x[1]) - 3.0            # all-negative utterance
    x[2] = np.round(x[2] * 100.0)         # int16-like magnitudes, as scipy.io.wavfile.read yields
    ref = np.stack([1.8 * (a - a.min()) / (a.max() - a.min()) - 0.9 for a in x])     # only_inference.py:81 verbatim
    got = m.minmax_normalize(torch.from_numpy(x).cuda()).cpu().numpy()
    assert got.dtype == np.float32 and np.array_equal(got, ref.astype(np.float32))
    assert got.min() == np.float32(-0.9) and abs(got.max() - 0.9) < 1e-6
    # ragged: extrema over the valid part only, zeros behind it
    lens = np.array([L, 1234, 40000, 7, L - 1])
    xr = x.copy()
    for b, n in enumerate(lens):
        xr[b, n:] = 1e9                   # garbage in the padding must not matter
    got = m.minmax_normalize(torch.from_numpy(xr).cuda(), lens).cpu().numpy()
    for b, n in enumerate(lens):
        a = x[b, :n]
        assert np.array_equal(got[b, :n], (1.8 * (a - a.min()) / (a.max() - a.min()) - 0.9).astype(np.float32))
        assert not got[b, n:].any()
    # constant signal: 0 / 0 like the reference
    c = torch.full((1, 1000), 0.25, device="cuda")
    assert torch.isnan(m.minmax_normalize(c)).all()


def test_sisdr_kernel_matches_reference_formula(cuda_models):
    """septfa_sisdr (one-pass moments in double) against calc_sisdr of model/combined_loss.py:16-56 evaluated
    element-wise in float64 on the host, over 0 .. 60 dB, both zero_mean settings; and the docstring example."""
    from septfa_b200.pit import calc_sisdr
    rng = np.random.default_rng(11)
    n = 48000
    tgt = rng.standard_normal((6, 2, n)).astype(np.float32) * 0.1 + 0.02
    noise = rng.standard_normal((6, 2, n)).astype(np.float32) * 0.1
    snr = np.array([0.0, 10.0, 20.0, 30.0, 45.0, 60.0])[:, None, None]
    est = (0.7 * tgt + noise * 10.0 ** (-snr / 20.0)).astype(np.float32)

    def ref_formula(p, t, zero_mean):
        p, t = p.astype(np.float64), t.astype(np.float64)
        eps = np.finfo(np.float32).eps
        if zero_mean:
            p, t = p - p.mean(-1, keepdims=True), t - t.mean(-1, keepdims=True)
        alpha = ((p * t).sum(-1, keepdims=True) + eps) / ((t ** 2).sum(-1, keepdims=True) + eps)
        ts = alpha * t
        return 10 * np.log10(((ts ** 2).sum(-1) + eps) / (((ts - p) ** 2).sum(-1) + eps))

    for zm in (True, False):
        got = calc_sisdr(torch.from_numpy(est).cuda(), torch.from_numpy(tgt).cuda(), zero_mean=zm).cpu().numpy()
        assert got.shape == (6, 2)
        assert np.abs(got - ref_formula(est, tgt, zm)).max() < 1e-2, (zm, got, ref_formula(est, tgt, zm))
    ex = calc_sisdr(torch.tensor([2.5, 0.0, 2.0, 8.0]).cuda(), torch.tensor([3.0, -0.5, 2.0, 7.0]).cuda(), zero_mean=False)
    assert abs(ex.item() - 18.4030) < 1e-3            # the example in the reference's docstring


def test_error_behaviour(cuda_models):
    m = cuda_models(synth.CONFIG_WITH_VAD, 33, 0)
    with pytest.raises(AssertionError):           # model/model.py:406
        m(torch.zeros(1, 2, 4000).cuda())
    with pytest.raises(KeyError):                 # missing inference_kw key, model/model.py:445-456
        m(torch.zeros(1, 4000).cuda(), {"filter_signals_by_smo_vad": True})
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 4000))                   # CPU tensor: no fallback
    from septfa_b200.lib import SeptfaError
    with pytest.raises(SeptfaError):
        m(torch.zeros(1, 200).cuda())             # shorter than the reflect padding


def test_online_driver_matches_reference(cuda_models):
    """OnlineSaving.calc_online: two streams as ONE batch vs the reference run once per stream."""
    from septfa_b200.online import OnlineSaving
    from septfa_b200.pit import PITLossWrapper
    g, meta = load_golden("online_with_vad_6s")
    m = cuda_models(meta["args"], meta["weight_seed"], 0)
    x = np.concatenate([synth.make_mixtures(1, meta["length"], meta["base_seed"] + s) for s in range(meta["n_streams"])])
    o = OnlineSaving(m, "/tmp/septfa_online_test", PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt"))
    o.num_save_samples = 0
    sig = o.calc_online(torch.from_numpy(x).cuda(), "n", 0, dict(meta["kw"])).cpu().numpy()
    ref = g["online_signal"]
    assert sig.shape == ref.shape
    for s in range(ref.shape[0]):
        for hop in range(ref.shape[-1] // 16000):
            a, r = sig[s, :, hop * 16000:(hop + 1) * 16000], ref[s, :, hop * 16000:(hop + 1) * 16000]
            assert np.abs(a - r).max() <= 5e-4, (s, hop, np.abs(a - r).max(), np.abs(a[::-1] - r).max())


def test_pit_kernel(cuda_models):
    from septfa_b200.pit import PITLossWrapper
    m = cuda_models(synth.CONFIG_WITH_VAD, 33, 0)
    torch.manual_seed(1)
    tgt = torch.randn(6, 2, 20000).cuda()
    est = tgt.clone()
    est[[1, 4]] = est[[1, 4]][:, [1, 0]]
    est += 0.05 * torch.randn_like(est)
    w = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt", per_stream=True, handle_provider=m._handle)
    loss, idx = w(est, tgt, return_incides=True)
    assert idx.cpu().tolist() == [[0, 1], [1, 0], [0, 1], [0, 1], [1, 0], [0, 1]]
    ref = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt", per_stream=True)(est.cpu(), tgt.cpu())
    assert abs(loss.item() - ref.item()) < 1e-5


def test_full_size_batch_against_oracle(cuda_models):
    """cfg2 size (256 x 4 s, VAD gate on): the batch holds 32 distinct utterances (8 copies each, interleaved so that
    copies sit in different tiles); EVERY one of the 256 results is compared with the oracle's result for its
    utterance - probabilities, decisions, gated waveforms. The golden utterance of cfg1 is one of the 32."""
    from oracle import septfa_oracle as O
    g, meta = load_golden("cfg1_with_vad_4s")
    m = cuda_models(meta["args"], meta["weight_seed"], 0)
    B, nd, L = 256, 32, 64000
    xd = synth.make_mixtures(nd, L, 9000)
    xd[13] = synth.make_mixtures(1, L, meta["base_seed"])[0]
    kw = dict(meta["kws"][0])
    W = O.OracleWeights(synth.make_state_dict_numpy(meta["args"], meta["weight_seed"]), meta["args"], np.float32)
    ref_out, ref_vad, _, _ = O.forward(xd, W, dict(kw))
    assert np.abs(ref_out[13] - g["kw0_out"][0]).max() < 2e-5 and np.abs(ref_vad[13] - g["kw0_vad"][0]).max() < 2e-5   # oracle == reference
    idx = np.arange(B) % nd
    m.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)
    try:
        out, vad, est = m(torch.from_numpy(xd[idx]).cuda(), kw)
    finally:
        m.materialize.update(estimated_stfts=True, mask_per_speaker=True, spectrum=True, masks_b=True)
    assert est is None
    o, v = out.cpu().numpy(), vad.cpu().numpy()
    assert np.isfinite(o).all() and np.isfinite(v).all()
    assert np.abs(v - ref_vad[idx]).max() < 1e-3, np.abs(v - ref_vad[idx]).max()
    check_decisions(v, ref_vad[idx], kw["threshold_activated_vad"])
    skipped = check_outputs(o, None, v, ref_out[idx], None, ref_vad[idx], kw, TOL[0])
    assert skipped <= 4, skipped      # frames whose gate legitimately differs (in-band decisions): a handful at most
    assert np.abs(o[13] - g["kw0_out"][0]).max() <= 5e-4


def test_online_many_streams_equals_per_stream_runs(cuda_models):
    """S streams as one batch == each stream driven on its own (per-stream permutation decisions)."""
    from septfa_b200.online import OnlineSaving
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 41, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    x = torch.from_numpy(synth.make_mixtures(6, 80000, 700)).cuda()   # 5 s -> 3 hops
    o = OnlineSaving(m, "/tmp/septfa_online_test2")
    o.num_save_samples = 0
    batch = o.calc_online(x, "n", 0, dict(kw))
    perms_batch = o.last_perms.cpu().numpy()
    assert batch.shape == (6, 2, 48000) and perms_batch.shape == (3, 6, 2)
    for s in (0, 5):
        single = o.calc_online(x[s:s + 1].contiguous(), "n", 0, dict(kw))
        # same permutation decisions, waveforms equal up to the fp16 batch-placement noise
        assert np.array_equal(o.last_perms.cpu().numpy()[:, 0], perms_batch[:, s])
        assert (single[0] - batch[s]).abs().max().item() < 5e-4


def test_online_1024_streams_equal_per_stream_runs_and_oracle(cuda_models):
    """cfg3 size: 1024 concurrent streams (16 distinct mixtures x 64 copies) driven as ONE batch for 3 hops. Every
    stream's permutation decisions and emitted audio must equal those of its mixture driven in a 16-stream batch, and
    two of the distinct streams are checked against the oracle's calc_online (the reference driver's semantics)."""
    from oracle import septfa_oracle as O
    from septfa_b200.online import OnlineSaving
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 41, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    xd = synth.make_mixtures(16, 80000, 700)                       # 5 s -> 3 hops
    o = OnlineSaving(m, "/tmp/septfa_online_test1024")
    o.num_save_samples = 0
    small = o.calc_online(torch.from_numpy(xd).cuda(), "n", 0, dict(kw)).cpu().numpy()
    perms_small = o.last_perms.cpu().numpy()                       # [hops, 16, 2]
    idx = np.arange(1024) % 16
    big = o.calc_online(torch.from_numpy(xd[idx]).cuda(), "n", 0, dict(kw)).cpu().numpy()
    perms_big = o.last_perms.cpu().numpy()
    assert big.shape == (1024, 2, 48000) and perms_big.shape == (3, 1024, 2)
    assert np.array_equal(perms_big, perms_small[:, idx])
    assert np.abs(big - small[idx]).max() < 5e-4, np.abs(big - small[idx]).max()
    W = O.OracleWeights(synth.make_state_dict_numpy(args, 41), args, np.float32)
    ref_sig, ref_perms = O.calc_online(xd[[0, 7]], W, dict(kw))
    assert np.array_equal(ref_perms, perms_small[:, [0, 7]])
    assert np.abs(small[[0, 7]] - ref_sig).max() < 1e-3, np.abs(small[[0, 7]] - ref_sig).max()


def test_precision_modes(cuda_models):
    """Option "precision": the split-precision (three-pass) contractions reproduce the oracle to fp32 level, the
    single-pass mode to the fp16 level; AUTO picks the split for config_without_vad (its stream is never re-normalised)."""
    from oracle import septfa_oracle as O
    x = synth.make_mixtures(2, 33000, 4242)
    for args, auto_is_accurate in ((synth.CONFIG_WITH_VAD, False), (synth.CONFIG_WITHOUT_VAD, True)):
        m = cuda_models(args, 9, 0)
        W = O.OracleWeights(synth.make_state_dict_numpy(args, 9), args, np.float64)
        _, ref_vad, _, _ = O.forward(x, W, {})
        err = {}
        try:
            for prec in (0, 1, 2):
                m.set_option("precision", prec)
                err[prec] = float(np.abs(m(torch.from_numpy(x).cuda(), {})[1].cpu().numpy() - ref_vad).max())
        finally:
            m.set_option("precision", 0)
        assert err[2] < 1e-4 and err[1] < 2e-3, err
        assert (err[0] == err[2]) if auto_is_accurate else (err[0] == err[1]), err
    with pytest.raises(Exception):
        m.set_option("precision", 3)
        m(torch.from_numpy(x).cuda(), {})
    m.set_option("precision", 0)


@pytest.mark.parametrize("B,L", [(3, 64000), (2, 40000), (1, 200000), (5, 33000), (1, 33024), (7, 48000)])
def test_tensor_core_depthwise_kernel_equals_cuda_core_producer(cuda_models, B, L):
    """dconv_mma2.cu (depthwise conv as block-diagonal tcgen05 GEMMs on the plane layout of p, edge rows corrected; CTA
    pairs with the res_out weights resident) against gemm_tc.cu MODE 1 (depthwise conv on the CUDA cores) on the same
    buffers: same network up to the fp16 rounding of the folded taps; even and odd tile counts, utterance boundaries
    inside tiles, a tile pair with an empty tile; run-to-run bit-reproducible; and both within the band of the oracle."""
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 34, 0)
    xh = synth.make_mixtures(B, L, 779)
    x = torch.from_numpy(xh).cuda()
    try:
        m.set_option("dconv_mma", 0)
        o0, v0, _ = m(x, {})
        m.set_option("dconv_mma", 1)
        o1, v1, _ = m(x, {})
        o2, v2, _ = m(x, {})
    finally:
        m.set_option("dconv_mma", 1)
    tail = (L % 256) if (L % 256) > 200 else 0     # samples only the last frame covers: overlap-add envelope ~1e-8 (SURVEY A.10)
    assert (o1 - o0)[..., :L - tail].abs().max().item() < 5e-4
    assert (v1 - v0).abs().max().item() < 1e-3
    assert torch.equal(o1, o2) and torch.equal(v1, v2)
    W = O.OracleWeights(synth.make_state_dict_numpy(args, 34), args, np.float64)
    _, ref_vad, _, _ = O.forward(xh, W, {})
    assert np.abs(v1.cpu().numpy() - ref_vad).max() < 1e-3


def test_retired_kernel_switches_are_refused():
    """Kernel-selection switches that only selected a path slower on every measured workload are gone:
    septfa_set_option refuses their names as unknown options (SEPTFA_E_INVALID), the model does not keep a refused
    name, and its forward is unchanged afterwards."""
    from conftest import build_cuda_model
    from septfa_b200.lib import SeptfaError
    m = build_cuda_model(synth.CONFIG_WITH_VAD, 34)   # not the shared cache: the options below go to this model only
    x = torch.from_numpy(synth.make_mixtures(2, 64000, 785)).cuda()
    o0, v0, _ = m(x, {})
    for name in ("dconv_pair", "dconv_w_tmap", "dconv_cluster", "dconv_desc_swap", "conv1_wres", "dconv_late_trigger",
                 "fused_pdl"):
        for value in (0, 1, 2):
            with pytest.raises(SeptfaError, match=f"^septfa error -1: unknown option {name}$"):
                m.set_option(name, value)
    o1, v1, _ = m(x, {})
    assert torch.equal(o0, o1) and torch.equal(v0, v1)


@pytest.mark.parametrize("B,L", [(3, 64000), (1, 200000), (5, 33000)])
def test_tf32_pair_conv1_equals_persistent_conv1(cuda_models, B, L):
    """gemm_conv1_pair.cu (blocks 1 .. n-1: the fp32 stream is the TF32 A operand itself, fetched by TMA; CTA pairs with the
    TF32 weight image resident; normalisation applied to the accumulator) against gemm_conv1_persist.cu (producer warps
    normalise and round to fp16): same precision class (11 significant bits in both operands), different roundings; both
    within the band of the oracle, bit-reproducible."""
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 34, 0)
    xh = synth.make_mixtures(B, L, 783)
    x = torch.from_numpy(xh).cuda()
    try:
        m.set_option("conv1_pair", 0)
        o0, v0, _ = m(x, {})
        m.set_option("conv1_pair", 2)       # 2 = at any size (1 = only from ~2.5 tiles per SM on)
        o1, v1, _ = m(x, {})
        o2, v2, _ = m(x, {})
    finally:
        m.set_option("conv1_pair", 1)
    tail = (L % 256) if (L % 256) > 200 else 0
    assert (o1 - o0)[..., :L - tail].abs().max().item() < 5e-4
    assert (v1 - v0).abs().max().item() < 1e-3
    assert not torch.equal(o1, o0)
    assert torch.equal(o1, o2) and torch.equal(v1, v2)
    W = O.OracleWeights(synth.make_state_dict_numpy(args, 34), args, np.float64)
    _, ref_vad, _, _ = O.forward(xh, W, {})
    assert np.abs(v1.cpu().numpy() - ref_vad).max() < 1e-3
    assert np.abs(v0.cpu().numpy() - ref_vad).max() < 1e-3


def test_half_stream_mode_is_opt_in_and_close(cuda_models):
    """Option "stream_half" (off by default): blocks 1 .. n-1 carry the residual stream as fp16 - written by the residual
    kernel, read by TMA as the A operand of gemm_conv1_tma.cu. 11 % faster, but the stream's rounding random-walks through
    all 24 blocks (worst VAD error on the shape sweep 9.5e-4 against 2.1e-4), so it stays outside the default parity
    envelope: checked here against the default mode with its own, looser bounds."""
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITH_VAD
    m = cuda_models(args, 31, 0)
    xh = synth.make_mixtures(3, 64000, 4242)
    x = torch.from_numpy(xh).cuda()
    o0, v0, _ = m(x, {})
    try:
        m.set_option("stream_half", 1)
        o1, v1, _ = m(x, {})
        o2, v2, _ = m(x, {})
    finally:
        m.set_option("stream_half", 0)
    o3, v3, _ = m(x, {})
    assert torch.equal(o0, o3) and torch.equal(v0, v3)          # the default path is unchanged by the round trip
    assert torch.equal(o1, o2) and torch.equal(v1, v2)
    assert not torch.equal(o0, o1)                              # the option does select another path
    W = O.OracleWeights(synth.make_state_dict_numpy(args, 31), args, np.float64)
    ref_out, ref_vad, _, _ = O.forward(xh, W, {})
    assert np.abs(v1.cpu().numpy() - ref_vad).max() < 2e-3
    assert sisdr_db(o1.cpu().numpy(), ref_out) >= 60.0


def test_host_16bit_formats(cuda_models):
    """septfa_forward_host_submit_fmt: int16 PCM input (only_inference.py:68-81 on the device: astype float32 + min-max
    normalisation, bit-identical to numpy) and fp16 output (save_audio's `-ps 16` cast, utlis_inference.py:30-32)."""
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    rng = np.random.default_rng(5)
    pcm = np.clip(np.round(synth.make_mixtures(3, 20000, 910) * 20000.0 + rng.integers(-3, 4, (3, 20000))), -32768, 32767).astype(np.int16)
    audio = pcm.astype(np.float32)                                                     # only_inference.py:69
    norm = np.stack([1.8 * (a - a.min()) / (a.max() - a.min()) - 0.9 for a in audio])  # only_inference.py:81
    ref_out, ref_vad, _ = m(torch.from_numpy(norm.astype(np.float32)).cuda(), kw)
    f = m.forward_host_submit(torch.from_numpy(pcm), kw, slot=0, out_dtype=torch.float16)
    out16, vad = f.result()
    assert out16.dtype == torch.float16 and out16.shape == (3, 2, 20000) and not out16.is_cuda
    # same device arithmetic on bit-identical inputs -> identical fp32 waveforms; the output is their fp16 rounding
    assert torch.equal(out16, ref_out.cpu().to(torch.float16))
    assert torch.equal(vad, ref_vad.cpu())
    # fp32 in / fp16 out and int16 in / fp32 out
    o2, _ = m.forward_host_submit(torch.from_numpy(norm.astype(np.float32)), kw, slot=1, out_dtype=torch.float16).result()
    assert torch.equal(o2, out16)
    o3, _ = m.forward_host_submit(torch.from_numpy(pcm), kw, slot=0).result()
    assert o3.dtype == torch.float32 and torch.equal(o3, ref_out.cpu())


def test_utterance_longer_than_200_s(cuda_models):
    """A 210 s file (T = 13126 frames): every kernel's shared memory is independent of T (the streaming gate kernel used
    to keep its per-frame means in shared memory and failed beyond ~190 s). Checked against the oracle."""
    from oracle import septfa_oracle as O
    args = synth.CONFIG_WITHOUT_VAD
    m = cuda_models(args, 4, 0)
    L = 210 * 16000
    x = np.tile(synth.make_mixtures(1, 160000, 31), (1, 21))[:, :L].copy()
    W = O.OracleWeights(synth.make_state_dict_numpy(args, 4), args, np.float32)
    ref_out, ref_vad, _, _ = O.forward(x, W, {})
    m.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)
    try:
        out, vad, _ = m(torch.from_numpy(x).cuda(), {})
    finally:
        m.materialize.update(estimated_stfts=True, mask_per_speaker=True, spectrum=True, masks_b=True)
    assert np.abs(vad.cpu().numpy() - ref_vad).max() < 1e-3
    assert np.abs(out.cpu().numpy() - ref_out).max() <= 5e-4
    from septfa_b200.lib import SeptfaError
    with pytest.raises(SeptfaError):
        m(torch.zeros(40000, 300).cuda())          # B above the per-call limit is rejected with a clear message


def test_unusual_weights_against_oracle(cuda_models):
    """Weights outside the benign random-init ranges: PReLU slopes > 1 and < 0 (the min-form / general PReLU code paths),
    a reg1 gamma that is (nearly) zero (the tensor-core depthwise kernel declines, the CUDA-core producer clamps), large
    weight_g. Checked against the fp64 oracle; probabilities stay within the band."""
    from oracle import septfa_oracle as O
    from conftest import build_cuda_model
    args = synth.CONFIG_WITH_VAD
    sd = synth.make_state_dict(args, 55)
    for i in range(24):
        sd[f"TCN.TCN.{i}.nonlinearity1.weight"].fill_(1.3 if i % 3 == 0 else (-0.2 if i % 3 == 1 else 0.25))
        sd[f"TCN.TCN.{i}.nonlinearity2.weight"].fill_(1.7 if i % 3 == 1 else (-0.1 if i % 3 == 2 else 0.3))
    sd["TCN.TCN.5.reg1.weight"][17] = 0.0
    sd["TCN.TCN.9.reg1.weight"][3] = 1e-6
    sd["TCN.TCN.2.res_out.weight_g"] *= 6.0
    sd["TCN.TCN.11.conv1d.weight_g"] *= 5.0
    import contextlib, io
    from septfa_b200.model import SeparationModel
    with contextlib.redirect_stdout(io.StringIO()):
        m = SeparationModel(**args)
    m.load_state_dict(sd, strict=True)
    m.eval().cuda()
    x = synth.make_mixtures(3, 40000, 56)
    W = O.OracleWeights({k: v.numpy() for k, v in sd.items()}, args, np.float64)
    ref_out, ref_vad, _, _ = O.forward(x, W, {})
    out, vad, _ = m(torch.from_numpy(x).cuda(), {})
    assert torch.isfinite(out).all()
    assert np.abs(vad.cpu().numpy() - ref_vad).max() < 1e-3, np.abs(vad.cpu().numpy() - ref_vad).max()
    assert sisdr_db(out.cpu().numpy(), ref_out) >= 60.0


@pytest.mark.parametrize("similarity", [False, True])
def test_known_targets_driver_matches_reference(cuda_models, similarity):
    """OnlineSaving (known targets), model/online_class_known_targets.py:85-154, against golden vectors produced by the
    reference's own class (driven through a 6-tuple shim, the file being stale: tests/golden/make_golden.py): left
    padding by 2 s, the remainder tail padding, per-window PIT against the true sources (or the L1 similarity stitch),
    the final PIT of the stitched signal, and both SI-SDR figures."""
    from septfa_b200.evaluate import pairwise_neg_sisdr
    from septfa_b200.online import OnlineSavingKnownTargets
    from septfa_b200.pit import PITLossWrapper
    g, meta = load_golden("online_known_sim_4s" if similarity else "online_known_pit_4s")
    m = cuda_models(meta["args"], meta["weight_seed"], 0)
    L = meta["length"]
    x = torch.from_numpy(synth.make_mixtures(1, L, meta["base_seed"]))
    rng = np.random.default_rng(meta["base_seed"])
    w = torch.from_numpy(rng.uniform(0.3, 0.7, size=(1, 1, L)).astype(np.float32))
    tgt = torch.cat([x[:, None] * w, x[:, None] * (1 - w)], dim=1)
    crit_sep = PITLossWrapper(pairwise_neg_sisdr, pit_from="pw_mtx")                       # test.py:49-56
    crit_sim = PITLossWrapper(torch.nn.L1Loss(), pit_from="pw_pt") if similarity else None
    drv = OnlineSavingKnownTargets(crit_sep, m, "/tmp/septfa_online_test3", "cuda", crit_sim)   # the reference's argument order
    sig = drv.calc_online(x.cuda(), tgt.cuda(), "n", 0).cpu().numpy()
    ref = g["online_signal"]
    # left-padded by 2 s (:92-93), then padded by the *remainder* (102000 - 48000) % 16000 = 6000 (:94-97, a quirk of
    # the reference: it pads by the remainder, not up to the next hop) -> 108000 -> floor(60000 / 16000) + 1 = 4 hops
    assert sig.shape == ref.shape == (1, 2, 4 * 16000)
    assert np.abs(sig - ref).max() <= 5e-4, np.abs(sig - ref).max()
    assert len(drv.online_sisdr) == 1 and len(drv.reference_sisdr) == 1
    assert abs(drv.online_sisdr[0] - float(g["online_sisdr"][0])) < 2e-2
    assert abs(drv.reference_sisdr[0] - float(g["reference_sisdr"][0])) < 2e-2
    # criteria the device stitch does not implement are refused, not silently replaced
    with pytest.raises(NotImplementedError):
        OnlineSavingKnownTargets(crit_sep, m, "/tmp/x", "cuda", PITLossWrapper(torch.nn.MSELoss(), pit_from="pw_pt"))


def test_evaluation_helpers_match_reference(cuda_models):
    """septfa_b200.evaluate against the reference's helpers: the pairwise negative SI-SDR matrix + PIT of test.py's
    separation criterion, the mask-based simple VAD; the VAD accuracy. The expected values are stored in
    tests/golden/reference_helpers.npz: computed by the reference's own functions where it can be imported, otherwise by
    tests/golden/make_helper_golden.py's restatement of their code, which shares nothing with septfa_b200."""
    from septfa_b200 import evaluate as E
    g, _ = load_golden("reference_helpers")
    rng = np.random.default_rng(3)          # the inputs tests/golden/make_helper_golden.py gave the reference helpers
    tgt = torch.from_numpy(rng.standard_normal((5, 2, 32000)).astype(np.float32) * 0.1)
    est = tgt.clone()
    est[[1, 3]] = est[[1, 3]][:, [1, 0]]
    est = est * 0.8 + 0.03 * torch.from_numpy(rng.standard_normal(est.shape).astype(np.float32))
    masks = torch.from_numpy(rng.random((3, 2, 257, 40), dtype=np.float32) * rng.random((3, 2, 1, 40), dtype=np.float32))
    got_pw = E.pairwise_neg_sisdr(est.cuda(), tgt.cuda()).cpu().numpy()
    assert np.abs(got_pw - g["eval_pw"]).max() < 1e-2
    loss, reordered, idx = E.pit_sisdr(est.cuda(), tgt.cuda())
    assert np.array_equal(idx.cpu().numpy(), g["eval_idx"]) and abs(loss.item() - g["eval_loss"].item()) < 1e-2
    mix = tgt.sum(dim=1)
    rep = E.separation_report(mix.cuda(), est.cuda(), tgt.cuda())
    assert np.abs(rep["si_sdr"].cpu().numpy() - g["eval_si_sdr"]).max() < 1e-2
    assert np.abs(rep["si_sdr_start"].cpu().numpy() - g["eval_si_sdr_start"]).max() < 1e-2
    assert np.array_equal(E.simple_vad_from_masks(masks.cuda()).cpu().numpy(), g["eval_vad"])
    p = torch.rand(4, 2, 50)
    t = (torch.rand(4, 2, 50) > 0.5).float()
    acc = E.vad_accuracy(p.cuda(), t.cuda())
    d = (p > 0.5).float()
    assert abs(acc[0].item() - (d == t).float().mean().item()) < 1e-6
    assert abs(acc[1].item() - (d[:, 0] == t[:, 0]).float().mean().item()) < 1e-6


def test_inference_cli_end_to_end(cuda_models, tmp_path):
    """`python -m septfa_b200.inference` (only_inference.py:27-137): a synthetic stereo int16 wav and a synthetic .pth in
    the checkpoint layout of only_inference.py:49-55, flags -c -r -pm -sp -o -ps -ikw; the written wav files are compared
    with what the UNMODIFIED reference script wrote for the same inputs (tests/golden/cli_with_vad_ps32.npz)."""
    import json
    from scipy.io.wavfile import read, write
    from septfa_b200 import inference
    g, meta = load_golden("cli_with_vad_ps32")
    wav, ckpt, cfg = tmp_path / "mix.wav", tmp_path / "model_with_vad.pth", tmp_path / "config.json"
    write(str(wav), 16000, synth.make_cli_wav(meta["weight_seed"], fs=16000))
    torch.save(synth.make_checkpoint(meta["args"], meta["weight_seed"]), str(ckpt))
    cfg.write_text(json.dumps({"name": "t", "arch": {"type": "SeparationModel", "args": meta["args"]}}))
    out_dir = tmp_path / "out"
    ikw = json.dumps({"filter_signals_by_smo_vad": True})
    out, vad = inference.main(["-c", str(cfg), "-r", str(ckpt), "-pm", str(wav), "-sp", str(out_dir), "-o", "", "-ps", "32",
                               "-ikw", ikw, "-d", "0"])
    assert out.shape == (1, 2, 48000)
    for name in ("Mixed_0", "Speaker_0", "Speaker_1"):
        sr, a = read(str(out_dir / f"{name}.wav"))
        assert sr == 16000 and a.dtype == np.float32
        tol = 1e-6 if name == "Mixed_0" else 5e-4
        assert np.abs(a - g[name]).max() <= tol, (name, np.abs(a - g[name]).max())
    # online mode (-o non-empty, the reference's bool-of-string flag) writes the stitched signals and the per-window dumps
    inference.main(["-c", str(cfg), "-r", str(ckpt), "-pm", str(wav), "-sp", str(out_dir), "-o", "1", "-ps", "16", "-ikw", ikw])
    for f in ("online_results/online_signal0.wav", "online_results/online_signal1.wav", "online_results/ref_mix.wav",
              "online_results/indx_0/mixed.wav", "online_results/indx_0/output_0.wav", "online_results/indx_0/output_1.wav"):
        assert (out_dir / f).exists(), f
    sr, a16 = read(str(out_dir / "Speaker_0.wav"))
    assert a16.dtype == np.int16                      # -ps 16: 16-bit PCM (the reference hands float16 to scipy, which raises)
    assert np.abs(a16 / 32767.0 - g["Speaker_0"]).max() < 1e-3
    sr, w0 = read(str(out_dir / "online_results/indx_0/output_0.wav"))
    assert w0.shape == (48000,) and np.isfinite(w0).all()
    # an 8 kHz input is resampled (the reference's own resampling branch ends in a TypeError at only_inference.py:82)
    wav8 = tmp_path / "mix8.wav"
    write(str(wav8), 8000, synth.make_cli_wav(3, fs=8000)[:, 0].copy())
    x8 = inference.read_mixture(str(wav8))
    assert x8.shape == (1, 48000) and abs(x8.max().item() - 0.9) < 1e-6 and abs(x8.min().item() + 0.9) < 1e-6
    # save_vad (Our_utils/utlis_inference.py:39-46)
    inference.save_vad(vad, str(out_dir / "vad"))
    assert any((out_dir / "vad").iterdir())
    # checkpoint loader: the 'state_dict' of a reference-layout checkpoint, incl. numpy scalars in monitor_best
    ck = synth.make_checkpoint(meta["args"], 1)
    ck["monitor_best"] = np.float64(3.5)
    torch.save(ck, str(tmp_path / "np.pth"))
    assert len(inference.load_checkpoint_state_dict(str(tmp_path / "np.pth"))) == 719


def test_graphed_forward_equals_eager(cuda_models):
    """SeparationModel.graphed (septfa_graph_capture / _launch): the forward of one small request replayed as a CUDA
    graph gives what the eager launch sequence gives, for successive inputs, and stays correct after eager calls in between."""
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    xs = torch.from_numpy(synth.make_mixtures(3, 64000, 4100)).cuda()
    g = m.graphed(1, 64000, kw)
    assert g.num_nodes > 70
    for i in range(3):
        out, vad = g(xs[i:i + 1])
        out, vad = out.clone(), vad.clone()
        eo, ev, _ = m(xs[i:i + 1].contiguous(), kw)
        assert (out - eo).abs().max().item() < 5e-4 and (vad - ev).abs().max().item() < 1e-3
    o1 = g(xs[0:1])[0].clone()
    o2 = g(xs[0:1])[0].clone()
    assert torch.equal(o1, o2)
    g8 = m.graphed(8, 16000, {})
    x8 = torch.from_numpy(synth.make_mixtures(8, 16000, 4200)).cuda()
    out8, vad8 = g8(x8)
    e8, v8, _ = m(x8, {})
    assert (out8 - e8).abs().max().item() < 5e-4 and (vad8 - v8).abs().max().item() < 1e-3


def test_separate_files_batched_pcm_pipeline(cuda_models, tmp_path):
    """septfa_b200.inference.separate_files: wav files -> int16 PCM batches -> device-side astype/normalise -> forward ->
    fp16/fp32 -> wav files; equal to the single-file path of only_inference.py per file."""
    from scipy.io.wavfile import read, write
    from septfa_b200 import inference
    m = cuda_models(synth.CONFIG_WITH_VAD, 31, 0)
    kw = {"filter_signals_by_smo_vad": True}
    paths = []
    for i, n in enumerate((20000, 20000, 20000, 31000)):
        pcm = np.round(synth.make_mixture(i, n, 6000) * 25000.0).astype(np.int16)
        pth = tmp_path / f"f{i}.wav"
        write(str(pth), 16000, pcm)
        paths.append(str(pth))
    vads = inference.separate_files(m, paths, str(tmp_path / "sep"), kw, precision_save=32, batch=2)
    assert set(vads) == set(paths)
    full_kw = dict(synth.DEFAULT_INFERENCE_KW, **kw)
    for pth in paths:
        x = inference.read_mixture(pth).cuda()
        ref_out, ref_vad, _ = m(x, full_kw)
        for s_ in range(2):
            sr, a = read(str(tmp_path / "sep" / f"{__import__('pathlib').Path(pth).stem}_Speaker_{s_}.wav"))
            assert sr == 16000 and a.dtype == np.float32
            assert np.abs(a - ref_out[0, s_].cpu().numpy()).max() < 5e-4
        assert (vads[pth] - ref_vad[0].cpu()).abs().max().item() < 1e-3




def test_check_finite_guard(cuda_models):
    """SeparationModel.check_finite (opt-in): a forward that returns non-finite samples raises instead of handing them on
    (here forced with a NaN in one input sample; the motivating case is fp16 overflow between the block kernels)."""
    m = cuda_models(synth.CONFIG_WITH_VAD, 9, 0)
    x = torch.from_numpy(synth.make_mixtures(2, 33000, 77)).cuda()
    m.check_finite = True
    try:
        out, _, _ = m(x, {})
        assert torch.isfinite(out).all()
        x[1, 5000] = float("nan")
        with pytest.raises(RuntimeError, match="non-finite"):
            m(x, {})
        m.check_finite = False
        out, _, _ = m(x, {})                       # without the guard: the reference's behaviour, NaNs are handed on
        assert torch.isfinite(out[0]).all() and not torch.isfinite(out[1]).all()
    finally:
        m.check_finite = False
