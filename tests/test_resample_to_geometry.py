"""septfa_resample_to_geometry and the output-rate rule of live sessions (no GPU needed).

The output direction resamples the model's 16 kHz output to `rate`: torchaudio.functional.resample(y, 16000, rate), so
the source is 16 kHz and orig = 16000 / g, new = rate / g with g = gcd(rate, 16000). The support of torchaudio's bank
is recomputed here from its formulas: for output phase p and tap c = j - width the scaled time is
t = base (c / orig - p / new) with base = 0.99 min(orig, new); the effective taps are those with |t| < 6. D_out is the
least delay (in output samples) such that every output before N Ho - D_out reads only y[0, N H), for every hop H that is
a multiple of orig (Ho = H new / orig). The history is the number of 16 kHz samples before a hop that the outputs of
the next push read.
"""
import math

import numpy as np
import pytest

from septfa_b200 import lib as L
from septfa_b200.live import check_geometry

STANDARD = [8000, 11025, 12000, 22050, 24000, 32000, 44100, 48000, 88200, 96000, 176400, 192000]
ODD = [44056, 8001, 191975]


def support(rate):
    """(orig, new, width, c_min[p], c_max[p]) of the 16000 -> rate bank, |t| < 6 decided exactly in integers."""
    g = math.gcd(rate, 16000)
    orig, new = 16000 // g, rate // g
    mn = min(orig, new)
    width = math.ceil(6 * orig / (mn * 0.99))
    c = np.arange(-width, width + orig, dtype=np.int64)[None]
    cmin, cmax = np.empty(new, np.int64), np.empty(new, np.int64)
    for p0 in range(0, new, 512):   # phases in chunks: 8001 Hz has 8001 phases of 16026 taps
        p = np.arange(p0, min(new, p0 + 512), dtype=np.int64)[:, None]
        # |t| < 6  <=>  0.99 mn |c new - p orig| / (orig new) < 6, in integers
        keep = 99 * mn * np.abs(c * new - p * orig) < 600 * orig * new
        assert keep.any(1).all()
        assert ((np.diff(keep.astype(np.int8), axis=1) != 0).sum(1) <= 2).all()   # one contiguous run per phase
        cmin[p0:p0 + 512] = np.where(keep, c, np.iinfo(np.int64).max).min(1)
        cmax[p0:p0 + 512] = np.where(keep, c, np.iinfo(np.int64).min).max(1)
    return orig, new, width, cmin, cmax


def hops(orig):
    """Hops (16 kHz samples) to check: the hop multiple itself and the smallest multiple a live session accepts."""
    return sorted({orig, orig * -(-256 // orig)})


def delay_and_history(rate, n_hops=3):
    """D_out and the history from the definition, over N = 1 .. n_hops pushes of each hop in hops()."""
    orig, new, width, cmin, cmax = support(rate)
    D = 0
    for H in hops(orig):
        Ho = H * new // orig
        for N in range(1, n_hops + 1):
            m = np.arange(N * Ho)
            last = (m // new) * orig + cmax[m % new]
            late = np.nonzero(last >= N * H)[0]
            if late.size:
                D = max(D, N * Ho - int(late.min()))
    hist = 0
    for H in hops(orig):
        Ho = H * new // orig
        for N in range(1, n_hops + 1):
            m = np.arange(N * Ho - D, (N + 1) * Ho - D)
            first = (m // new) * orig + cmin[m % new]
            hist = max(hist, N * H - int(first.min()))
    return D, hist


@pytest.mark.parametrize("rate", STANDARD + ODD)
def test_resample_to_geometry_matches_the_support(rate):
    d, mult = L.resample_to_geometry(rate)
    orig, new, width, cmin, cmax = support(rate)
    D, hist = delay_and_history(rate)
    assert mult == orig == 16000 // math.gcd(rate, 16000)
    assert d == D
    assert d <= 0.75e-3 * rate   # at most 0.75 ms
    # a live session keeps `hist` 16 kHz samples per channel and needs hist <= H: no hop it accepts (>= 256) is refused
    assert hist <= 24 and hist <= 256


@pytest.mark.parametrize("rate", [22050, 44100, 48000, 8000, 11025])
def test_output_taps_outside_the_support_are_negligible(rate):
    """What the cut drops: torchaudio's own float64 taps of 16000 -> rate with |t| >= 6 are ~1e-20 or smaller."""
    torch = pytest.importorskip("torch")
    F = pytest.importorskip("torchaudio.functional.functional")
    orig, new, width, cmin, cmax = support(rate)
    k, w = F._get_sinc_resample_kernel(16000, rate, math.gcd(rate, 16000), dtype=torch.float64)
    assert w == width
    k = k[:, 0].numpy()
    c = np.arange(-width, width + orig)[None]
    inside = (c >= cmin[:, None]) & (c <= cmax[:, None])
    assert k.shape == inside.shape
    assert np.abs(k[~inside]).max(initial=0.0) < 1e-15
    assert np.allclose(k[0][inside[0]].sum(), 1.0, atol=0.02)   # the kept taps carry the gain


@pytest.mark.parametrize("rate", [8000, 11025, 22050, 44100, 48000, 192000])
def test_output_before_the_delay_is_causal(rate):
    """With float64 torchaudio: resampling y[:N H] and y give the same first N Ho - D_out outputs."""
    torch = pytest.importorskip("torch")
    AF = pytest.importorskip("torchaudio.functional")
    D, mult = L.resample_to_geometry(rate)
    H = mult * -(-256 // mult)
    Ho = H * rate // 16000
    y = torch.from_numpy(np.random.default_rng(rate).uniform(-0.9, 0.9, (1, 5 * H)))
    full = AF.resample(y, 16000, rate)
    for N in (1, 2, 4):
        part = AF.resample(y[:, :N * H], 16000, rate)
        n = N * Ho - D
        assert (part[:, :n] - full[:, :n]).abs().max().item() <= 1e-12


def test_resample_to_geometry_identity_rate():
    assert L.resample_to_geometry(16000) == (0, 1)


@pytest.mark.parametrize("rate", [7999, 192001, 0, -44100])
def test_resample_to_geometry_refuses(rate):
    lib = L.load()
    d, m = L.C.c_int(-7), L.C.c_int(-7)
    assert lib.septfa_resample_to_geometry(rate, L.C.byref(d), L.C.byref(m)) == -1   # SEPTFA_E_INVALID
    assert f"rate {rate}" in lib.septfa_last_error(None).decode()
    assert (d.value, m.value) == (-7, -7)
    assert lib.septfa_resample_geometry(rate, None, None) == -1   # the input direction refuses the same rates


@pytest.mark.parametrize("window,hop,rate,out_rate", [
    (48000, 16000, 16000, 48000), (48000, 16000, 48000, 48000), (48000, 16000, 44100, 44100),
    (48000, 16000, 8000, 8000), (48000, 16000, 16000, 8000), (48000, 8000, 16000, 44100),
    (48000, 4160, 16000, 48000), (48000, 16000, 16000, 191975), (48000, 16000, 8000, np.int64(22050)),
    (48000, 4000, 44100, 16000)])
def test_check_geometry_accepts_out_rates(window, hop, rate, out_rate):
    assert check_geometry(window, hop, rate, out_rate) == (window, hop)
    assert check_geometry(window, hop, rate=rate, out_rate=out_rate) == (window, hop)


@pytest.mark.parametrize("window,hop,rate,out_rate", [
    (48000, 4080, 48000, 44100),    # 160 does not divide the hop at the output rate
    (48000, 8000, 16000, 11025),    # 640 does not divide the hop
    (48000, 4000, 16000, 22050),    # 320 does not divide the hop
    (48000, 4080, 44100, 48000),    # the input rate's rule still applies
    (48000, 16000, 16000, 7999),    # below 8 kHz
    (48000, 16000, 16000, 192001),  # above 192 kHz
    (48000, 16000, 16000, 0),
    (48000, 16000, 16000, 48000.0),  # not an integer
    (48000, 16000, 16000, True),
    (48000, 240, 16000, 48000),     # the 16 kHz rules still apply
])
def test_check_geometry_refuses_out_rates(window, hop, rate, out_rate):
    with pytest.raises(ValueError):
        check_geometry(window, hop, rate, out_rate)
