"""septfa_resample_geometry and the rate rule of live sessions (no GPU needed).

The support of torchaudio's resampling bank (sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99) is recomputed
here from torchaudio's formulas: for output phase p and tap j the scaled time is t = base ((j - width) / orig - p / new)
with base = 0.99 min(orig, new); the effective taps are those with |t| < 6. D is the least delay (in 16 kHz samples)
such that every output before N H - D reads only native samples before N Hn, for every hop H that is a multiple of new.
"""
import math

import numpy as np
import pytest

from septfa_b200 import lib as L
from septfa_b200.live import check_geometry

TABLE = {8000: 12, 11025: 8, 12000: 8, 22050: 6, 24000: 6, 32000: 6, 44100: 6, 48000: 6, 88200: 6, 96000: 6,
         176400: 6, 192000: 6}
ODD = [44056, 8001, 191975]


def support(rate):
    """(orig, new, width, first tap offset c_min[p], last c_max[p]) with c = j - width, |t| < 6 decided exactly."""
    g = math.gcd(rate, 16000)
    orig, new = rate // g, 16000 // g
    mn = min(orig, new)
    width = math.ceil(6 * orig / (mn * 0.99))
    c = np.arange(-width, width + orig, dtype=np.int64)[None]
    p = np.arange(new, dtype=np.int64)[:, None]
    # |t| < 6  <=>  0.99 mn |c new - p orig| / (orig new) < 6, in integers
    keep = 99 * mn * np.abs(c * new - p * orig) < 600 * orig * new
    assert keep.any(1).all()
    runs = np.diff(keep.astype(np.int8), axis=1)
    assert ((runs != 0).sum(1) <= 2).all()   # one contiguous run per phase
    cmin = np.where(keep, c, np.iinfo(np.int64).max).min(1)
    cmax = np.where(keep, c, np.iinfo(np.int64).min).max(1)
    return orig, new, width, cmin, cmax


def delay_bruteforce(rate, n_hops=3):
    """D from the definition: for N = 1 .. n_hops pushes of the smallest hop H (a multiple of new, >= 256), the least D
    such that every output m < N H - D reads only native samples < N Hn."""
    orig, new, width, cmin, cmax = support(rate)
    H = new * -(-256 // new)
    Hn = H * orig // new
    D = 0
    for N in range(1, n_hops + 1):
        m = np.arange(N * H)
        last = (m // new) * orig + cmax[m % new]
        late = np.nonzero(last >= N * Hn)[0]
        if late.size:
            D = max(D, N * H - int(late.min()))
    return D


@pytest.mark.parametrize("rate", sorted(TABLE) + ODD)
def test_resample_geometry_matches_the_support(rate):
    d, mult = L.resample_geometry(rate)
    orig, new, width, cmin, cmax = support(rate)
    assert mult == new
    assert d == delay_bruteforce(rate)
    if rate in TABLE:
        assert d == TABLE[rate]
    assert d <= 12   # <= 0.75 ms at 16 kHz


@pytest.mark.parametrize("rate", [22050, 44100, 48000, 8000])
def test_taps_outside_the_support_are_negligible(rate):
    """What the cut drops: torchaudio's own float64 taps with |t| >= 6 are ~1e-20 or smaller."""
    torch = pytest.importorskip("torch")
    F = pytest.importorskip("torchaudio.functional.functional")
    orig, new, width, cmin, cmax = support(rate)
    k, w = F._get_sinc_resample_kernel(rate, 16000, math.gcd(rate, 16000), dtype=torch.float64)
    assert w == width
    k = k[:, 0].numpy()
    c = np.arange(-width, width + orig)[None]
    inside = (c >= cmin[:, None]) & (c <= cmax[:, None])
    assert np.abs(k[~inside]).max(initial=0.0) < 1e-15
    assert np.allclose(k[0][inside[0]].sum(), 1.0, atol=0.02)   # the kept taps carry the gain


def test_resample_geometry_identity_rate():
    assert L.resample_geometry(16000) == (0, 1)


@pytest.mark.parametrize("rate", [7999, 192001, 0, -44100])
def test_resample_geometry_refuses(rate):
    lib = L.load()
    d, m = L.C.c_int(-7), L.C.c_int(-7)
    assert lib.septfa_resample_geometry(rate, L.C.byref(d), L.C.byref(m)) == -1   # SEPTFA_E_INVALID
    assert f"rate {rate}" in lib.septfa_last_error(None).decode()
    assert (d.value, m.value) == (-7, -7)


@pytest.mark.parametrize("window,hop,rate", [(48000, 16000, 44100), (48000, 16000, 8000), (48000, 16000, 11025),
                                             (48000, 8000, 48000), (48000, 4000, 44100), (48000, 4160, 48000),
                                             (48000, 16000, 192000), (48000, 16000, 44056), (48000, 16000, 191975),
                                             (48000, 16000, np.int64(22050)), (48000, 4000, 16000)])
def test_check_geometry_accepts_rates(window, hop, rate):
    assert check_geometry(window, hop, rate) == (window, hop)


@pytest.mark.parametrize("window,hop,rate", [
    (48000, 4080, 44100),     # 160 does not divide the hop
    (48000, 8000, 11025),     # 640 does not divide the hop
    (48000, 4000, 22050),     # 320 does not divide the hop
    (48000, 16000, 7999),     # below 8 kHz
    (48000, 16000, 192001),   # above 192 kHz
    (48000, 16000, 0),
    (48000, 16000, 44100.0),  # not an integer
    (48000, 16000, True),
    (48000, 240, 48000),      # the 16 kHz rules still apply
])
def test_check_geometry_refuses_rates(window, hop, rate):
    with pytest.raises(ValueError):
        check_geometry(window, hop, rate)
