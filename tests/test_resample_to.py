"""septfa_resample_to / SeparationModel.resample_to on the GPU against torchaudio.functional.resample(y, 16000, rate)
with its defaults: the model's 16 kHz output back at a caller's rate."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torchaudio.functional as AF

from septfa_b200 import synth

pytestmark = pytest.mark.gpu

INVALID = -1   # SEPTFA_E_INVALID
RATES = [8000, 11025, 22050, 32000, 44100, 48000, 96000, 192000, 44056]


def width(rate):
    g = math.gcd(rate, 16000)
    orig, new = 16000 // g, rate // g
    return math.ceil(6 * orig / (min(orig, new) * 0.99))


def lengths(rate):
    orig = 16000 // math.gcd(rate, 16000)
    return [max(width(rate) - 2, 1), 3 * orig + 1, 48007]   # shorter than the filter, not a multiple of orig, 3 s


@pytest.fixture(scope="module")
def model(cuda_models):
    return cuda_models(synth.CONFIG_WITH_VAD, 41, 0)


@pytest.mark.parametrize("rate", RATES)
def test_resample_to_matches_torchaudio(model, rate):
    rng = np.random.default_rng(rate + 1)
    worst64 = worst32 = own32 = 0.0
    for L in lengths(rate):
        for B in (1, 7):
            y = torch.from_numpy(rng.uniform(-0.9, 0.9, (B, L))).float()
            z = model.resample_to(y.cuda(), rate).cpu()
            ref64 = AF.resample(y.double(), 16000, rate)
            ref32 = AF.resample(y, 16000, rate)
            assert z.shape == ref64.shape == (B, -(-rate * L // 16000))
            worst64 = max(worst64, (z.double() - ref64).abs().max().item())
            worst32 = max(worst32, (z - ref32).abs().max().item())
            own32 = max(own32, (ref32.double() - ref64).abs().max().item())
    print(f"16000 -> {rate}: max |d| {worst64:.3g} against float64 torchaudio, {worst32:.3g} against float32 "
          f"(float32 torchaudio itself: {own32:.3g} off float64)")
    assert worst64 <= 1e-6
    # float32 torchaudio builds its bank in float32; at an odd rate that alone moves it off its float64 result
    assert worst32 <= max(5e-5, own32 + 1e-6)


def test_resample_to_takes_a_forward_output(model):
    """[B, 2, L] in: the leading dimensions are rows."""
    y = torch.from_numpy(np.random.default_rng(2).uniform(-0.9, 0.9, (3, 2, 16001))).float().cuda()
    z = model.resample_to(y, 44100)
    assert z.shape == (3, 2, -(-44100 * 16001 // 16000))
    assert torch.equal(z.view(6, -1).view(torch.int32), model.resample_to(y.view(6, -1), 44100).view(torch.int32))
    assert torch.equal(z[1, 0].view(torch.int32), model.resample_to(y[1, 0:1], 44100)[0].view(torch.int32))


def test_resample_to_16k_is_the_identity(model):
    y = torch.from_numpy(np.random.default_rng(4).uniform(-0.9, 0.9, (3, 1001))).float().cuda()
    assert torch.equal(model.resample_to(y, 16000), y)


def test_resample_to_is_deterministic(model):
    y = torch.from_numpy(np.random.default_rng(5).uniform(-0.9, 0.9, (5, 16000))).float().cuda()
    for rate in (44100, 8000, 48000):
        a, b = model.resample_to(y, rate), model.resample_to(y, rate)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        assert model.last_launch_count == 1


def test_resample_to_and_resample_keep_their_own_banks(model):
    """The two directions at one rate are different banks: the cache keys them apart."""
    y = torch.from_numpy(np.random.default_rng(6).uniform(-0.9, 0.9, (2, 16000))).float().cuda()
    up = model.resample_to(y, 48000)
    down = model.resample(up, 48000)
    up2 = model.resample_to(y, 48000)
    assert up.shape == (2, 48000) and down.shape == (2, 16000)
    assert torch.equal(up.view(torch.int32), up2.view(torch.int32))
    ref = AF.resample(AF.resample(y.cpu().double(), 16000, 48000), 48000, 16000)
    assert (down.cpu().double() - ref).abs().max().item() <= 5e-6


@pytest.mark.parametrize("rate", [7999, 192001, 0, -48000])
def test_resample_to_refuses_rates(model, rate):
    y = torch.zeros((2, 1000), device="cuda")
    out = torch.full((2, 13000), 7.0, device="cuda")
    h = model._handle(y.device)
    model.resample_to(y, 48000)
    assert h.lib.septfa_last_launch_count(h.ptr) == 1
    rc = h.lib.septfa_resample_to(h.ptr, C.c_void_p(y.data_ptr()), 2, 1000, rate, C.c_void_p(out.data_ptr()),
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == INVALID
    assert f"rate {rate}" in h.lib.septfa_last_error(h.ptr).decode()
    assert h.lib.septfa_last_launch_count(h.ptr) == 0
    torch.cuda.synchronize()
    assert bool((out == 7.0).all())
