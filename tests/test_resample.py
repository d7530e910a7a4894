"""septfa_resample / SeparationModel.resample on the GPU against torchaudio.functional.resample (its defaults, what
read_mixture runs through transforms.Resample)."""
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
    orig, new = rate // g, 16000 // g
    return math.ceil(6 * orig / (min(orig, new) * 0.99))


def lengths(rate):
    orig = rate // math.gcd(rate, 16000)
    return [max(width(rate) - 2, 1), 3 * orig + 1, 48007]   # shorter than the filter, not a multiple of orig, 3 s


@pytest.fixture(scope="module")
def model(cuda_models):
    return cuda_models(synth.CONFIG_WITH_VAD, 41, 0)


@pytest.mark.parametrize("rate", RATES)
def test_resample_matches_torchaudio(model, rate):
    rng = np.random.default_rng(rate)
    worst64 = worst32 = own32 = 0.0
    for L in lengths(rate):
        for B in (1, 7):
            x = torch.from_numpy(rng.uniform(-0.9, 0.9, (B, L))).float()
            y = model.resample(x.cuda(), rate).cpu()
            ref64 = AF.resample(x.double(), rate, 16000)
            ref32 = AF.resample(x, rate, 16000)
            assert y.shape == ref64.shape == (B, -(-16000 * L // rate))
            worst64 = max(worst64, (y.double() - ref64).abs().max().item())
            worst32 = max(worst32, (y - ref32).abs().max().item())
            own32 = max(own32, (ref32.double() - ref64).abs().max().item())
    print(f"rate {rate}: max |d| {worst64:.3g} against float64 torchaudio, {worst32:.3g} against float32 "
          f"(float32 torchaudio itself: {own32:.3g} off float64)")
    assert worst64 <= 1e-6
    # float32 torchaudio computes its bank in float32; at an odd rate such as 44056 Hz (orig = 5507) that alone puts it
    # ~1e-4 off its float64 result, so there the bound is its own error
    assert worst32 <= max(5e-5, own32 + 1e-6)


@pytest.mark.parametrize("rate", [8000, 44100, 48000])
def test_resample_pcm16_equals_float_input(model, rate):
    rng = np.random.default_rng(3)
    pcm = torch.from_numpy(rng.integers(-32768, 32768, (3, 20011)).astype(np.int16)).cuda()
    a = model.resample(pcm, rate)
    b = model.resample(pcm.float(), rate)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_resample_16k_is_the_identity(model):
    x = torch.from_numpy(np.random.default_rng(4).uniform(-0.9, 0.9, (3, 1001))).float().cuda()
    assert torch.equal(model.resample(x, 16000), x)
    pcm = (x * 30000).to(torch.int16)
    assert torch.equal(model.resample(pcm, 16000), pcm.float())


def test_resample_is_deterministic(model):
    x = torch.from_numpy(np.random.default_rng(5).uniform(-0.9, 0.9, (5, 44100))).float().cuda()
    for rate in (44100, 8000):
        a, b = model.resample(x, rate), model.resample(x, rate)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        assert model.last_launch_count == 1


@pytest.mark.parametrize("rate", [7999, 192001, 0, -48000])
def test_resample_refuses_rates(model, rate):
    x = torch.zeros((2, 1000), device="cuda")
    out = torch.full((2, 4000), 7.0, device="cuda")
    h = model._handle(x.device)
    model.resample(x, 48000)
    assert h.lib.septfa_last_launch_count(h.ptr) == 1
    rc = h.lib.septfa_resample(h.ptr, C.c_void_p(x.data_ptr()), 0, 2, 1000, rate, C.c_void_p(out.data_ptr()),
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == INVALID
    assert f"rate {rate}" in h.lib.septfa_last_error(h.ptr).decode()
    assert h.lib.septfa_last_launch_count(h.ptr) == 0
    torch.cuda.synchronize()
    assert bool((out == 7.0).all())
