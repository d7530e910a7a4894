"""The back end writes every element of the waveform and of the est / mask / logits exports exactly as the model path.

septfa_forward is called through the C ABI with every output buffer (and the workspace) pre-filled with NaN, at
utterance lengths whose frame count T = 1 + L / 256 straddles the back end's CTA of 15 output blocks (T = 15, 16, 16
with a ragged tail, 17, 31, 130, 188). model.forward allocates with torch.empty, so the caching allocator can hand it the
previous call's buffer and a frame a kernel skipped would go unnoticed there.

The values are compared bit for bit where the forward reproduces itself bit for bit: one utterance, or utterances of at
least 128 frames. Several short utterances in one 128-row tile of the block kernels take their statistics from double
atomics in a varying order, so two forwards of such a batch differ in the last bits from the block chain on (the VAD
too); there every element is checked for being written.
"""
import ctypes as C

import pytest

from conftest import build_cuda_model

RAGGED_L = (3584, 3840, 3841, 4096, 7680, 33024, 48000)


@pytest.fixture(scope="module")
def vad_model():
    from septfa_b200 import synth
    return build_cuda_model(synth.CONFIG_WITH_VAD, 21)


@pytest.mark.gpu
@pytest.mark.parametrize("L", RAGGED_L)
@pytest.mark.parametrize("B", (1, 3, 7))
def test_exports_cover_every_element(vad_model, B, L):
    import torch
    from septfa_b200 import lib as _lib
    from septfa_b200 import synth

    m = vad_model
    kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
    x = torch.from_numpy(synth.make_mixtures(B, L, 900 + L)).cuda()
    ref_out, _, _ = m(x, dict(kw))
    ref = {"out": ref_out.clone(), "est": torch.view_as_real(m.estimated_stfts).clone(),
           "mask": m.mask_per_speaker.clone(), "logits": m.masks_b.clone()}

    dev = x.device
    h = m._handle(dev)
    T = _lib.num_frames(L)
    nan = lambda *shape: torch.full(shape, float("nan"), dtype=torch.float32, device=dev)  # noqa: E731
    got = {"out": nan(B, 2, L), "est": nan(B, 2, 257, T, 2), "mask": nan(B, 2, 257, T), "logits": nan(B, 514, T)}
    vad = nan(B, 2, T)
    need = h.lib.septfa_workspace_bytes(h.ptr, B, L)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    ikw = _lib.InferKw.from_dict(kw)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    rc = h.lib.septfa_forward(h.ptr, p(x), B, L, C.byref(ikw), p(got["out"]), p(vad), p(got["est"]), p(got["mask"]), None,
                              p(got["logits"]), p(ws), need, stream)
    _lib.check(h.ptr, rc)
    torch.cuda.synchronize()
    for k, v in got.items():
        assert bool(torch.isfinite(v).all()), f"{k}: {int((~torch.isfinite(v)).sum())} elements not written (B={B}, L={L}, T={T})"
        if B == 1 or T >= 128:
            assert torch.equal(v, ref[k]), f"{k} differs from the model path (B={B}, L={L}, T={T})"
