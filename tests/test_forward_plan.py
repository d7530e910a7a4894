"""Kernel selection of the forward: for each shape class and each kernel option, the ordered list of the library's
kernels one forward launches (torch.profiler, CUDA activities). The option tests elsewhere compare outputs of two
paths; this pins that each option and shape actually selects the kernels it names, and that no launcher falls back
to another kernel on its own. Kernels are named by base name and template arguments (the AMAX arguments follow the
signs of the seeded weights' PReLU slopes)."""
import re

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from septfa_b200 import synth

DEFAULTS = {"conv1_persist": 1, "conv1_pair": 1, "dconv_mma": 1, "fused_resid": 1, "stream_half": 0, "precision": 0}
KW = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)

PERSIST, PAIR, TMA = "k_conv1_persist<true,true>", "k_conv1_pair<true>", "k_conv1_tma<true>"
MMA2 = "k_dconv_mma2<true>"
CLUSTER = ("k_resid_persist<false,false>",)
STREAMING_H, STREAMING = ("k_tf_gate", "k_resid<0,true>", "k_resid<1,true>"), ("k_tf_gate", "k_resid<0,false>", "k_resid<1,false>")
TC1, TC2 = "k_tc_gemm<0,true,true,false>", "k_tc_gemm<1,true,true,false>"               # fp16 p / racc
TC1S, TC2S = "k_tc_gemm<0,false,true,true>", "k_tc_gemm<1,false,true,true>"             # split precision, fp32 p / racc
HEAD = ("k_frontend<false>",)
TAIL = ("k_out_stats", "k_tc_gemm<2,false,true,false>", "k_vad_final", "k_mask_istft")

# id: (config, B, samples, options, engine, exports, head, [(repeat, block)], tail) - 24 blocks at both configs
CASES = {
    "256x4s": ("with", 256, 64000, {}, 0, False, HEAD, [(1, (PERSIST, MMA2) + CLUSTER), (23, (PAIR, MMA2) + CLUSTER)], TAIL),
    "8x4s": ("with", 8, 64000, {}, 0, False, HEAD, [(24, (PERSIST, MMA2) + CLUSTER)], TAIL),
    "4x1s": ("with", 4, 16000, {}, 0, False, HEAD, [(24, (TC1, TC2) + CLUSTER)], TAIL),   # T = 63 < 128
    "without_vad": ("without", 8, 64000, {}, 0, False, HEAD, [(24, (TC1S, TC2S) + STREAMING)], TAIL),
    "precision2": ("with", 8, 64000, {"precision": 2}, 0, False, HEAD, [(24, (TC1S, TC2S) + STREAMING)], TAIL),
    "engine7": ("with", 8, 64000, {}, 7, False, HEAD, [(24, ("k_ref_conv1", "k_ref_dconv") + STREAMING)],
                ("k_out_stats", "k_ref_outconv", "k_vad_final", "k_mask_istft")),
    "conv1_persist0": ("with", 8, 64000, {"conv1_persist": 0}, 0, False, HEAD, [(24, (TC1, TC2) + CLUSTER)], TAIL),
    "conv1_pair0": ("with", 256, 64000, {"conv1_pair": 0}, 0, False, HEAD, [(24, (PERSIST, MMA2) + CLUSTER)], TAIL),
    "conv1_pair2": ("with", 8, 64000, {"conv1_pair": 2}, 0, False, HEAD,
                    [(1, (PERSIST, MMA2) + CLUSTER), (23, (PAIR, MMA2) + CLUSTER)], TAIL),
    "dconv_mma0": ("with", 8, 64000, {"dconv_mma": 0}, 0, False, HEAD,
                   [(24, ("k_conv1_persist<true,false>", TC2) + CLUSTER)], TAIL),
    "fused_resid0": ("with", 8, 64000, {"fused_resid": 0}, 0, False, HEAD, [(24, (PERSIST, MMA2) + STREAMING_H)], TAIL),
    "stream_half1": ("with", 8, 64000, {"stream_half": 1}, 0, False, HEAD,
                     [(1, (PERSIST, MMA2, "k_resid_persist<false,true>")), (22, (TMA, MMA2, "k_resid_persist<true,true>")),
                      (1, (TMA, MMA2, "k_resid_persist<true,false>"))], TAIL),
    "exports": ("with", 8, 64000, {}, 0, True, ("k_frontend<true>",), [(24, (PERSIST, MMA2) + CLUSTER)],
                TAIL[:-1] + ("k_mask_istft_export",)),
}


def short_name(name):
    """'void septfa::(anonymous namespace)::k_tc_gemm<0, true, true, false>(septfa::...)' -> 'k_tc_gemm<0,true,true,false>';
    None for anything that is not one of the library's kernels (memsets, copies, torch kernels)."""
    m = re.search(r"(?:^|::|\s)(k_\w+)(<[^<>()]*>)?\(", name)
    if m is None or "septfa::" not in name:
        return None
    return m.group(1) + (m.group(2) or "").replace(" ", "")


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_forward_kernel_selection(cuda_models, case):
    which, B, L, options, engine, exports, head, blocks, tail = CASES[case]
    m = cuda_models(synth.CONFIG_WITH_VAD if which == "with" else synth.CONFIG_WITHOUT_VAD, 9, engine)
    try:
        for k, v in dict(DEFAULTS, **options).items():
            m.set_option(k, v)
        m.materialize.update(estimated_stfts=exports, mask_per_speaker=exports, spectrum=exports, masks_b=exports)
        x = torch.from_numpy(synth.make_mixtures(B, L, 4321)).cuda()
        m(x, dict(KW))   # warm-up: module loading, lazily filled caches
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m(x, dict(KW))
            torch.cuda.synchronize()
        launches = m.last_launch_count
    finally:
        for k, v in DEFAULTS.items():
            m.set_option(k, v)
        m.materialize.update(estimated_stfts=True, mask_per_speaker=True, spectrum=True, masks_b=True)
        m.set_engine(0)
    events = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                    key=lambda e: e.time_range.start)
    got = [n for n in (short_name(e.name) for e in events) if n is not None]
    want = list(head) + [k for n, block in blocks for _ in range(n) for k in block] + list(tail)
    assert got == want
    assert launches == len(want)
