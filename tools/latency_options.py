#!/usr/bin/env python
"""Small-request latency (one / eight 4 s mixtures) with single kernel-selection options flipped: which kernels should small batches run?"""
import contextlib, io, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from septfa_b200 import synth
from septfa_b200.model import SeparationModel
args = synth.CONFIG_WITH_VAD
with contextlib.redirect_stdout(io.StringIO()):
    m = SeparationModel(**args)
m.load_state_dict(synth.make_state_dict(args, 0), strict=True)
m.eval().cuda()
kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
m.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)

def p50(x):
    for _ in range(5): m(x, kw)
    ts = []
    for _ in range(40):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); m(x, kw); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[20]

opts = [("default", None, None)] + [(f"{n}={v}", n, v) for n, v in (("dconv_mma", 0), ("conv1_pair", 2), ("fused_resid", 0))]
for B in (1, 8, 32):
    x = torch.from_numpy(synth.make_mixtures(B, 64000, 1)).cuda()
    line = []
    for name, n, v in opts:
        try:
            if n: m.set_option(n, v)
            line.append(f"{name} {p50(x):.3f}")
        except Exception as e:
            line.append(f"{name} ERR {type(e).__name__}")
        finally:
            if n: m.set_option(n, 1)
    m.set_profile(True)
    for _ in range(5): m(x, kw)
    prof = m.read_profile(); m.set_profile(False)
    print(f"B={B}: " + " | ".join(line), flush=True)
    print("   per class (serialised, ms):", {k: round(v[0] / 5, 3) for k, v in prof.items()}, flush=True)
