import contextlib, io, os, sys
import numpy as np, torch
sys.path.insert(0, "/root/repo")
from septfa_b200 import synth
from septfa_b200.model import SeparationModel
args = synth.CONFIG_WITH_VAD
with contextlib.redirect_stdout(io.StringIO()):
    m = SeparationModel(**args)
m.load_state_dict(synth.make_state_dict(args, 9), strict=True)
m.eval().cuda()
m.materialize.update(estimated_stfts=False, mask_per_speaker=False, spectrum=False, masks_b=False)
kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
for B in (1, 128, 256):
    x = torch.from_numpy(synth.make_mixtures(B, 64000, 1)).cuda()
    for cp in (0, 1, 2):
        m.set_option("conv1_pair", cp)
        for _ in range(5): m(x, kw)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50): m(x, kw)
        e1.record(); torch.cuda.synchronize()
        print(f"B={B} conv1_pair={cp}: {e0.elapsed_time(e1)/50:.4f} ms", flush=True)
