import contextlib, io, sys
import numpy as np, torch
sys.path.insert(0, "/root/repo")
from oracle import septfa_oracle as O
from septfa_b200 import synth
from septfa_b200.model import SeparationModel
args = synth.CONFIG_WITH_VAD
kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True)
for wseed in (0, 9):
    with contextlib.redirect_stdout(io.StringIO()):
        m = SeparationModel(**args)
    m.load_state_dict(synth.make_state_dict(args, wseed), strict=True)
    m.eval().cuda()
    W = O.OracleWeights(synth.make_state_dict_numpy(args, wseed), args, np.float64)
    for xseed in (1234, 4242):
        x = synth.make_mixtures(2, 64000, xseed)
        ref_out, ref_vad, _, _ = O.forward(x, W, dict(kw))
        xt = torch.from_numpy(x).cuda()
        for opts in ({}, {"dconv_mma": 0}, {"precision": 2}, {"engine": 7}):
            for k, v in {"dconv_mma": 1, "precision": 0}.items(): m.set_option(k, v)
            m.engine = 0
            for k, v in opts.items():
                if k == "engine": m.engine = v
                else: m.set_option(k, v)
            out, vad, _ = m(xt, dict(kw))
            dv = np.abs(vad.cpu().numpy() - ref_vad).max()
            print(f"w{wseed} x{xseed} {opts}: dvad {dv:.2e}", flush=True)
