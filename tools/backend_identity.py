#!/usr/bin/env python
"""Byte-identity of the forward's outputs between two builds (for back-end changes that must not move a bit).

    python tools/backend_identity.py --root TREE_A --save DIR_A     # with TREE_A's libseptfa.so
    python tools/backend_identity.py --root TREE_B --save DIR_B
    python tools/backend_identity.py --compare DIR_A DIR_B          # np.array_equal per output and shape

Every run uses the same seeded weights and mixtures. Shapes: 256 x 64000 (config_with_vad, VAD gate on), 32 x 960000
(config_without_vad), and B = 1, 3, 7 at lengths whose T = 1 + L / 256 straddles the back end's 15-frame CTA boundary
(T = 15, 16, 16 with a ragged tail, 17, 31, 130, 188), config_with_vad with the VAD gate on. Outputs compared: the
waveform, the VAD, est, mask, logits_out and spectrum. The two large shapes are compared on a fixed seeded sample of
their rows (the whole of them would be several GB on disk).

Save each tree twice: a batch of several utterances shorter than 128 frames is not bit-reproducible from one forward to
the next (double atomics of the block statistics in a varying order, the VAD differs too), so a difference between the
trees there means something only where the tree's own two runs agree.
"""
import argparse
import contextlib
import io
import os
import sys

import numpy as np

RAGGED_L = (3584, 3840, 3841, 4096, 7680, 33024, 48000)


def cases():
    yield "vad_256x64000", "with", 256, 64000
    yield "novad_32x960000", "without", 32, 960000
    for L in RAGGED_L:
        for B in (1, 3, 7):
            yield f"vad_{B}x{L}", "with", B, L


def run(root, out_dir):
    sys.path.insert(0, root)
    import torch
    from septfa_b200 import synth
    from septfa_b200.model import SeparationModel

    os.makedirs(out_dir, exist_ok=True)
    models = {}
    for name, cfg, B, L in cases():
        args = synth.CONFIG_WITH_VAD if cfg == "with" else synth.CONFIG_WITHOUT_VAD
        if cfg not in models:
            with contextlib.redirect_stdout(io.StringIO()):
                m = SeparationModel(**args)
            m.load_state_dict(synth.make_state_dict(args, 5), strict=True)
            models[cfg] = m.eval().cuda()
        m = models[cfg]
        kw = dict(synth.DEFAULT_INFERENCE_KW, filter_signals_by_smo_vad=True) if cfg == "with" else {}
        x = torch.from_numpy(synth.make_mixtures(B, L, 4242)).cuda()
        out, vad, _ = m(x, kw)
        torch.cuda.synchronize()
        res = {"out": out, "est": torch.view_as_real(m.estimated_stfts), "mask": m.mask_per_speaker,
               "logits_out": m.masks_b, "spectrum": m.spectrum}
        if cfg == "with":
            res["vad"] = vad
        rows = np.random.default_rng(7).choice(B, size=min(B, 8), replace=False) if B > 8 else np.arange(B)
        res = {k: v.cpu().numpy()[np.sort(rows)] for k, v in res.items()}
        np.savez(os.path.join(out_dir, name + ".npz"), **res)
        print(f"{name}: saved {', '.join(sorted(res))}", flush=True)


def compare(a_dir, b_dir):
    bad = 0
    for name, *_ in cases():
        a = np.load(os.path.join(a_dir, name + ".npz"))
        b = np.load(os.path.join(b_dir, name + ".npz"))
        diff = []
        for k in sorted(a.files):
            if not (a[k].shape == b[k].shape and np.array_equal(a[k], b[k])):
                d = np.abs(a[k].astype(np.float64) - b[k]).max() if a[k].shape == b[k].shape else float("nan")
                diff.append(f"{k} (max |d| {d:.3e})")
        bad += len(diff)
        print(f"{name}: " + ("identical" if not diff else "DIFF " + ", ".join(diff)) + f"  [{', '.join(sorted(a.files))}]",
              flush=True)
    print("ALL IDENTICAL" if bad == 0 else f"{bad} DIFFERENCES")
    return 0 if bad == 0 else 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    help="repository tree whose septfa_b200 (and built libseptfa.so) to run")
    ap.add_argument("--save", metavar="DIR")
    ap.add_argument("--compare", nargs=2, metavar=("DIR_A", "DIR_B"))
    a = ap.parse_args()
    if a.compare:
        sys.exit(compare(*a.compare))
    if not a.save:
        ap.error("--save DIR or --compare DIR_A DIR_B")
    run(os.path.abspath(a.root), a.save)


if __name__ == "__main__":
    main()
