#!/usr/bin/env python
"""Generate tests/golden/reference_helpers.npz: the results of the reference's PIT, SI-SDR and simple-VAD helpers on
the seeded inputs of two tests, so that those tests need nothing outside the repository:

    python tests/golden/make_helper_golden.py

* ``pit_*``  - tests/test_host_logic.py::test_pit_helpers_equal_reference_functions (inputs stored with the results):
  ``PITLossWrapper.find_best_perm_factorial`` (model/pit_wrapper.py:261-312), ``get_pw_losses`` (:149-177) and the
  ``pw_pt`` wrapper with ``nn.L1Loss``;
* ``eval_*`` - tests/test_gpu_parity.py::test_evaluation_helpers_match_reference (inputs regenerated from
  ``numpy.random.default_rng(3)`` exactly as there): the pairwise negative SI-SDR matrix (``pairwise_neg_sisdr``,
  model/sdr.py:48-85), its PIT (``pit_from='pw_mtx'``), ``calc_sisdr`` of the reordered estimates and of the mixture
  (model/combined_loss.py:16-78), and ``calc_vad`` (Our_utils/utils_test.py:67-72).

Where the reference can be imported (oracle/ref_loader.py), its own functions compute every value. Elsewhere the
script falls back to the restatement below, which follows the reference's code (its PIT wrapper and pairwise SI-SDR
are asteroid's ``PITLossWrapper`` and ``PairwiseNegSDR``; ``calc_sisdr`` is the torchmetrics SI-SDR) and shares no code
with septfa_b200, so that the tests never compare the project's helpers with themselves. ``meta["source"]`` records
which of the two produced the file.
"""
import json
import os
import sys
import types
from itertools import permutations

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


class Restated:
    """The reference helpers, restated from their code (float32 on the CPU, like the reference)."""
    EPS = 1e-8   # PairwiseNegSDR's EPS

    class PITLossWrapper:
        def __init__(self, loss_func, pit_from="pw_mtx"):
            self.loss_func, self.pit_from = loss_func, pit_from

        @staticmethod
        def get_pw_losses(loss_func, est_targets, targets):
            n_src = targets.shape[1]
            pw = targets.new_empty(targets.shape[0], n_src, n_src)
            for i, est_src in enumerate(est_targets.transpose(0, 1)):
                for j, target_src in enumerate(targets.transpose(0, 1)):
                    pw[:, i, j] = loss_func(est_src, target_src)
            return pw

        @staticmethod
        def find_best_perm_factorial(pair_wise_losses):
            n_src = pair_wise_losses.shape[-1]
            pwl = pair_wise_losses.transpose(-1, -2)
            perms = pwl.new_tensor(list(permutations(range(n_src))), dtype=torch.long)
            one_hot = pwl.new_zeros((*perms.size(), n_src)).scatter_(2, perms.unsqueeze(2), 1)
            loss_set = torch.einsum("bij,pij->bp", [pwl, one_hot]) / n_src
            min_loss, min_idx = torch.min(loss_set, dim=1)
            return min_loss, torch.stack([perms[m] for m in min_idx], dim=0)

        def __call__(self, est_targets, targets, return_incides=False):
            if self.pit_from == "pw_mtx":
                pw = self.loss_func(est_targets, targets)
            else:
                pw = self.get_pw_losses(self.loss_func, est_targets, targets)
            min_loss, idx = self.find_best_perm_factorial(pw)
            return torch.mean(min_loss), idx

    @staticmethod
    def pairwise_neg_sisdr(est_targets, targets):
        targets = targets - targets.mean(dim=2, keepdim=True)
        est_targets = est_targets - est_targets.mean(dim=2, keepdim=True)
        s_target, s_estimate = targets.unsqueeze(1), est_targets.unsqueeze(2)
        dot = torch.sum(s_estimate * s_target, dim=3, keepdim=True)
        proj = dot * s_target / (torch.sum(s_target ** 2, dim=3, keepdim=True) + Restated.EPS)
        e_noise = s_estimate - proj
        sdr = torch.sum(proj ** 2, dim=3) / (torch.sum(e_noise ** 2, dim=3) + Restated.EPS)
        return -10 * torch.log10(sdr + Restated.EPS)

    @staticmethod
    def calc_sisdr(preds, target, zero_mean=True):
        eps = torch.finfo(preds.dtype).eps
        if zero_mean:
            target = target - torch.mean(target, dim=-1, keepdim=True)
            preds = preds - torch.mean(preds, dim=-1, keepdim=True)
        alpha = (torch.sum(preds * target, dim=-1, keepdim=True) + eps) / (torch.sum(target ** 2, dim=-1, keepdim=True) + eps)
        target_scaled = alpha * target
        noise = target_scaled - preds
        return 10 * torch.log10((torch.sum(target_scaled ** 2, dim=-1) + eps) / (torch.sum(noise ** 2, dim=-1) + eps))

    @staticmethod
    def reorder_source_mse(preds, batch_indices):
        return torch.stack([torch.index_select(s, 0, b) for s, b in zip(preds, batch_indices)])

    @staticmethod
    def calc_vad(masks):
        """A frame is active when at least a quarter of the 257 bins have mask >= 0.5."""
        return ((masks >= 0.5).long().sum(dim=2) >= 257 * 0.25).long()


def helpers():
    """(source, namespace of the helpers): the reference's own when it can be imported, the restatement otherwise."""
    import importlib
    from oracle import ref_loader
    if not ref_loader.available():
        return "restated", Restated
    ns = ref_loader.load()
    sdr, ut = importlib.import_module("model.sdr"), importlib.import_module("Our_utils.utils_test")
    return f"reference ({ns.kind} import)", types.SimpleNamespace(
        PITLossWrapper=ns.pit_wrapper.PITLossWrapper, pairwise_neg_sisdr=sdr.pairwise_neg_sisdr,
        calc_sisdr=ns.combined_loss.calc_sisdr, reorder_source_mse=ns.combined_loss.reorder_source_mse,
        calc_vad=ut.calc_vad)


def pit_case(rec, R):
    g = torch.Generator().manual_seed(5)
    for n_src in (2, 3):
        pw = torch.rand(64, n_src, n_src, generator=g)
        pw[::7] = 0.25                                     # all permutations tie
        pw[1::9, 0, 0] = pw[1::9, 1, 0]                    # partial ties
        pw[1::9, 1, 1] = pw[1::9, 0, 1]
        loss, idx = R.PITLossWrapper.find_best_perm_factorial(pw)
        rec[f"pit_pw{n_src}"], rec[f"pit_loss{n_src}"], rec[f"pit_idx{n_src}"] = pw.numpy(), loss.numpy(), idx.numpy()
    est, tgt = torch.randn(3, 2, 500, generator=g), torch.randn(3, 2, 500, generator=g)
    l1 = torch.nn.L1Loss()
    loss, idx = R.PITLossWrapper(l1, pit_from="pw_pt")(est, tgt, return_incides=True)
    rec.update(pit_est=est.numpy(), pit_tgt=tgt.numpy(), pit_pw_l1=R.PITLossWrapper.get_pw_losses(l1, est, tgt).numpy(),
               pit_wrapper_loss=loss.numpy(), pit_wrapper_idx=idx.numpy())


def eval_case(rec, R):
    rng = np.random.default_rng(3)
    tgt = torch.from_numpy(rng.standard_normal((5, 2, 32000)).astype(np.float32) * 0.1)
    est = tgt.clone()
    est[[1, 3]] = est[[1, 3]][:, [1, 0]]
    est = est * 0.8 + 0.03 * torch.from_numpy(rng.standard_normal(est.shape).astype(np.float32))
    # a random level per frame, so that some frames are active and others not
    masks = torch.from_numpy(rng.random((3, 2, 257, 40), dtype=np.float32) * rng.random((3, 2, 1, 40), dtype=np.float32))
    loss, idx = R.PITLossWrapper(R.pairwise_neg_sisdr, pit_from="pw_mtx")(est, tgt, return_incides=True)
    mix = tgt.sum(dim=1)
    rec.update(eval_pw=R.pairwise_neg_sisdr(est, tgt).numpy(), eval_loss=loss.numpy(), eval_idx=idx.numpy(),
               eval_si_sdr=R.calc_sisdr(R.reorder_source_mse(est, idx), tgt).numpy(),
               eval_si_sdr_start=R.calc_sisdr(mix[:, None].repeat(1, 2, 1), tgt).numpy(),
               eval_vad=np.asarray(R.calc_vad(masks), dtype=np.int64))


def main():
    source, R = helpers()
    rec = {"meta": json.dumps({"source": source, "torch": torch.__version__, "numpy": np.__version__})}
    pit_case(rec, R)
    eval_case(rec, R)
    np.savez_compressed(os.path.join(HERE, "reference_helpers.npz"), **rec)
    print(source, {k: v.shape for k, v in rec.items() if k != "meta"})


if __name__ == "__main__":
    main()
