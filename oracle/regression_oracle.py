"""TEST INFRASTRUCTURE ONLY -- the regression objectives restated with torch CPU ops (any float dtype: the tests run it in
fp32, which is what the reference computes, and in fp64, the truth the CUDA kernels are held to).

  * `masked_loss`: L1Loss / L2Loss (bm/losses.py:11-26), mean over `mask.expand_as(estimate)` of |e - o|^p.  The reference
    gathers the selected elements with a boolean index; `torch.where` selects them here without a gather, so a NaN or inf
    in an unselected position reaches neither the loss nor, through autograd, the gradient, exactly as there.
  * `regression_step`: `bm_oracle.training_step` with the masked loss in place of ClipLoss (the solver's 'l1' / 'mse'
    objectives, bm/solver.py:76-94), against mel-like targets instead of candidates.
"""
from __future__ import annotations

import torch

from oracle import bm_oracle


def masked_loss(estimate: torch.Tensor, output: torch.Tensor, mask: torch.Tensor, p: int) -> torch.Tensor:
    """0-dim mean of |estimate - output|^p over the selected elements; NaN (0/0) when nothing is selected."""
    assert p in (1, 2) and mask.dtype == torch.bool
    sel = mask.expand_as(estimate)
    d = torch.where(sel, estimate - output, torch.zeros((), dtype=estimate.dtype))
    per = d.abs() if p == 1 else d * d
    return per.sum() / sel.sum().to(estimate.dtype)


def regression_step(p, cfg, meg, rec_positions, rec_of_sample, subject_index, targets, mask, loss_p: int,
                    ban_centre=None, training=True, target_grad=False):
    """forward + masked L1 / L2 loss + backward.  Returns dict(estimate, loss, grads{name: tensor}, bn_updates) and, with
    `target_grad`, the gradient of the loss with respect to the targets under `target_grad`."""
    params = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and
                  not k.endswith(("running_mean", "running_var")) else v) for k, v in p.items()}
    bn_updates: dict = {}
    est = bm_oracle.simpleconv_forward(params, cfg, meg, rec_positions, rec_of_sample, subject_index, training, ban_centre,
                                       bn_updates)
    out = targets.detach().clone().requires_grad_(target_grad)
    loss = masked_loss(est, out, mask, loss_p)
    names = [k for k, v in params.items() if v.requires_grad]
    leaves = [params[k] for k in names] + ([out] if target_grad else [])
    grads = torch.autograd.grad(loss, leaves, allow_unused=True)
    res = dict(estimate=est.detach(), loss=loss.detach(), grads={k: g for k, g in zip(names, grads)},
               bn_updates=bn_updates)
    if target_grad:
        res["target_grad"] = grads[-1]
    return res
