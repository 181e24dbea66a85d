"""Drop-in `ClipLoss` (reference: bm/losses.py:29-114): same constructor, `forward(estimate, candidate, mask)`,
`get_scores`, `get_probabilities`, `trim_samples`.  Scores, softmax / cross-entropy and their gradient run in
CUDA through the C ABI (`functional.clip_loss`, `functional.clip_scores`).

Reference semantics kept on purpose: only the CANDIDATES are L2-normalised (losses.py:91-94), no temperature,
the `linear` projection is constructed but never applied (losses.py:35,82), targets are the first B candidates.

Extension (SURVEY.md 8(e), not in the reference): `global_negatives=True` all-gathers the candidates over the
default process group before scoring, so every rank contrasts against the global batch; when the candidates require
grad (a trainable feature model) the gather is differentiable (reduce-scatter of the candidate gradients).

Drop-in `L1Loss` / `L2Loss` (reference: bm/losses.py:11-26, the solver's 'l1' and 'mse' objectives): no-argument
constructor, `forward(estimate, output, mask)`; the masked mean and its gradient run in CUDA (`functional.regression_loss`).
"""
from __future__ import annotations

import weakref

import torch

from . import common as CM
from . import functional as BF
from . import distrib


class _MaskedLoss(torch.nn.Module):
    """bm/losses.py:11-14: the mean of the per-element loss over `mask.expand_as(estimate)`, on one CUDA pass forward and
    one backward (`functional.regression_loss`) instead of a boolean gather, which synchronises with the host."""
    _p = 0

    def forward(self, estimate, output, mask=None):
        for name, t in (("estimate", estimate), ("output", output)):
            CM._require_cuda_fp32(t, f"{type(self).__name__} ({name})")
        return BF.regression_loss(estimate, output, mask, self._p)


class L1Loss(_MaskedLoss):
    """The solver's `optim.loss=l1` (bm/solver.py:76-94): mean |estimate - output| over the masked elements."""
    _p = 1

    def __init__(self):
        super().__init__()
        self._loss = torch.nn.L1Loss()           # never called; kept so that repr() and state_dict() match the reference


class L2Loss(_MaskedLoss):
    """The solver's `optim.loss=mse`: mean (estimate - output)^2 over the masked elements."""
    _p = 2

    def __init__(self):
        super().__init__()
        self._loss = torch.nn.MSELoss()          # never called; kept so that repr() and state_dict() match the reference


class ClipLoss(torch.nn.Module):
    def __init__(self, linear=None, twin=True, pool=False, tmin=None, tmax=None,
                 tmin_train=None, tmax_train=None, dset_args=None, center=False, global_negatives=False,
                 uniform_batches=False):
        super().__init__()
        self.linear = None                      # the reference never applies its projection (losses.py:35)
        self.pool = pool
        self.center = center
        if linear is not None:                  # kept for state_dict compatibility only
            self.linear_est = torch.nn.LazyLinear(linear)
            self.linear_gt = self.linear_est if twin else torch.nn.LazyLinear(linear)
        self.tmin, self.tmax = tmin, tmax
        self.tmin_train, self.tmax_train = tmin_train, tmax_train
        self.dset_args = dset_args
        self.global_negatives = global_negatives
        # global_negatives only: True = every rank holds the same number of rows each step (drop_last loaders, no
        # rejection), which saves the per-step exchange of the per-rank counts; False = counts are exchanged and ragged
        # batches are handled (the reference's loaders have no drop_last, and ScaleReject drops samples per rank)
        self.uniform_batches = uniform_batches
        self._prefetched = None
        self._mask_ok = None

    # -- time cropping (losses.py:50-75) ---------------------------------------------------------------
    def _window(self, n_samples: int):
        use_train = self.training and (self.tmin_train is not None or self.tmax_train is not None)
        tmin, tmax = (self.tmin_train, self.tmax_train) if use_train else (self.tmin, self.tmax)
        start, stop = 0, n_samples
        if tmin is not None or tmax is not None:
            assert self.dset_args is not None and self.dset_args.tmin is not None
            origin, rate = self.dset_args.tmin, self.dset_args.sample_rate
            if tmin is not None:
                assert tmin >= origin, 'clip.tmin should be above dset.tmin'
                start = int((tmin - origin) * rate)
            if tmax is not None:
                stop = int((tmax - origin) * rate)
        return start, stop

    def trim_samples(self, estimates, candidates):
        start, stop = self._window(estimates.shape[-1])
        return estimates[..., start:stop], candidates[..., start:stop]

    def _prepare(self, estimates, candidates):
        estimates, candidates = self.trim_samples(estimates, candidates)
        if self.pool:                            # losses.py:85-87
            estimates = estimates.mean(dim=2, keepdim=True)
            candidates = candidates.mean(dim=2, keepdim=True)
        if self.center:                          # losses.py:88-90
            estimates = estimates - estimates.mean(dim=(1, 2), keepdim=True)
            candidates = candidates - candidates.mean(dim=(1, 2), keepdim=True)
        return estimates, candidates

    def get_scores(self, estimates: torch.Tensor, candidates: torch.Tensor):
        """[B, C, T] x [B', C, T] -> [B, B'] matching scores (no autograd; use forward() for training)."""
        estimates, candidates = self._prepare(estimates, candidates)
        return BF.clip_scores(estimates, candidates)

    def get_probabilities(self, estimates, candidates):
        estimates, candidates = self._prepare(estimates, candidates)
        return BF.clip_scores(estimates, candidates, want_probs=True)

    def prefetch_candidates(self, candidate: torch.Tensor) -> None:
        """Optional (multi-GPU, global_negatives): start the candidate all-gather now -- e.g. right after the batch reaches
        the device, before the encoder forward -- so that it overlaps compute.  `forward` picks it up when it is called
        with the same tensor; without this call the gather simply happens inside `forward`."""
        if self.global_negatives and distrib.world_size() > 1 and not candidate.requires_grad \
                and not (self.pool or self.center) \
                and self._window(candidate.shape[-1]) == (0, candidate.shape[-1]):
            self._prefetched = distrib.CandidateGather(candidate, self.uniform_batches)

    def _check_mask(self, mask) -> None:
        """losses.py:110 `assert mask.all()`: on a CUDA mask that is a device->host sync per call.  The verdict is kept per
        mask tensor OBJECT (weak reference + version counter), so a caller that reuses one all-true mask pays it once; a fresh
        mask per batch (what bm/solver.py passes) is checked every time, exactly like the reference."""
        seen = self._mask_ok
        if seen is not None and seen[0]() is mask and seen[1] == mask._version:
            return
        assert mask.all(), "mask is not supported for now"
        self._mask_ok = (weakref.ref(mask), mask._version)

    def forward(self, estimate, candidate, mask=None):
        self._check_mask(mask)
        assert estimate.size(0) <= candidate.size(0), "need at least as many targets as estimates"
        pre, self._prefetched = self._prefetched, None
        if candidate.requires_grad and torch.is_grad_enabled() and self.global_negatives and distrib.world_size() > 1:
            # a trainable feature model made the candidates: differentiable gather (reduce-scatter of dC in backward)
            estimate, candidate = self._prepare(estimate, candidate)
            candidate, offset = distrib.all_gather_candidates_with_grad(candidate, self.uniform_batches)
            return BF.clip_loss(estimate, candidate, offset)
        if pre is not None and pre.source is candidate:
            estimate, _ = self._prepare(estimate, candidate)
            candidate, offset = pre.wait()
            return BF.clip_loss(estimate, candidate, offset)
        estimate, candidate = self._prepare(estimate, candidate)
        offset = 0
        if self.global_negatives and distrib.world_size() > 1:
            candidate, offset = distrib.all_gather_candidates(candidate, self.uniform_batches)
        return BF.clip_loss(estimate, candidate, offset)
