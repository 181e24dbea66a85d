"""TEST INFRASTRUCTURE ONLY -- generates the regression-objective fixtures by running the VERBATIM reference modules
(bm/losses.py L1Loss / L2Loss, bm/models/simpleconv.py, loaded by `oracle/ref_loader.py`) on small seeded inputs.

    python oracle/make_regression_golden.py          # rewrites tests/golden/regression_{losses,train}.npz

regression_losses.npz, per case `<case>.`: estimate, output, mask, and for p = 1 (L1Loss) and 2 (L2Loss) `l<p>.loss`,
`l<p>.grad_estimate`, `l<p>.grad_output` (both inputs require grad).  The cases cover the masks the solver and its users
pass: all-true and half-true [B,1,T] (features_mask), a full [B,F,T] mask, one selected element, NaN / inf planted where
nothing is selected, and exact ties e == o (where L1's gradient is sign(0) = 0).
regression_train.npz: one step of a depth-10 clip_conv SimpleConv against mel-like targets (F = 40) under a partial
[B,1,T] mask and L2Loss, in the layout of `make_golden._model_case` (initial state as seed + digest, sampled gradients).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import make_golden, ref_loader  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name: (B, F, T, mask kind)
LOSS_CASES = {
    "all_true": (2, 6, 8, "all"),
    "half": (3, 5, 9, "half"),
    "full_mask": (2, 4, 12, "full"),
    "single": (1, 3, 5, "single"),
    "nonfinite": (3, 4, 8, "nonfinite"),
    "ties": (2, 5, 7, "ties"),
}
TRAIN = dict(seed=611, B=5, C=12, T=33, F=40, S=3, hidden=24, MC=16, IL=20, P=72, n_valid=[12, 8, 12])


def loss_case_inputs(B, F, T, kind, g: torch.Generator):
    """(estimate, output, mask) of one case, drawn from `g`."""
    est = torch.randn(B, F, T, generator=g)
    out = torch.randn(B, F, T, generator=g)
    if kind == "all":
        mask = torch.ones(B, 1, T, dtype=torch.bool)
    elif kind == "full":
        mask = torch.rand(B, F, T, generator=g) < 0.5
    elif kind == "single":
        mask = torch.zeros(B, F, T, dtype=torch.bool)
        mask[0, F // 2, T // 2] = True
    else:
        mask = torch.rand(B, 1, T, generator=g) < 0.5
        mask[0, 0, 0], mask[-1, 0, -1] = True, False            # never empty, never full
    if kind == "nonfinite":
        off = ~mask.expand_as(est)
        vals = torch.tensor([float("nan"), float("inf"), -float("inf")])
        idx = torch.nonzero(off)
        for i, (b, f, t) in enumerate(idx.tolist()):
            if i % 2 == 0:
                est[b, f, t] = vals[i % 3]
            else:
                out[b, f, t] = vals[(i + 1) % 3]
    if kind == "ties":
        tie = torch.rand(B, F, T, generator=g) < 0.3
        out = torch.where(tie, est, out)
    return est, out, mask


def run_losses(name="regression_losses"):
    _, _, losses = ref_loader.load_reference()
    g = torch.Generator().manual_seed(4242)
    out = {}
    for case, (B, F, T, kind) in LOSS_CASES.items():
        est, tgt, mask = loss_case_inputs(B, F, T, kind, g)
        out[case + ".estimate"], out[case + ".output"], out[case + ".mask"] = est.numpy(), tgt.numpy(), mask.numpy()
        for p, cls in ((1, losses.L1Loss), (2, losses.L2Loss)):
            e, o = est.clone().requires_grad_(True), tgt.clone().requires_grad_(True)
            loss = cls()(e, o, mask)
            loss.backward()
            out[f"{case}.l{p}.loss"] = loss.detach().numpy()
            out[f"{case}.l{p}.grad_estimate"] = e.grad.numpy()
            out[f"{case}.l{p}.grad_output"] = o.grad.numpy()
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: {len(LOSS_CASES)} cases, size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


def run_train(name="regression_train"):
    """The reference's estimate, L2 loss and parameter gradients after one train-mode forward/backward of clip_conv
    against mel-like targets under a partial features mask."""
    c = TRAIN
    common, simpleconv, losses = ref_loader.load_reference()
    seed, B, C, T, F, S = c["seed"], c["B"], c["C"], c["T"], c["F"], c["S"]
    torch.manual_seed(seed)
    kw = ref_loader.clip_conv_kwargs(hidden=c["hidden"], depth=10, merger_channels=c["MC"], initial_linear=c["IL"],
                                     merger_pos_dim=c["P"])
    model = simpleconv.SimpleConv(in_channels=dict(meg=C), out_channels=F, n_subjects=S, **kw)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    meg = torch.randn(B, C, T).clamp_(-20, 20)
    targets = torch.randn(B, F, T).abs()                       # mel-like: non-negative
    mask = torch.rand(B, 1, T) < 0.7
    subj = torch.randint(0, S, (B,))
    n_valid = c["n_valid"]
    recs = [ref_loader.FakeRecording(s, C, n_valid[s], seed=seed) for s in range(S)]
    for b in range(B):
        meg[b, n_valid[int(subj[b])]:] = 0
    batch = ref_loader.FakeBatch(meg, subj, [recs[int(s)] for s in subj])
    pos = torch.full((S, C, 2), common.PositionGetter.INVALID)
    for s in range(S):
        lay = model.merger.position_getter.get_recording_layout(recs[s])
        pos[s, :len(lay)] = lay
    model.train()
    torch.manual_seed(seed + 1)
    ban = torch.rand(2)
    torch.manual_seed(seed + 1)
    est = model(dict(meg=meg.clone()), batch)
    loss = losses.L2Loss()(est, targets, mask)
    loss.backward()
    out = make_golden._model_case([B, B, C, T, F, S, c["hidden"], 10, c["MC"], c["IL"], c["P"], 1], meg, targets, subj,
                                  pos, ban, est, loss, state, model.named_parameters())
    out["features_mask"] = mask.numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: loss={loss.item():.6f} size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


if __name__ == "__main__":
    torch.set_num_threads(1)
    run_losses()
    run_train()
