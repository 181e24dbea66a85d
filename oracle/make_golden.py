"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the VERBATIM reference modules
(bm/models/simpleconv.py, bm/models/common.py, bm/losses.py loaded by `oracle/ref_loader.py`) on small seeded
inputs, in this build container (the reference tree does not travel to the GPU box; the fixtures do).

    python oracle/make_golden.py            # rewrites tests/golden/

Each fixture holds: the configuration, the reference state_dict (`p.<key>`), the inputs, and the reference's
outputs: estimate, scores, loss, probabilities, every parameter gradient (`g.<key>`), and BN running stats after
the step (`bn.<key>`).  Everything fp32, produced by the reference's own code path:
    estimate = SimpleConv(...)(dict(meg=meg), batch)            simpleconv.py:198
    loss     = ClipLoss()(estimate, candidates, mask)           losses.py:104
    loss.backward()                                             solver.py:385
The fixtures of `run_fresh` / `run_train_forward` keep them smaller: a digest of the initial state instead of the state,
and a fixed sample of each larger gradient (`_model_case`); `seeded_init.json` holds per-tensor digests only.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import zlib

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = {
    # name: dict(B, Bc, C, T, F, S, hidden, depth, MC, IL, P, train, n_valid per recording)
    "train_small": dict(B=6, Bc=6, C=10, T=24, F=8, S=3, hidden=16, depth=10, MC=12, IL=12, P=32,
                        train=True, n_valid=None, seed=1),
    "eval_small": dict(B=5, Bc=5, C=10, T=24, F=8, S=3, hidden=16, depth=10, MC=12, IL=12, P=32,
                       train=False, n_valid=None, seed=2),
    "train_padded_negs": dict(B=8, Bc=11, C=14, T=37, F=12, S=4, hidden=32, depth=10, MC=20, IL=24, P=72,
                              train=True, n_valid=[14, 9, 6, 14], seed=3),
    "train_depth4": dict(B=4, Bc=4, C=7, T=50, F=5, S=2, hidden=24, depth=4, MC=8, IL=8, P=8,
                         train=True, n_valid=None, seed=4),
}


def run_case(name, c):
    common, simpleconv, losses = ref_loader.load_reference()
    torch.manual_seed(100 + c["seed"])
    kw = ref_loader.clip_conv_kwargs(hidden=c["hidden"], depth=c["depth"], merger_channels=c["MC"],
                                     initial_linear=c["IL"], merger_pos_dim=c["P"])
    model = simpleconv.SimpleConv(in_channels=dict(meg=c["C"]), out_channels=c["F"], n_subjects=c["S"], **kw)
    clip = losses.ClipLoss()
    # make BN affine / running stats non-trivial so that parity actually exercises them
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.add_(0.1 * torch.randn_like(m.weight))
                m.bias.add_(0.1 * torch.randn_like(m.bias))
                m.running_mean.add_(0.1 * torch.randn_like(m.running_mean))
                m.running_var.mul_(1 + 0.2 * torch.rand_like(m.running_var))
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}

    B, Bc, C, T, F, S = c["B"], c["Bc"], c["C"], c["T"], c["F"], c["S"]
    meg = torch.randn(B, C, T).clamp_(-20, 20)
    cand = torch.randn(Bc, F, T)
    subj = torch.randint(0, S, (B,))
    nv = c["n_valid"] or [C] * S
    recs = [ref_loader.FakeRecording(s, C, nv[s], seed=c["seed"]) for s in range(S)]
    for b in range(B):
        meg[b, nv[int(subj[b])]:] = 0
    batch = ref_loader.FakeBatch(meg, subj, [recs[int(s)] for s in subj])
    pos_rec = torch.stack([model.merger.position_getter.get_recording_layout(r).clone() for r in recs])
    full = torch.full((S, C, 2), common.PositionGetter.INVALID)
    full[:, :pos_rec.shape[1]] = pos_rec

    model.train(c["train"])
    clip.train(c["train"])
    torch.manual_seed(9000 + c["seed"])
    ban = torch.rand(2)                       # the ONE rand(2) the forward will draw (common.py:343)
    torch.manual_seed(9000 + c["seed"])
    est = model(dict(meg=meg.clone()), batch)
    mask = torch.ones(B, 1, T, dtype=torch.bool)
    loss = clip(est, cand, mask)
    scores = clip.get_scores(est, cand)
    probs = clip.get_probabilities(est, cand)
    loss.backward()

    out = dict(cfg=np.array([B, Bc, C, T, F, S, c["hidden"], c["depth"], c["MC"], c["IL"], c["P"],
                             int(c["train"])], dtype=np.int64),
               meg=meg.numpy(), candidates=cand.numpy(), subject_index=subj.numpy(),
               rec_positions=full.numpy(), rec_of_sample=subj.numpy(), ban_centre=ban.numpy(),
               estimate=est.detach().numpy(), scores=scores.detach().numpy(), loss=loss.detach().numpy(),
               probs=probs.detach().numpy())
    for k, v in state.items():
        out["p." + k] = v.numpy()
    for k, v in model.named_parameters():
        out["g." + k] = v.grad.numpy() if v.grad is not None else np.zeros(0, np.float32)
    for k, v in model.state_dict().items():
        if "running" in k or "num_batches" in k:
            out["bn." + k] = v.numpy()
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: loss={loss.item():.6f} est.std={est.std().item():.4f} "
          f"size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


def run_prep(name="prep_small"):
    """bm/norm.py verbatim (RobustScaler.fit/transform, StandardScaler, BatchScaler._transform, ScaleReject) on a
    small batch that mixes three recordings, holds an out-of-range sample, a zero-padded channel and an empty
    features mask; plus the offset crop of solver.py:262-274 applied with plain slicing."""
    norm = ref_loader.load_reference_norm()
    torch.manual_seed(4242)
    B, C, T, off = 7, 6, 30, 3
    fb = ref_loader.FakeFeaturesBuilder({"a": (3, True), "b": (2, False)})
    rec_ids = [4, 9, 11]
    out = {}
    for per_channel in (False, True):
        scaler = norm.BatchScaler(fb, per_channel=per_channel)
        torch.manual_seed(4242)
        for i, r in enumerate(rec_ids):
            fit = torch.randn(400, C) * (0.5 + i) + 0.3 * i
            fit[:, C - 1] = 0 if i == 1 else fit[:, C - 1]      # padded channel -> scale_ forced to 1 (norm.py:73-76)
            s = norm.RobustScaler()
            s.fit(fit)
            scaler.meg_scalers[r] = s
            out[f"fit.meg.{r}"] = fit.numpy()
        feats_fit = torch.randn(50, fb.dimension, T) * 2 + 1
        mask_fit = torch.ones(50, 1, T, dtype=torch.bool)
        mask_fit[::7, :, ::3] = False
        out["fit.features"], out["fit.features_mask"] = feats_fit.numpy(), mask_fit.numpy()
        for fname, fs in scaler.feature_scalers.items():
            fs.fit(norm._as_nd(feats_fit[:, fb.get_slice(fname)]), norm._as_nd(mask_fit))
        meg = torch.randn(B, C, T) * 2
        meg[2, 1, 5] = 90.0                                      # > limit after scaling -> rejected / clipped
        meg[5, 0, 0] = -75.0
        rec = torch.tensor([4, 11, 9, 9, 4, 11, 4])
        features = torch.randn(B, fb.dimension, T)
        fmask = torch.ones(B, 1, T, dtype=torch.bool)
        fmask[3] = False                                         # empty features (exclude_empty_features)
        tag = "pc1." if per_channel else "pc0."
        out[tag + "meg_center"] = np.stack([scaler.meg_scalers[r].center_.numpy() for r in rec_ids])
        out[tag + "meg_scale"] = np.stack([scaler.meg_scalers[r].scale_.numpy() for r in rec_ids])
        fc = torch.zeros(fb.dimension)
        fsc = torch.ones(fb.dimension)
        for fname, fs in scaler.feature_scalers.items():
            if isinstance(fs, norm.StandardScaler):
                fc[fb.get_slice(fname)] = fs.center_
                fsc[fb.get_slice(fname)] = fs.scale_
        out[tag + "feat_center"], out[tag + "feat_scale"] = fc.numpy(), fsc.numpy()
        batch = ref_loader.FakeSegmentBatch(meg.clone(), features.clone(), fmask.clone(), rec.clone())
        tr = scaler.transform(batch)
        out[tag + "transform.meg"], out[tag + "transform.features"] = tr.meg.numpy(), tr.features.numpy()
        inv = scaler.inverse_transform(tr)
        out[tag + "inverse.meg"], out[tag + "inverse.features"] = inv.meg.numpy(), inv.features.numpy()
        for clip in (False, True):
            for excl in (False, True):
                sr = norm.ScaleReject(scaler, limit=20.0, exclude_empty_features=excl, clip=clip)
                kept, keep = sr(ref_loader.FakeSegmentBatch(meg.clone(), features.clone(), fmask.clone(), rec.clone()))
                k = f"{tag}clip{int(clip)}.excl{int(excl)}."
                out[k + "keep"] = keep.numpy()
                out[k + "meg"] = kept.meg[..., off:].contiguous().numpy()               # solver.py:264
                out[k + "features"] = kept.features[..., :-off].contiguous().numpy()    # solver.py:273
                out[k + "features_mask"] = kept.features_mask[..., :-off].contiguous().numpy()
                out[k + "rejection_rate"] = np.float64(sr.rejection_rate)
    out.update(meg=meg.numpy(), features=features.numpy(), features_mask=fmask.numpy(), recording_index=rec.numpy(),
               rec_ids=np.array(rec_ids), offset=np.int64(off), limit=np.float32(20.0))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: {len(out)} arrays, size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


def run_retrieval(name="retrieval_small"):
    """Verbatim `ClipLoss.get_probabilities` (bm/losses.py:97-102) driven by the evaluation loops of
    scripts/run_eval_probs.py:237-307 and bm/wer.py:80-116.  Those two files import flashy / dora / omegaconf and a
    Solver, so the loops themselves are the restatement in `oracle/eval_oracle.py`; the arithmetic is the reference's."""
    from oracle import eval_oracle
    _, _, losses = ref_loader.load_reference()
    clip = losses.ClipLoss().eval()
    probs_fn = lambda e, c: clip.get_probabilities(e, c)   # noqa: E731
    torch.manual_seed(777)
    N, M, F, T = 24, 17, 6, 20
    trues = torch.randn(M, F, T)
    seg_of_pred = torch.randint(0, M, (N,))
    preds = 0.12 * trues[seg_of_pred] + torch.randn(N, F, T)
    vocab_labels = torch.randperm(10_000)[:M] * 7919 - 31_000_000          # int64 "segment hashes"
    target_labels = vocab_labels[seg_of_pred]
    out = dict(preds=preds.numpy(), trues=trues.numpy(), vocab_labels=vocab_labels.numpy(),
               target_labels=target_labels.numpy())
    probs = eval_oracle.builds_probs(preds, trues, batch_size=10, probabilities=probs_fn)
    out["probs"] = probs.numpy()
    out["acc"] = np.array([eval_oracle.accuracy_from_probs(probs, target_labels, vocab_labels, k) for k in (1, 5, 10)])
    window = eval_oracle.crop_window(-0.5, 120.0, -0.45, -0.4)
    out["window"] = np.array(window)
    out["probs_window"] = eval_oracle.builds_probs(preds, trues, 10, window, probs_fn).numpy()
    # wer ranking: 12 estimates, 5 distinct words, 9 negatives
    n, n_neg, topx = 12, 9, 3
    word_hashes = torch.tensor([11, 23, 11, 35, 47, 23, 59, 11, 35, 47, 23, 59], dtype=torch.int32)
    outputs = torch.randn(n, F, T)
    estimates = 0.15 * outputs + torch.randn(n, F, T)
    kept = torch.randperm(n)[:n_neg]
    negatives, negative_hashes = outputs[kept], word_hashes[kept]
    res = eval_oracle.wer_ranking(estimates, word_hashes, outputs, negatives, negative_hashes, topx, probs_fn)
    out.update(wer_estimates=estimates.numpy(), wer_outputs=outputs.numpy(), wer_word_hashes=word_hashes.numpy(),
               wer_negatives=negatives.numpy(), wer_negative_hashes=negative_hashes.numpy(), wer_topx=np.int64(topx),
               wer=np.float64(res["wer"]), wer_vocab=np.float64(res["wer_vocab"]),
               wer_soft=np.float64(res["soft_correct"]))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: acc@1/5/10={out['acc']} wer={res} window={window}")


DEEPMEL_CASES = {
    # conf/feature_model/deep_mel.yaml scaled down; "b" has a residual on its very first layer and GELU
    "deepmel_small": dict(n_in=10, params=dict(n_hidden_channels=16, n_hidden_layers=4, n_out_channels=24, kernel=3,
                                                stride=1, dilation_growth=2, dilation_period=5, batch_norm=True,
                                                activation_on_last=False, skip=True, glu_context=1, glu=2),
                          B=5, T=20, seed=31),
    "deepmel_nobn": dict(n_in=12, params=dict(n_hidden_channels=12, n_hidden_layers=3, n_out_channels=12, kernel=3,
                                               stride=1, dilation_growth=2, dilation_period=2, batch_norm=False,
                                               activation_on_last=False, skip=True, glu_context=0, glu=3,
                                               leakiness=0.1),
                         B=4, T=17, seed=32),
}


def run_deepmel(name, c):
    """Verbatim DeepMel (bm/models/features.py) -> candidates, verbatim ClipLoss against a random `estimate` that
    requires grad; one training forward/backward (parameter, estimate AND candidate-side gradients), then an eval-mode
    forward with the updated running statistics."""
    import importlib.util
    _, _, losses = ref_loader.load_reference()
    spec = importlib.util.spec_from_file_location("bm.models.features", ref_loader.REF + "/models/features.py")
    feats = importlib.util.module_from_spec(spec)
    sys.modules["bm.models.features"] = feats
    spec.loader.exec_module(feats)
    torch.manual_seed(c["seed"])
    model = feats.DeepMel(n_in_channels=c["n_in"], **c["params"])
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.add_(0.1 * torch.randn_like(m.weight))
                m.bias.add_(0.1 * torch.randn_like(m.bias))
                m.running_mean.add_(0.1 * torch.randn_like(m.running_mean))
                m.running_var.mul_(1 + 0.2 * torch.rand_like(m.running_var))
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    B, T = c["B"], c["T"]
    mel = torch.randn(B, c["n_in"], T)
    n_out = c["params"]["n_out_channels"]
    estimate = torch.randn(B, n_out, T, requires_grad=True)
    clip = losses.ClipLoss()
    model.train()
    cand = model(mel)
    cand.retain_grad()
    loss = clip(estimate, cand, torch.ones(B, 1, T, dtype=torch.bool))
    loss.backward()
    out = dict(mel=mel.numpy(), estimate=estimate.detach().numpy(), candidates=cand.detach().numpy(),
               loss=loss.detach().numpy(), **{"g.estimate": estimate.grad.numpy(), "g.candidates": cand.grad.numpy()})
    for k, v in state.items():
        out["p." + k] = v.numpy()
    for k, v in model.named_parameters():
        out["g." + k] = v.grad.numpy()
    for k, v in model.state_dict().items():
        if "running" in k or "num_batches" in k:
            out["bn." + k] = v.numpy()
    model.eval()
    with torch.no_grad():
        out["candidates_eval"] = model(mel).numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: loss={float(loss):.6f} cand.std={float(cand.std()):.4f} "
          f"|d_cand|={float(cand.grad.norm()):.4e} size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


# The ablation table of the paper (grids/nmi/ablation_final.py:42-52), each as a change to the small clip_conv case
ABLATION_BASE = dict(B=6, C=10, T=24, F=8, S=3, hidden=16, depth=4, MC=12, IL=12, P=32, seed=41)
ABLATIONS = {
    "ablation_reference": {},
    "ablation_no_merger": dict(merger=False),
    "ablation_no_initial_linear": dict(initial_linear=0),
    "ablation_no_glu": dict(glu=0),
    "ablation_relu": dict(gelu=False),
    "ablation_no_skip": dict(skip=False),
    "ablation_no_complex_out": dict(complex_out=False),
    "ablation_no_subject_layers": dict(subject_layers=False),
    "ablation_subject_embedding": dict(subject_layers=False, subject_dim=5),
    "ablation_subsample_channels": dict(subsample_meg_channels=6),
}


def run_ablation(name, change):
    """Verbatim SimpleConv with one constructor change, one training step with the verbatim ClipLoss."""
    c = dict(ABLATION_BASE)
    common, simpleconv, losses = ref_loader.load_reference()
    torch.manual_seed(c["seed"])
    kw = ref_loader.clip_conv_kwargs(hidden=c["hidden"], depth=c["depth"], merger_channels=c["MC"],
                                     initial_linear=c["IL"], merger_pos_dim=c["P"])
    kw.update(change)
    model = simpleconv.SimpleConv(in_channels=dict(meg=c["C"]), out_channels=c["F"], n_subjects=c["S"], **kw)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.add_(0.1 * torch.randn_like(m.weight))
                m.bias.add_(0.1 * torch.randn_like(m.bias))
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    B, C, T, F, S = c["B"], c["C"], c["T"], c["F"], c["S"]
    meg = torch.randn(B, C, T).clamp_(-20, 20)
    cand = torch.randn(B, F, T)
    subj = torch.randint(0, S, (B,))
    recs = [ref_loader.FakeRecording(s, C, C, seed=c["seed"]) for s in range(S)]
    batch = ref_loader.FakeBatch(meg, subj, [recs[int(s)] for s in subj])
    getter = common.PositionGetter()
    pos = torch.stack([getter.get_recording_layout(r).clone() for r in recs])
    model.train()
    torch.manual_seed(9100 + c["seed"])
    ban = torch.rand(2)
    torch.manual_seed(9100 + c["seed"])
    est = model(dict(meg=meg.clone()), batch)
    loss = losses.ClipLoss()(est, cand, torch.ones(B, 1, T, dtype=torch.bool))
    loss.backward()
    out = dict(meg=meg.numpy(), candidates=cand.numpy(), subject_index=subj.numpy(), rec_positions=pos.numpy(),
               ban_centre=ban.numpy(), estimate=est.detach().numpy(), loss=loss.detach().numpy())
    for k, v in state.items():
        out["p." + k] = v.numpy()
    for k, v in model.named_parameters():
        out["g." + k] = v.grad.numpy() if v.grad is not None else np.zeros(0, np.float32)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: loss={loss.item():.6f} est.std={est.std().item():.4f} params={sum(v.numel() for v in state.values())}")


GRAD_SAMPLE = 256


def tensor_sha256(t) -> str:
    return hashlib.sha256(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def state_sha256(state) -> str:
    """One digest over the keys, shapes, dtypes and bytes of a state_dict, in its order."""
    h = hashlib.sha256()
    for k, v in state.items():
        h.update(f"{k} {tuple(v.shape)} {v.dtype} {tensor_sha256(v)}\n".encode())
    return h.hexdigest()


def grad_sample(key: str, numel: int) -> np.ndarray:
    """The flat entries of parameter `key`'s gradient a fixture keeps: all of them up to GRAD_SAMPLE, else a fixed
    sample of GRAD_SAMPLE (seeded by the name; numpy's legacy RandomState stream does not change between versions)."""
    if numel <= GRAD_SAMPLE:
        return np.arange(numel)
    return np.sort(np.random.RandomState(zlib.crc32(key.encode())).choice(numel, GRAD_SAMPLE, replace=False))


def seeded_state(cfg, seed, sha256):
    """The initial clip_conv state_dict of the package's SimpleConv under torch.manual_seed(seed), checked against the
    digest of the reference's (`sha256`: the raw bytes a `_model_case` fixture stores)."""
    import brainmagick_b200 as bb
    torch.manual_seed(seed)
    model = bb.SimpleConv(in_channels=dict(meg=cfg.in_channels), out_channels=cfg.out_channels, n_subjects=cfg.n_subjects,
                          **ref_loader.clip_conv_kwargs(hidden=cfg.hidden, depth=cfg.depth, merger_channels=cfg.merger_channels,
                                                        initial_linear=cfg.initial_linear, merger_pos_dim=cfg.merger_pos_dim))
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    assert state_sha256(state) == bytes(np.asarray(sha256, dtype=np.uint8)).hex(), \
        "the seeded initial state is not the reference's"
    return state


def _model_case(cfg, meg, cand, subj, pos, ban, est, loss, state, params=()):
    """A fixture in the layout of `run_case` (readable by tests/conftest.load_golden) that holds the digest of the
    reference's initial state instead of the state itself: the package's SimpleConv rebuilds it bit for bit from the same
    seed (tests/test_boundary.py).  Gradients of `params`: the `grad_sample` entries and the norm of the whole."""
    out = dict(cfg=np.array(cfg, dtype=np.int64), meg=meg.numpy(), candidates=cand.numpy(), subject_index=subj.numpy(),
               rec_positions=pos.numpy(), rec_of_sample=subj.numpy(), ban_centre=ban.numpy(),
               estimate=est.detach().numpy(), loss=loss.detach().numpy(),
               state_sha256=np.frombuffer(bytes.fromhex(state_sha256(state)), dtype=np.uint8))
    for k, v in params:
        if v.grad is not None:
            out["g." + k] = v.grad.numpy().ravel()[grad_sample(k, v.grad.numel())]
            out["gnorm." + k] = np.float64(v.grad.double().norm())
    return out


FRESH_CASES = {"fresh_train": dict(seed=501, train=True), "fresh_eval": dict(seed=502, train=False)}


def run_fresh(name, c):
    """A depth-10 clip_conv with partly valid recordings, neither BN-perturbed nor shaped like the CASES: the
    reference's estimate, loss and parameter gradients after one forward/backward in train or eval mode."""
    seed, train = c["seed"], c["train"]
    common, simpleconv, losses = ref_loader.load_reference()
    torch.manual_seed(seed)
    B, C, T, F, S, hidden, MC, IL, P = 7, 13, 41, 9, 4, 24, 16, 20, 72
    kw = ref_loader.clip_conv_kwargs(hidden=hidden, depth=10, merger_channels=MC, initial_linear=IL, merger_pos_dim=P)
    model = simpleconv.SimpleConv(in_channels=dict(meg=C), out_channels=F, n_subjects=S, **kw)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    meg = torch.randn(B, C, T).clamp_(-20, 20)
    cand = torch.randn(B + 3, F, T)
    subj = torch.randint(0, S, (B,))
    n_valid = [13, 9, 13, 6]
    recs = [ref_loader.FakeRecording(s, C, n_valid[s], seed=seed) for s in range(S)]
    for b in range(B):
        meg[b, n_valid[int(subj[b])]:] = 0
    batch = ref_loader.FakeBatch(meg, subj, [recs[int(s)] for s in subj])
    pos = torch.full((S, C, 2), common.PositionGetter.INVALID)
    for s in range(S):
        lay = model.merger.position_getter.get_recording_layout(recs[s])
        pos[s, :len(lay)] = lay
    model.train(train)
    torch.manual_seed(seed + 1)
    ban = torch.rand(2)
    torch.manual_seed(seed + 1)
    est = model(dict(meg=meg.clone()), batch)
    loss = losses.ClipLoss()(est, cand, torch.ones(B, 1, T, dtype=torch.bool))
    loss.backward()
    out = _model_case([B, B + 3, C, T, F, S, hidden, 10, MC, IL, P, int(train)], meg, cand, subj, pos, ban, est, loss,
                      state, model.named_parameters())
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: loss={loss.item():.6f} size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


def run_train_forward(name="train_forward"):
    """A train-mode forward and loss at merger_pos_dim 128 with every channel valid (no backward)."""
    common, simpleconv, losses = ref_loader.load_reference()
    torch.manual_seed(1234)
    C, F, S, T, B = 9, 6, 3, 31, 5
    kw = ref_loader.clip_conv_kwargs(hidden=20, depth=10, merger_channels=8, initial_linear=12, merger_pos_dim=128)
    model = simpleconv.SimpleConv(in_channels=dict(meg=C), out_channels=F, n_subjects=S, **kw)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    meg, cand = torch.randn(B, C, T), torch.randn(B, F, T)
    subj = torch.randint(0, S, (B,))
    recs = [ref_loader.FakeRecording(s, C, seed=5) for s in range(S)]
    batch = ref_loader.FakeBatch(meg, subj, [recs[int(s)] for s in subj])
    pos = torch.stack([model.merger.position_getter.get_recording_layout(r) for r in recs])
    model.train()
    torch.manual_seed(7)
    ban = torch.rand(2)
    torch.manual_seed(7)
    est = model(dict(meg=meg.clone()), batch)
    loss = losses.ClipLoss()(est, cand, torch.ones(B, 1, T, dtype=torch.bool))
    out = _model_case([B, B, C, T, F, S, 20, 10, 8, 12, 128, 1], meg, cand, subj, pos, ban, est, loss, state)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: loss={loss.item():.6f} size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


def run_prep_fresh(name="prep_fresh"):
    """bm/norm.py ScaleReject (clip off and on) on scalers fitted to other data than prep_small's, per channel."""
    norm = ref_loader.load_reference_norm()
    torch.manual_seed(77)
    B, C, T, off = 9, 8, 25, 2
    fb = ref_loader.FakeFeaturesBuilder({"w": (4, True), "p": (3, False)})
    scaler = norm.BatchScaler(fb, per_channel=True)
    ids = [2, 3, 10]
    for r in ids:
        scaler.meg_scalers[r] = norm.RobustScaler().fit(torch.randn(300, C) * (1 + r))
    feats_fit = torch.randn(40, fb.dimension, T)
    for fname, fs in scaler.feature_scalers.items():
        fs.fit(norm._as_nd(feats_fit[:, fb.get_slice(fname)]), norm._as_nd(torch.ones(40, 1, T, dtype=torch.bool)))
    meg = torch.randn(B, C, T) * 40
    rec = torch.tensor([2, 10, 3, 3, 2, 10, 10, 2, 3])
    feats = torch.randn(B, fb.dimension, T)
    mask = torch.ones(B, 1, T, dtype=torch.bool)
    fc, fs_ = torch.zeros(fb.dimension), torch.ones(fb.dimension)
    for fname, sc in scaler.feature_scalers.items():
        if isinstance(sc, norm.StandardScaler):
            fc[fb.get_slice(fname)], fs_[fb.get_slice(fname)] = sc.center_, sc.scale_
    out = dict(rec_ids=np.array(ids), meg_center=np.stack([scaler.meg_scalers[r].center_.numpy() for r in ids]),
               meg_scale=np.stack([scaler.meg_scalers[r].scale_.numpy() for r in ids]), feat_center=fc.numpy(),
               feat_scale=fs_.numpy(), meg=meg.numpy(), recording_index=rec.numpy(), features=feats.numpy(),
               features_mask=mask.numpy(), offset=np.int64(off), limit=np.float32(20.0))
    for clip in (False, True):
        sr = norm.ScaleReject(scaler, limit=20.0, clip=clip)
        kept, keep = sr(ref_loader.FakeSegmentBatch(meg.clone(), feats.clone(), mask.clone(), rec.clone()))
        out[f"clip{int(clip)}.keep"] = keep.numpy()
        out[f"clip{int(clip)}.meg"] = kept.meg[..., off:].contiguous().numpy()
        out[f"clip{int(clip)}.features"] = kept.features[..., :-off].contiguous().numpy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: {len(out)} arrays, size={os.path.getsize(os.path.join(OUT, name + '.npz')) / 1024:.0f} KiB")


SEEDED_INIT = dict(seed=77, C=30, F=17, S=5, hidden=48, MC=20, IL=24, P=128)


def run_seeded_init(name="seeded_init"):
    """The reference's freshly constructed clip_conv state_dict under torch.manual_seed (bm/train.py:76,109 model_hash)."""
    c = SEEDED_INIT
    _, simpleconv, _ = ref_loader.load_reference()
    kw = dict(ref_loader.CLIP_CONV, hidden=dict(meg=c["hidden"]), merger_channels=c["MC"], initial_linear=c["IL"],
              merger_pos_dim=c["P"])
    torch.manual_seed(c["seed"])
    model = simpleconv.SimpleConv(in_channels=dict(meg=c["C"]), out_channels=c["F"], n_subjects=c["S"], **kw)
    out = dict(spec=c, subject_layers_repr=repr(model.subject_layers),
               state=[dict(key=k, shape=list(v.shape), dtype=str(v.dtype), sha256=tensor_sha256(v))
                      for k, v in model.state_dict().items()])
    with open(os.path.join(OUT, name + ".json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(f"{name}: {len(out['state'])} tensors")


if __name__ == "__main__":
    torch.set_num_threads(1)
    wanted = sys.argv[1:]
    for name, c in CASES.items():
        if not wanted or name in wanted:
            run_case(name, c)
    if not wanted or "prep_small" in wanted:
        run_prep()
    if not wanted or "retrieval_small" in wanted:
        run_retrieval()
    for name, c in DEEPMEL_CASES.items():
        if not wanted or name in wanted:
            run_deepmel(name, c)
    for name, change in ABLATIONS.items():
        if not wanted or name in wanted:
            run_ablation(name, change)
    for name, c in FRESH_CASES.items():
        if not wanted or name in wanted:
            run_fresh(name, c)
    for name, fn in (("train_forward", run_train_forward), ("prep_fresh", run_prep_fresh), ("seeded_init", run_seeded_init)):
        if not wanted or name in wanted:
            fn(name)
