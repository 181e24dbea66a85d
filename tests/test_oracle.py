"""CPU: pins the oracle restatement (oracle/bm_oracle.py) against the golden vectors produced by the verbatim
reference modules (oracle/make_golden.py), among them a second, separately seeded configuration (train_forward)."""
import torch

from oracle import bm_oracle, make_golden
from conftest import load_golden, rel_err

TOL = 2e-5   # fp32-vs-fp32 with different summation orders; the stated parity bar is 1e-4


def _params(t):
    return {k[2:]: v for k, v in t.items() if k.startswith("p.")}


def test_oracle_matches_golden(golden):
    name, cfg, train, t = golden
    out = bm_oracle.training_step(_params(t), cfg, t["meg"], t["rec_positions"], t["rec_of_sample"],
                                  t["subject_index"], t["candidates"], ban_centre=t["ban_centre"], training=train)
    assert rel_err(out["estimate"], t["estimate"]) < TOL
    assert rel_err(out["scores"], t["scores"]) < TOL
    assert abs(out["loss"].item() - t["loss"].item()) < TOL * max(1.0, abs(t["loss"].item()))
    probs = torch.softmax(out["scores"], dim=1)
    assert rel_err(probs, t["probs"]) < TOL
    # identical top-k ranking (north-star: "top-k retrieval ranks identical")
    k = min(5, probs.shape[1])
    assert torch.equal(probs.topk(k, dim=1).indices, t["probs"].topk(k, dim=1).indices)
    wscale = max(t[k2].norm().item() for k2 in t if k2.startswith("g.") and k2.endswith("weight"))
    for key, g in out["grads"].items():
        ref = t["g." + key]
        if g is None:
            assert ref.numel() == 0 or ref.abs().max() == 0
            continue
        if ".0.bias" in key and "sequence" in key:
            # conv bias followed by train-mode BN: true gradient is 0, both sides hold rounding noise
            if train:
                assert g.abs().max().item() < 1e-5 * wscale + 1e-7
                continue
        assert rel_err(g, ref) < 50 * TOL, key
    if train:
        for key, v in out["bn_updates"].items():
            assert rel_err(v, t["bn." + key]) < TOL, key


def test_oracle_fp64_agrees_with_fp32(golden):
    name, cfg, train, t = golden
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in _params(t).items()}
    est64 = bm_oracle.simpleconv_forward(p64, cfg, t["meg"].double(), t["rec_positions"].double(),
                                         t["rec_of_sample"], t["subject_index"], train,
                                         t["ban_centre"].double())
    assert rel_err(est64.float(), t["estimate"]) < 2e-5


def test_oracle_matches_live_reference():
    """The reference's train-mode forward and loss at merger_pos_dim 128 (oracle/make_golden.py run_train_forward),
    from its seeded initial state."""
    cfg, train, t = load_golden("train_forward")
    assert train and cfg.dilations() == [1, 2, 4, 8, 16, 1, 2, 4, 8, 16]
    p = make_golden.seeded_state(cfg, 1234, t["state_sha256"])
    subj = t["subject_index"]
    est_o = bm_oracle.simpleconv_forward(p, cfg, t["meg"], t["rec_positions"], subj, subj, True, t["ban_centre"])
    assert rel_err(est_o, t["estimate"]) < TOL
    assert abs(bm_oracle.clip_loss(est_o, t["candidates"]).item() - t["loss"].item()) < 1e-5


def test_synthetic_batch_shapes():
    cfg = bm_oracle.Config(in_channels=12, out_channels=5, n_subjects=4, hidden=8, merger_channels=6,
                           initial_linear=6, merger_pos_dim=32)
    d = bm_oracle.synthetic_batch(cfg, batch=3, T=20, n_valid=(12, 7))
    assert d["meg"].shape == (3, 12, 20) and d["candidates"].shape == (3, 5, 20)
    assert (d["rec_positions"][1, 7:] == bm_oracle.INVALID).all()
    p = bm_oracle.init_state_dict(cfg)
    est = bm_oracle.simpleconv_forward(p, cfg, d["meg"], d["rec_positions"], d["rec_of_sample"],
                                       d["subject_index"], False)
    assert est.shape == (3, 5, 20) and torch.isfinite(est).all()
