"""Pin of the oracles against the VERBATIM reference modules.  Two things are checked: (1) the committed fixtures are
exactly what the committed generator produces from the reference today -- only where a brainmagick source tree is at hand
(`oracle/ref_loader.py`, BM_REFERENCE_ROOT); (2) on inputs that no other fixture holds, oracle == reference, against what
the reference computed on them (oracle/make_golden.py: fresh_train, fresh_eval, prep_fresh)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, load_arrays, load_golden, rel_err
from oracle import bm_oracle, make_golden, prep_oracle, ref_loader


@pytest.mark.skipif(not ref_loader.reference_available(), reason="needs the brainmagick source tree (BM_REFERENCE_ROOT)")
@pytest.mark.parametrize("kind,name", [("case", "train_depth4"), ("case", "eval_small"), ("prep", "prep_small"),
                                       ("retrieval", "retrieval_small"), ("deepmel", "deepmel_nobn"),
                                       ("ablation", "ablation_subject_embedding")])
def test_fixtures_are_reproducible_from_the_reference(kind, name, tmp_path, monkeypatch):
    from oracle import make_golden
    monkeypatch.setattr(make_golden, "OUT", str(tmp_path))
    torch.set_num_threads(1)
    if kind == "case":
        make_golden.run_case(name, make_golden.CASES[name])
    elif kind == "prep":
        make_golden.run_prep(name)
    elif kind == "retrieval":
        make_golden.run_retrieval(name)
    elif kind == "deepmel":
        make_golden.run_deepmel(name, make_golden.DEEPMEL_CASES[name])
    else:
        make_golden.run_ablation(name, make_golden.ABLATIONS[name])
    fresh = np.load(os.path.join(str(tmp_path), name + ".npz"))
    committed = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    assert sorted(fresh.files) == sorted(committed.files)
    for k in committed.files:
        a, b = fresh[k], committed[k]
        assert a.shape == b.shape, k
        if a.dtype.kind == "f":
            assert np.allclose(a, b, rtol=1e-5, atol=1e-7, equal_nan=True), k
        else:
            assert np.array_equal(a, b), k


@pytest.mark.parametrize("seed,train", [(501, True), (502, False)])
def test_oracle_equals_live_reference_on_fresh_inputs(seed, train):
    name = "fresh_train" if train else "fresh_eval"
    assert make_golden.FRESH_CASES[name] == dict(seed=seed, train=train)
    cfg, train_, t = load_golden(name)
    assert train_ == train
    state = make_golden.seeded_state(cfg, seed, t["state_sha256"])
    subj = t["subject_index"]
    ref = bm_oracle.training_step(state, cfg, t["meg"], t["rec_positions"], subj, subj, t["candidates"],
                                  ban_centre=t["ban_centre"], training=train)
    assert rel_err(ref["estimate"], t["estimate"]) < 2e-6
    assert abs(float(ref["loss"]) - float(t["loss"])) < 1e-6
    grads = [k[2:] for k in t if k.startswith("g.")]
    assert grads and set(grads) <= set(ref["grads"])
    for key in grads:                      # the reference's gradient at the fixture's `grad_sample` entries
        g = ref["grads"][key].reshape(-1)[torch.from_numpy(make_golden.grad_sample(key, ref["grads"][key].numel()))]
        if t["gnorm." + key] < 1e-6:
            assert ref["grads"][key].abs().max() < 1e-5, key
        else:
            assert rel_err(g, t["g." + key]) < 3e-5, key


def test_prep_oracle_equals_live_reference_on_fresh_inputs():
    t = load_arrays("prep_fresh")
    ids, off = [int(r) for r in t["rec_ids"]], int(t["offset"])
    center = {r: t["meg_center"][i] for i, r in enumerate(ids)}
    scale = {r: t["meg_scale"][i] for i, r in enumerate(ids)}
    for clip in (False, True):
        got = prep_oracle.prepare(t["meg"], t["recording_index"], center, scale, t["features"], t["features_mask"],
                                  t["feat_center"], t["feat_scale"], limit=float(t["limit"]), clip=clip, offset_samples=off)
        assert np.array_equal(got["keep"], t[f"clip{int(clip)}.keep"])
        assert np.array_equal(got["meg"], t[f"clip{int(clip)}.meg"])
        assert np.array_equal(got["features"], t[f"clip{int(clip)}.features"])
