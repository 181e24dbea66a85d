"""CPU: the regression objectives (L1Loss / L2Loss, bm/losses.py:11-26; the solver's 'l1' and 'mse').

  * the oracle (oracle/regression_oracle.py) against what the verbatim reference computed (tests/golden/regression_*.npz,
    made by oracle/make_regression_golden.py);
  * the drop-in modules' host path on `abi_emulator.emulated()`, with the two new entry points emulated here from their
    documented contract (include/bm_b200.h), against the same fixtures -- alone and after a SimpleConv step;
  * the module surface and its errors.
The kernels themselves are checked on the GPU (tests/test_gpu_regression.py)."""
import os
import re

import numpy as np
import pytest
import torch

import abi_emulator
from abi_emulator import _v
from conftest import GOLDEN_DIR, ROOT, load_arrays, load_golden, rel_err
from oracle import make_golden, make_regression_golden, ref_loader, regression_oracle

CASES = list(make_regression_golden.LOSS_CASES)


def _emu_fwd(self, est, out, mask, B, F, Fm, T, p, ws, loss, stream):
    """bm_regression_loss_fwd: fp32 difference, fp64 sum and count over the selection; the count kept in the workspace."""
    e, o = _v(est, B, F, T), _v(out, B, F, T)
    sel = _v(mask, B, Fm, T).bool().expand(B, F, T)
    d = torch.where(sel, e - o, torch.zeros(())).double()
    n = sel.sum().double()
    _v(ws, 1)[0] = n
    _v(loss, 1)[0] = ((d.abs() if p == 1 else d * d).sum() / n).float()


def _emu_bwd(self, est, out, mask, gout, ws, B, F, Fm, T, p, dest, dout, stream):
    """bm_regression_loss_bwd: selected ? p |d|^(p-1) sign(d) gout / count : 0, and its negation for the targets."""
    e, o = _v(est, B, F, T), _v(out, B, F, T)
    sel = _v(mask, B, Fm, T).bool().expand(B, F, T)
    scale = ((2.0 if p == 2 else 1.0) * _v(gout, 1)[0].double() / _v(ws, 1)[0]).float()
    d = e - o
    g = torch.where(sel, (d if p == 2 else torch.sign(d)) * scale, torch.zeros(()))
    if dest is not None:
        _v(dest, B, F, T).copy_(g)
    if dout is not None:
        _v(dout, B, F, T).copy_(torch.where(sel, -g, torch.zeros(())))


@pytest.fixture
def emulated(monkeypatch):
    monkeypatch.setattr(abi_emulator.Emulator, "bm_regression_loss_fwd", _emu_fwd, raising=False)
    monkeypatch.setattr(abi_emulator.Emulator, "bm_regression_loss_bwd", _emu_bwd, raising=False)
    with abi_emulator.emulated() as emu:
        yield emu


def _case(t, case):
    return (torch.from_numpy(t[case + ".estimate"]), torch.from_numpy(t[case + ".output"]),
            torch.from_numpy(t[case + ".mask"]))


def _check_against_fixture(loss, ge, go, t, case, p, tol=1e-6):
    want = float(t[f"{case}.l{p}.loss"])
    assert abs(float(loss) - want) <= tol * max(1.0, abs(want)), (case, p, float(loss), want)
    for got, key in ((ge, "grad_estimate"), (go, "grad_output")):
        ref = torch.from_numpy(t[f"{case}.l{p}.{key}"])
        assert torch.isfinite(got).all() and torch.isfinite(ref).all(), (case, p, key)
        assert torch.equal(got == 0, ref == 0), (case, p, key)            # unselected and (L1) tied elements are exactly 0
        assert torch.allclose(got, ref, rtol=tol, atol=tol * ref.abs().max().item()), (case, p, key)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("p", [1, 2])
@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_reference_fixtures(case, p, dtype):
    t = load_arrays("regression_losses")
    est, out, mask = _case(t, case)
    e, o = est.to(dtype).requires_grad_(True), out.to(dtype).requires_grad_(True)
    loss = regression_oracle.masked_loss(e, o, mask, p)
    loss.backward()
    _check_against_fixture(loss.detach(), e.grad.float(), o.grad.float(), t, case, p)


def test_fixture_cases_cover_the_masks_they_name():
    t = load_arrays("regression_losses")
    sel = {c: np.broadcast_to(t[c + ".mask"], t[c + ".estimate"].shape) for c in CASES}
    assert sel["all_true"].all() and t["all_true.mask"].shape[1] == 1
    assert 0 < sel["half"].mean() < 1 and t["half.mask"].shape[1] == 1
    assert t["full_mask.mask"].shape == t["full_mask.estimate"].shape and 0 < sel["full_mask"].mean() < 1
    assert sel["single"].sum() == 1
    bad = ~np.isfinite(t["nonfinite.estimate"]) | ~np.isfinite(t["nonfinite.output"])
    assert bad.any() and not (bad & sel["nonfinite"]).any()
    ties = (t["ties.estimate"] == t["ties.output"]) & sel["ties"]
    assert ties.any() and (t["ties.l1.grad_estimate"][ties] == 0).all()


@pytest.mark.parametrize("p", [1, 2])
@pytest.mark.parametrize("case", CASES)
def test_drop_in_losses_on_the_emulator(case, p, emulated):
    import brainmagick_b200 as bb
    t = load_arrays("regression_losses")
    est, out, mask = _case(t, case)
    e, o = est.clone().requires_grad_(True), out.clone().requires_grad_(True)
    loss = (bb.L1Loss() if p == 1 else bb.L2Loss())(e, o, mask)
    assert loss.shape == () and loss.dtype == torch.float32
    loss.backward()
    _check_against_fixture(loss.detach(), e.grad, o.grad, t, case, p)


def test_cropped_target_view_and_broadcast_masks_on_the_emulator(emulated):
    """The solver's targets are `features[..., :-offset]` (a non-contiguous view); masks that broadcast over B or T reach
    the same selection as their expanded form."""
    import brainmagick_b200 as bb
    g = torch.Generator().manual_seed(3)
    est = torch.randn(3, 4, 10, generator=g)
    feats = torch.randn(3, 4, 13, generator=g)
    out = feats[..., :-3]
    for mask in (torch.rand(3, 1, 10, generator=g) < 0.5, torch.rand(1, 1, 10, generator=g) < 0.5,
                 torch.rand(3, 1, 1, generator=g) < 0.5, torch.rand(1, 4, 10, generator=g) < 0.5):
        for p, cls in ((1, bb.L1Loss), (2, bb.L2Loss)):
            e = est.clone().requires_grad_(True)
            loss = cls()(e, out, mask)
            loss.backward()
            e64 = est.double().requires_grad_(True)
            ref = regression_oracle.masked_loss(e64, out.double(), mask, p)
            ref.backward()
            assert abs(loss.item() - ref.item()) < 1e-6 * max(1.0, abs(ref.item()))
            assert rel_err(e.grad, e64.grad) < 1e-6


def test_empty_mask_gives_nan_loss_and_zero_gradients_on_the_emulator(emulated):
    import brainmagick_b200 as bb
    est, out = torch.randn(2, 3, 5).requires_grad_(True), torch.randn(2, 3, 5).requires_grad_(True)
    loss = bb.L2Loss()(est, out, torch.zeros(2, 1, 5, dtype=torch.bool))
    loss.backward()
    assert torch.isnan(loss)
    assert (est.grad == 0).all() and (out.grad == 0).all()


def _step_model(cfg, t):
    import brainmagick_b200 as bb
    state = make_golden.seeded_state(cfg, make_regression_golden.TRAIN["seed"], t["state_sha256"])
    model = bb.SimpleConv(in_channels=dict(meg=cfg.in_channels), out_channels=cfg.out_channels, n_subjects=cfg.n_subjects,
                          **ref_loader.clip_conv_kwargs(hidden=cfg.hidden, depth=cfg.depth, merger_channels=cfg.merger_channels,
                                                        initial_linear=cfg.initial_linear, merger_pos_dim=cfg.merger_pos_dim))
    model.load_state_dict(state)
    return state, model


def _check_step(est, loss, grads, t, tol):
    assert rel_err(est, t["estimate"]) < tol
    assert abs(float(loss) - float(t["loss"])) < tol * max(1.0, abs(float(t["loss"])))
    keys = [k[2:] for k in t if k.startswith("g.")]
    assert keys and set(keys) <= set(grads)
    for key in keys:
        g = grads[key].reshape(-1)[torch.from_numpy(make_golden.grad_sample(key, grads[key].numel()))]
        if t["gnorm." + key] < 1e-6:
            assert grads[key].abs().max() < 1e-5, key
        else:
            assert rel_err(g, t["g." + key]) < tol, (key, rel_err(g, t["g." + key]))


def test_regression_step_oracle_matches_reference_fixture():
    cfg, train, t = load_golden("regression_train")
    assert train and cfg.out_channels == make_regression_golden.TRAIN["F"]
    state, _ = _step_model(cfg, t)
    subj = t["subject_index"]
    ref = regression_oracle.regression_step(state, cfg, t["meg"], t["rec_positions"], subj, subj, t["candidates"],
                                            t["features_mask"], 2, ban_centre=t["ban_centre"])
    _check_step(ref["estimate"], ref["loss"], ref["grads"], t, 3e-5)


def test_simpleconv_with_l2loss_step_on_the_emulator(emulated):
    import brainmagick_b200 as bb
    from brainmagick_b200 import synthetic
    cfg, _, t = load_golden("regression_train")
    _, model = _step_model(cfg, t)
    model.train()
    model.merger.ban_centre_override = t["ban_centre"]
    batch = synthetic.make_batch(t["meg"], t["subject_index"], t["rec_positions"], t["rec_of_sample"])
    est = model(dict(meg=t["meg"]), batch)
    loss = bb.L2Loss().train()(est, t["candidates"], t["features_mask"])
    loss.backward()
    _check_step(est.detach(), loss.detach(), {k: p.grad for k, p in model.named_parameters()}, t, 3e-5)


def test_surface_matches_the_reference():
    import brainmagick_b200 as bb
    assert "L1Loss" in bb.__all__ and "L2Loss" in bb.__all__
    for cls, inner in ((bb.L1Loss, torch.nn.L1Loss), (bb.L2Loss, torch.nn.MSELoss)):
        m = cls()
        assert isinstance(m._loss, inner)
        assert repr(m) == f"{cls.__name__}(\n  (_loss): {inner.__name__}()\n)"
        assert len(m.state_dict()) == 0
        assert len(list(m.parameters())) == 0
        assert m.train() is m and m.training and not m.eval().training
        assert m.to(torch.device("cpu")) is m


def test_errors_match_the_package_conventions(emulated):
    import brainmagick_b200 as bb
    est, out, mask = torch.randn(2, 3, 5), torch.randn(2, 3, 5), torch.ones(2, 1, 5, dtype=torch.bool)
    with pytest.raises(TypeError):                          # the mask selects: the reference's index rejects a float one
        bb.L2Loss()(est, out, mask.float())
    with pytest.raises(TypeError):                          # bm/losses.py:13 calls mask.expand_as
        bb.L1Loss()(est, out, None)
    with pytest.raises(ValueError):
        bb.L2Loss()(est, out[:, :2], mask)
    with pytest.raises(RuntimeError):                        # mask.expand_as(estimate) fails
        bb.L2Loss()(est, out, torch.ones(2, 1, 4, dtype=torch.bool))


def test_cpu_and_non_fp32_tensors_raise():
    import brainmagick_b200 as bb
    est, out, mask = torch.randn(2, 3, 5), torch.randn(2, 3, 5), torch.ones(2, 1, 5, dtype=torch.bool)
    with pytest.raises(RuntimeError):                        # no CPU fallback
        bb.L2Loss()(est, out, mask)
    with pytest.raises(RuntimeError):
        bb.L1Loss()(est, out, mask)
    with pytest.raises(TypeError):
        bb.L2Loss()(est.double(), out.double(), mask)
    with pytest.raises(TypeError):
        bb.L1Loss()(est.half(), out.half(), mask)


def test_workspace_size_matches_the_header():
    from brainmagick_b200 import functional as BF
    header = open(os.path.join(ROOT, "include", "bm_b200.h")).read()
    assert int(re.search(r"#define BM_REGRESSION_WS_DOUBLES (\d+)", header).group(1)) == BF.REGRESSION_WS_DOUBLES


@pytest.mark.skipif(not ref_loader.reference_available(), reason="needs the brainmagick source tree (BM_REFERENCE_ROOT)")
@pytest.mark.parametrize("name", ["regression_losses", "regression_train"])
def test_regression_fixtures_are_reproducible_from_the_reference(name, tmp_path, monkeypatch):
    monkeypatch.setattr(make_regression_golden, "OUT", str(tmp_path))
    torch.set_num_threads(1)
    (make_regression_golden.run_losses if name == "regression_losses" else make_regression_golden.run_train)(name)
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
