"""GPU: the regression objectives (L1Loss / L2Loss, bm/losses.py:11-26) on the CUDA kernels of csrc/regression.cuh.

  * kernels against the fp64 restatement (oracle/regression_oracle.py) at odd sizes (T % 4 != 0: the scalar path), at cfg4
    (F = 120 mel bands) and at cfg2 widths (F = 1024), with every mask kind of the fixtures;
  * the drop-in modules against what the verbatim reference computed (tests/golden/regression_losses.npz);
  * determinism, no host synchronisation, and a whole SimpleConv regression step against the fp64 oracle."""
import pytest
import torch

from conftest import load_arrays, rel_err
from oracle import bm_oracle, make_regression_golden, regression_oracle

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1, 1), (3, 7, 5), (2, 20, 361), (256, 120, 360), (256, 1024, 360)]
MASKS = ["all", "half", "full", "single", "nonfinite", "ties"]


def _inputs(shape, kind, seed):
    """(estimate, output, mask) on the GPU for one of the fixtures' mask kinds, drawn on the device (cfg2 widths hold 94 M
    elements per tensor)."""
    B, F, T = shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev = "cuda"
    est = torch.randn(B, F, T, generator=g, device=dev)
    out = torch.randn(B, F, T, generator=g, device=dev)
    if kind == "all":
        mask = torch.ones(B, 1, T, dtype=torch.bool, device=dev)
    elif kind == "full":
        mask = torch.rand(B, F, T, generator=g, device=dev) < 0.5
    elif kind == "single":
        mask = torch.zeros(B, F, T, dtype=torch.bool, device=dev)
        mask[B // 2, F // 2, T // 2] = True
    else:
        mask = torch.rand(B, 1, T, generator=g, device=dev) < 0.5
    if kind != "single":
        mask[0, 0, 0] = True
    if kind == "nonfinite":
        off = ~mask.expand_as(est)
        pick = torch.randint(0, 3, (B, F, T), generator=g, device=dev)
        bad = torch.tensor([float("nan"), float("inf"), -float("inf")], device=dev)[pick]
        est = torch.where(off & (pick != 1), bad, est)
        out = torch.where(off & (pick != 2), bad, out)
    if kind == "ties":
        out = torch.where(torch.rand(B, F, T, generator=g, device=dev) < 0.3, est, out)
    return est, out, mask


def _run(est, out, mask, p, target_grad=True):
    import brainmagick_b200 as bb
    e = est.clone().requires_grad_(True)
    o = out.clone().requires_grad_(target_grad)
    loss = (bb.L1Loss() if p == 1 else bb.L2Loss())(e, o, mask)
    loss.backward()
    return loss.detach(), e.grad, (o.grad if target_grad else None)


def _truth(est, out, mask, p):
    e, o = est.double().requires_grad_(True), out.double().requires_grad_(True)
    loss = regression_oracle.masked_loss(e, o, mask, p)
    loss.backward()
    return loss.detach(), e.grad, o.grad


def _check_elementwise(got, ref, what):
    """<= 4e-7 relative per element (three fp32 roundings), exact 0 where the truth is 0 (unselected, or an L1 tie)."""
    ref32 = ref.float()
    assert torch.isfinite(got).all(), what
    assert torch.equal(got == 0, ref32 == 0), what
    err = ((got.double() - ref).abs() - 4e-7 * ref.abs()).max().item()
    assert err <= 0, (what, err)


@pytest.mark.parametrize("kind", MASKS)
@pytest.mark.parametrize("shape", SHAPES, ids=["x".join(map(str, s)) for s in SHAPES])
@pytest.mark.parametrize("p", [1, 2])
def test_kernels_match_fp64(p, shape, kind):
    est, out, mask = _inputs(shape, kind, seed=sum(shape) + 7 * p)
    loss, ge, go = _run(est, out, mask, p)
    ref, re, ro = _truth(est, out, mask, p)
    assert torch.isfinite(loss)
    assert abs(loss.double().item() - ref.item()) <= 1e-6 * abs(ref.item()), (loss.item(), ref.item())
    _check_elementwise(ge, re, "grad estimate")
    _check_elementwise(go, ro, "grad output")
    assert torch.equal(go, torch.where(ge == 0, ge, -ge))
    del est, out, mask, ge, go, re, ro
    torch.cuda.empty_cache()


@pytest.mark.parametrize("Fm", [1, "F"])
@pytest.mark.parametrize("p", [1, 2])
def test_empty_mask_gives_nan_and_zero_gradients(p, Fm):
    B, F, T = 4, 6, 36
    est, out = torch.randn(B, F, T, device="cuda"), torch.randn(B, F, T, device="cuda")
    mask = torch.zeros(B, 1 if Fm == 1 else F, T, dtype=torch.bool, device="cuda")
    loss, ge, go = _run(est, out, mask, p)
    assert torch.isnan(loss)
    assert (ge == 0).all() and (go == 0).all()


@pytest.mark.parametrize("p", [1, 2])
@pytest.mark.parametrize("case", list(make_regression_golden.LOSS_CASES))
def test_drop_in_matches_reference_fixtures(case, p):
    from test_regression_cpu import _case, _check_against_fixture
    t = load_arrays("regression_losses")
    est, out, mask = (x.cuda() for x in _case(t, case))
    loss, ge, go = _run(est, out, mask, p)
    _check_against_fixture(loss.cpu(), ge.cpu(), go.cpu(), t, case, p)


@pytest.mark.parametrize("shape", [(256, 120, 360), (3, 7, 5)])
@pytest.mark.parametrize("p", [1, 2])
def test_two_calls_are_bitwise_equal(p, shape):
    est, out, mask = _inputs(shape, "half", seed=99)
    a, b = _run(est, out, mask, p), _run(est, out, mask, p)
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))


def test_forward_and_backward_do_not_synchronise():
    import brainmagick_b200 as bb
    est, out, mask = _inputs((16, 120, 360), "half", seed=5)
    e = est.clone().requires_grad_(True)
    crit = bb.L2Loss()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss = crit(e, out, mask)
        loss.backward()
        with pytest.raises(RuntimeError):                 # the reference's boolean gather does synchronise
            e.detach()[mask.expand_as(e)]
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ref, re, _ = _truth(est, out, mask, 2)
    assert abs(loss.item() - ref.item()) <= 1e-6 * abs(ref.item())
    _check_elementwise(e.grad, re, "grad estimate")


def test_target_gradient_matches_fp64():
    """output.requires_grad (a trainable feature model produces the targets): dL/doutput = -dL/destimate."""
    est, out, mask = _inputs((8, 120, 360), "full", seed=17)
    for p in (1, 2):
        loss, ge, go = _run(est, out, mask, p)
        _, _, ro = _truth(est, out, mask, p)
        _check_elementwise(go, ro, f"grad output p={p}")
        loss2, ge2, go2 = _run(est, out, mask, p, target_grad=False)
        assert go2 is None and torch.equal(ge2, ge) and torch.equal(loss2, loss)


# ---- a whole regression step: SimpleConv + masked L1 / L2 against the fp64 oracle --------------------------------------------
TOL = 1e-4


def _step(F, loss_p, B=4, target_grad=False):
    from brainmagick_b200 import synthetic
    from test_gpu_parity import _build_model
    import brainmagick_b200 as bb
    cfg = bm_oracle.Config(in_channels=128, out_channels=F, n_subjects=19)             # cfg4 (broderick2019, mel targets)
    params = bm_oracle.init_state_dict(cfg, seed=31)
    d = bm_oracle.synthetic_batch(cfg, batch=B, T=360, seed=12)
    d["rec_positions"] = synthetic.normalised_positions(cfg.n_subjects, cfg.in_channels, (), seed=4)
    g = torch.Generator().manual_seed(13)
    # targets at least 0.05 away from the estimate: L1's gradient sign(e - o) is then the same for the kernels and the oracle
    with torch.no_grad():
        est32 = bm_oracle.simpleconv_forward(params, cfg, d["meg"], d["rec_positions"], d["rec_of_sample"],
                                             d["subject_index"], True, d["ban_centre"])
    gap = 0.05 + torch.rand(est32.shape, generator=g)
    targets = est32 + torch.where(torch.rand(est32.shape, generator=g) < 0.5, -gap, gap)
    mask = torch.rand(B, 1, 360, generator=g) < 0.7

    def oracle(dtype):
        cast = lambda t: t.to(dtype) if t.is_floating_point() else t          # noqa: E731
        return regression_oracle.regression_step({k: cast(v) for k, v in params.items()}, cfg, cast(d["meg"]),
                                                 cast(d["rec_positions"]), d["rec_of_sample"], d["subject_index"],
                                                 cast(targets), mask, loss_p, ban_centre=cast(d["ban_centre"]),
                                                 target_grad=target_grad)
    ref = oracle(torch.float64)
    model = _build_model(cfg, params).train()
    model.merger.ban_centre_override = d["ban_centre"]
    meg = d["meg"].cuda()
    batch = synthetic.make_batch(meg, d["subject_index"].cuda(), d["rec_positions"], d["rec_of_sample"])
    est = model(dict(meg=meg), batch)
    out = targets.cuda().requires_grad_(target_grad)
    loss = (bb.L1Loss() if loss_p == 1 else bb.L2Loss())(est, out, mask.cuda())
    loss.backward()
    torch.cuda.synchronize()
    from brainmagick_b200 import functional as BF
    BF.check_tc_status()
    assert rel_err(est.detach().cpu(), ref["estimate"]) < TOL
    assert abs(loss.item() - ref["loss"].item()) < TOL * max(1.0, abs(ref["loss"].item()))
    wscale = max(v.norm().item() for k, v in ref["grads"].items() if k.endswith("weight") and v.numel())
    for name, prm in model.named_parameters():
        gg = prm.grad.detach().cpu()
        if "sequence" in name and name.endswith(".0.bias"):
            assert gg.abs().max().item() < 1e-4 * wscale + 1e-6, name               # true gradient is 0 (BatchNorm follows)
            continue
        assert rel_err(gg, ref["grads"][name]) < TOL, (F, loss_p, name, rel_err(gg, ref["grads"][name]))
    sd = model.state_dict()
    for key, v in ref["bn_updates"].items():
        assert rel_err(sd[key].cpu(), v) < TOL, key
    if target_grad:
        assert rel_err(out.grad.cpu(), ref["target_grad"]) < TOL


@pytest.mark.parametrize("loss_p", [2, 1])
def test_regression_step_at_cfg4_matches_fp64_oracle(loss_p):
    """cfg4 (C = 128 sensors, F = 120 mel bands, 19 subjects, T = 360) with a partial [B,1,T] features mask: estimate, loss,
    BatchNorm running statistics and EVERY parameter gradient within 1e-4 of the fp64 oracle."""
    _step(120, loss_p)


@pytest.mark.parametrize("F", [20, 40, 80])
def test_regression_step_at_nmels_widths_matches_fp64_oracle(F):
    """bm/grids/nmi/nmels.py: the same step at the other mel widths."""
    _step(F, 2)


def test_regression_step_target_gradient():
    _step(120, 2, B=2, target_grad=True)
