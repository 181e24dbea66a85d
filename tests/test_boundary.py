"""CPU: the drop-in boundary -- constructor surface, state_dict layout, error behaviour, C-ABI symbols -- without
any compute call (no GPU here)."""
import ctypes
import json
import os
import re

import pytest
import torch

from conftest import GOLDEN_CASES, GOLDEN_DIR, ROOT, load_golden

CLIP_CONV = dict(hidden=dict(meg=320), batch_norm=True, depth=10, dilation_period=5, kernel_size=3, skip=True,
                 subject_layers=True, subject_dim=0, complex_out=True, glu=2, glu_context=1, merger=True,
                 initial_linear=270, gelu=True, merger_pos_dim=2048)


def _kw(**over):
    kw = {k: (dict(v) if isinstance(v, dict) else v) for k, v in CLIP_CONV.items()}
    kw.update(over)
    return kw


def test_c_abi_exports_every_declared_symbol():
    """dlopen libbm_b200.so and resolve every function include/bm_b200.h declares."""
    import __graft_entry__
    __graft_entry__.build()
    from brainmagick_b200 import _lib
    header = open(os.path.join(ROOT, "include", "bm_b200.h")).read()
    declared = set(re.findall(r"\b(bm_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 30
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/bm_b200.h but not exported"
    bound = set(_lib.SIGNATURES) | {"bm_last_error", "bm_abi_version", "bm_launch_count", "bm_tc_wgrad_workspace",
             "bm_clip_workspace", "bm_tc_wgrad_conv_workspace"}
    assert declared == bound, (declared ^ bound)
    _lib.load()
    assert _lib.load().bm_abi_version() == 1
    assert _lib.load().bm_tc_conv_supported(360, 320, 320, 3, 0) == 1
    assert _lib.load().bm_tc_conv_supported(360, 270, 320, 3, 0) == 0      # K must be a multiple of 32
    assert _lib.load().bm_tc_wgrad_supported(320, 320) == 1


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_state_dict_layout_matches_reference(name):
    """keys, shapes and ORDER of state_dict() equal the reference's (fixtures carry the reference state_dict)."""
    import brainmagick_b200 as bb
    cfg, train, t = load_golden(name)
    ref = {k[2:]: v for k, v in t.items() if k.startswith("p.")}
    model = bb.SimpleConv(in_channels=dict(meg=cfg.in_channels), out_channels=cfg.out_channels,
                          n_subjects=cfg.n_subjects,
                          **_kw(hidden=dict(meg=cfg.hidden), depth=cfg.depth, merger_channels=cfg.merger_channels,
                                initial_linear=cfg.initial_linear, merger_pos_dim=cfg.merger_pos_dim))
    sd = model.state_dict()
    assert list(sd.keys()) == list(ref.keys())
    for k in sd:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k
    model.load_state_dict(ref, strict=True)
    assert [n for n, _ in model.named_parameters()] == [k for k in ref if "running" not in k and "num_batches" not in k]


def test_seeded_constructor_is_rng_identical_to_reference():
    """same torch.manual_seed => bit-identical initial parameters (bm/train.py:76,109 model_hash), against the digests of
    the reference's state_dict (oracle/make_golden.py run_seeded_init)."""
    import brainmagick_b200 as bb
    from oracle import make_golden
    with open(os.path.join(GOLDEN_DIR, "seeded_init.json")) as f:
        ref = json.load(f)
    c = ref["spec"]
    assert c == make_golden.SEEDED_INIT
    kw = _kw(hidden=dict(meg=c["hidden"]), merger_channels=c["MC"], initial_linear=c["IL"], merger_pos_dim=c["P"])
    torch.manual_seed(c["seed"])
    mine = bb.SimpleConv(in_channels=dict(meg=c["C"]), out_channels=c["F"], n_subjects=c["S"], **kw)
    ms = mine.state_dict()
    assert list(ms) == [e["key"] for e in ref["state"]]
    for e in ref["state"]:
        v = ms[e["key"]]
        assert [list(v.shape), str(v.dtype), make_golden.tensor_sha256(v)] == [e["shape"], e["dtype"], e["sha256"]], e["key"]
    assert repr(mine.subject_layers) == ref["subject_layers_repr"]


def test_constructor_errors_and_unsupported_options():
    import brainmagick_b200 as bb
    with pytest.raises(ValueError):                       # simpleconv.py:79-81
        bb.SimpleConv(in_channels=dict(meg=8), out_channels=4, hidden=dict(other=8))
    with pytest.raises(AssertionError):                   # simpleconv.py:92
        bb.SimpleConv(in_channels=dict(meg=8), out_channels=4, n_subjects=2, **_kw(kernel_size=4))
    for bad in (dict(batch_norm=False), dict(dual_path=2), dict(initial_depth=2),
                dict(n_fft=64), dict(dropout=0.1), dict(merger_per_subject=True)):
        with pytest.raises(NotImplementedError):
            bb.SimpleConv(in_channels=dict(meg=8), out_channels=4, n_subjects=2, **_kw(**bad))
    model = bb.SimpleConv(in_channels=dict(meg=8), out_channels=4, n_subjects=2,
                          **_kw(hidden=dict(meg=16), merger_channels=8, initial_linear=8, merger_pos_dim=32))
    assert float(model.merger.training_penalty) == 0.0    # bm/solver.py:376-378 hook
    with pytest.raises(RuntimeError):                      # no CPU fallback
        model(dict(meg=torch.zeros(1, 8, 10)), None)


def test_cliploss_surface():
    import types
    import brainmagick_b200 as bb
    clip = bb.ClipLoss()
    assert clip.linear is None and len(list(clip.parameters())) == 0
    est, cand = torch.zeros(3, 4, 20), torch.zeros(2, 4, 20)
    with pytest.raises(AssertionError):                   # losses.py:110
        clip(est, est, torch.zeros(3, 1, 20, dtype=torch.bool))
    with pytest.raises(AssertionError):                   # losses.py:111
        clip(est, cand, torch.ones(3, 1, 20, dtype=torch.bool))
    # trim_samples (losses.py:50-75): tmin/tmax in seconds relative to dset.tmin
    dset = types.SimpleNamespace(tmin=-0.5, sample_rate=120)
    clip = bb.ClipLoss(tmin=0.0, tmax=1.0, dset_args=dset)
    e, c = clip.trim_samples(torch.zeros(2, 3, 360), torch.zeros(5, 3, 360))
    assert e.shape[-1] == 120 and c.shape[-1] == 120
    clip = bb.ClipLoss(tmin=0.0, tmax=1.0, tmin_train=0.5, dset_args=dset).train()
    e, _ = clip.trim_samples(torch.zeros(2, 3, 360), torch.zeros(5, 3, 360))
    assert e.shape[-1] == 240          # training window [tmin_train, tmax_train=None]
    e, _ = clip.eval().trim_samples(torch.zeros(2, 3, 360), torch.zeros(5, 3, 360))
    assert e.shape[-1] == 120


def test_position_getter_matches_oracle_normalisation():
    from brainmagick_b200 import common, synthetic
    pos = synthetic.normalised_positions(3, 9, (9, 5), seed=4)
    recs = [synthetic.SyntheticRecording(i, pos[i]) for i in range(3)]
    pg = common.PositionGetter()
    for i, r in enumerate(recs):
        assert torch.equal(pg.get_recording_layout(r), pos[i])
    batch = synthetic.SyntheticBatch(torch.zeros(4, 9, 5), torch.tensor([0, 1, 2, 1]), [recs[i] for i in (0, 1, 2, 1)])
    full = pg.get_positions(batch)
    assert full.shape == (4, 9, 2) and pg.is_invalid(full)[1, 5:].all() and not pg.is_invalid(full)[0].any()
    emb = common.FourierEmb(32)(full)
    from oracle import bm_oracle
    assert torch.allclose(emb, bm_oracle.fourier_emb(full, 32), atol=1e-6)
