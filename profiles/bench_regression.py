"""Measures the regression objective (L1Loss / L2Loss, bm/losses.py:11-26) on one B200.  GPU only: fails without one.

    python profiles/bench_regression.py OUT_DIR [--rounds 5 --steps 10 --warmup 3]     # writes OUT_DIR/regression_bench.json

(a) The regression training step at cfg4 (128 sensors, F = 120 mel bands, 19 subjects, T = 360, B = 256): SimpleConv
    forward, masked MSE, backward, Adam, against the solver's time-cropped targets `features[..., :-offset]` and a partial
    [B,1,T] features mask.  Two loss arms in the same process, alternating round by round after a warm-up of each:
      package    brainmagick_b200.L2Loss (csrc/regression.cuh: no host synchronisation)
      reference  bm/losses.py's expression: est[mask.expand_as(est)] and F.mse_loss (the boolean index runs `nonzero`, a
                 device->host synchronisation; the host cannot enqueue the backward until the forward has finished)
    Device time per step (CUDA events around `steps` steps) and host time per step (wall clock of the first two steps after a
    synchronise, i.e. the enqueue time while the launch queue is far from full).  The difference between the arms is the
    cost of the synchronisation.
(b) The two loss kernels alone at F = 120 and F = 1024 (B = 256, T = 360): `launches` calls captured in one CUDA graph, so the
    time is the kernels' and not the Python call's, over operand sets rotated beyond the 126 MB L2; GB/s from the
    algorithmic bytes (forward: 8 B per element + the mask, backward: 12 B per element + the mask), set against the copy
    bandwidth bench.py reports (MEASURED_PEAKS.json, else its fallback) and a device-to-device copy timed in this run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn.functional as TF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench                                                          # noqa: E402
import brainmagick_b200 as bb                                         # noqa: E402
from brainmagick_b200 import _lib, functional as BF, synthetic        # noqa: E402

DEV = "cuda"


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return dict(name=name, power_limit=power, clocks_max_sm=clock, torch_name=torch.cuda.get_device_name(0))


def step_arms(rounds: int, steps: int, warmup: int, batch: int = 256) -> dict:
    cfg = bench.CONFIGS["cfg4"]
    C, T, F, S = cfg["C"], cfg["T"], cfg["F"], cfg["S"]
    offset = 18                                   # clip_conv.yaml offset_meg_ms: 150 at 120 Hz
    torch.manual_seed(2036)
    model = bb.SimpleConv(in_channels=dict(meg=C), out_channels=F, n_subjects=S,
                          **{k: (dict(v) if isinstance(v, dict) else v) for k, v in bench.CLIP_CONV.items()}).to(DEV).train()
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, betas=(0.9, 0.999), fused=True)
    positions = synthetic.normalised_positions(S, C, seed=7)
    recs = [synthetic.SyntheticRecording(s, positions[s]) for s in range(S)]
    g = torch.Generator(device=DEV).manual_seed(5)
    meg = torch.randn(batch, C, T, generator=g, device=DEV)
    features = torch.randn(batch, F, T + offset, generator=g, device=DEV).abs()
    targets = features[..., :-offset]             # the solver's crop: a non-contiguous view
    mask = torch.rand(batch, 1, T, generator=g, device=DEV) < 0.9
    subj_h = torch.randint(0, S, (batch,)).tolist()
    subj = torch.tensor(subj_h, device=DEV)
    l2 = bb.L2Loss()

    def package(est):
        return l2(est, targets, mask)

    def reference(est):
        fm = mask.expand_as(est)
        return TF.mse_loss(est[fm], targets[fm])

    def step(loss_fn):
        opt.zero_grad(set_to_none=True)
        est = model(dict(meg=meg), synthetic.SyntheticBatch(meg, subj, [recs[s] for s in subj_h]))
        loss = loss_fn(est)
        loss.backward()
        opt.step()
        return loss

    arms = dict(package=package, reference=reference)
    for fn in arms.values():
        for _ in range(warmup):
            step(fn)
    torch.cuda.synchronize()
    res = {k: dict(ms_per_step=[], host_ms_per_step=[]) for k in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t0 = time.perf_counter()
            for i in range(steps):
                step(fn)
                if i == 1:
                    res[name]["host_ms_per_step"].append((time.perf_counter() - t0) * 1e3 / 2)
            e1.record()
            torch.cuda.synchronize()
            res[name]["ms_per_step"].append(e0.elapsed_time(e1) / steps)
    BF.check_tc_status()
    for r in res.values():
        r["median_ms_per_step"] = statistics.median(r["ms_per_step"])
        r["median_host_ms_per_step"] = statistics.median(r["host_ms_per_step"])
        r["segments_per_s"] = batch / r["median_ms_per_step"] * 1e3
    with torch.no_grad():                         # the two arms compute the same loss
        est = model(dict(meg=meg), synthetic.SyntheticBatch(meg, subj, [recs[s] for s in subj_h]))
        same = dict(package=float(package(est)), reference=float(reference(est)))
    return dict(workload=f"cfg4 regression step: SimpleConv C={C} F={F} S={S} T={T} B={batch} + masked MSE + backward + "
                         f"Adam; targets features[..., :-{offset}], [B,1,T] mask {float(mask.float().mean()):.3f} true",
                rounds=rounds, steps_per_round=steps, warmup_steps_per_arm=warmup, arms=res, loss_check=same,
                sync_cost_ms_per_step=res["reference"]["median_ms_per_step"] - res["package"]["median_ms_per_step"])


def copy_gbs(nbytes: int = 1 << 30, iters: int = 20) -> float:
    a = torch.empty(nbytes // 4, device=DEV)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * iters / (e0.elapsed_time(e1) * 1e-3) / 1e9


def kernels_alone(F: int, launches: int = 200, B: int = 256, T: int = 360, l2_bytes: int = 126 << 20) -> dict:
    n = B * F * T
    per_set = 8 * n + B * T
    n_sets = max(2, -(-3 * l2_bytes // per_set))            # >= 3x the L2 between two uses of one set
    g = torch.Generator(device=DEV).manual_seed(F)
    sets = []
    for _ in range(n_sets):
        est = torch.randn(B, F, T, generator=g, device=DEV)
        out = torch.randn(B, F, T, generator=g, device=DEV)
        mask = (torch.rand(B, 1, T, generator=g, device=DEV) < 0.9).view(torch.uint8)
        ws = torch.empty(BF.REGRESSION_WS_DOUBLES, device=DEV, dtype=torch.float64)
        loss = torch.empty(1, device=DEV)
        dest = torch.empty_like(est)
        sets.append((est, out, mask, ws, loss, dest))
    gout = torch.ones(1, device=DEV)
    P = _lib.ptr

    def fwd(s, p):
        est, out, mask, ws, loss, _ = s
        _lib.call("bm_regression_loss_fwd", P(est), P(out), P(mask), B, F, 1, T, p, P(ws), P(loss), _lib.stream())

    def bwd(s, p):
        est, out, mask, ws, _, dest = s
        _lib.call("bm_regression_loss_bwd", P(est), P(out), P(mask), P(gout), P(ws), B, F, 1, T, p, P(dest), None,
                  _lib.stream())

    res = dict(shape=[B, F, T], operand_sets=n_sets, bytes_per_set=per_set, launches=launches)
    for p in (2, 1):
        for s in sets:
            fwd(s, p)
            bwd(s, p)
        torch.cuda.synchronize()
        for name, fn, alg in (("fwd", fwd, 8 * n + B * T), ("bwd", bwd, 12 * n + B * T)):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for i in range(launches):
                    fn(sets[i % n_sets], p)
            graph.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / launches
            res[f"p{p}.{name}"] = dict(us_per_launch=us, algorithmic_bytes=alg, gb_per_s=alg / (us * 1e-6) / 1e9)
            del graph
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_regression.py measures on a CUDA device; none is available")
    torch.cuda.set_device(0)
    _lib.load()
    peaks = bench.load_peaks()
    res = dict(card=card(), step=step_arms(args.rounds, args.steps, args.warmup))
    torch.cuda.empty_cache()
    copy = copy_gbs()
    res["copy_bandwidth"] = dict(bench_py_gbs=peaks["hbm_gbs"], bench_py_source=peaks["source"], measured_here_gbs=copy,
                                 measured_here="1 GiB device-to-device copy_, read + write bytes")
    res["kernels"] = {}
    for F in (120, 1024):
        k = kernels_alone(F)
        for key, v in k.items():
            if isinstance(v, dict):
                v["frac_of_bench_py_copy"] = v["gb_per_s"] / peaks["hbm_gbs"]
                v["frac_of_copy_measured_here"] = v["gb_per_s"] / copy
        res["kernels"][f"F{F}"] = k
        torch.cuda.empty_cache()
    res["card_after"] = card()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "regression_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
