#!/usr/bin/env python
"""Benchmark of the contrastive training step (BASELINE.json metric: 3 s-segments/sec).

    python bench.py --gpus N --steps K --warmup W [--config cfg2|cfg3|cfg4|cfg5]   # B200 arm (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K --warmup W                 # reference arm: the reference's OWN
                                                                                   # modules on the host cores

One "step" = SimpleConv forward + ClipLoss forward + backward of both + Adam(lr 3e-4) update on one synthetic batch
(bm/solver.py:297,373,384-387; bm/train.py:119); for N > 1 the candidates are all-gathered before the contrastive matmul
and the gradients all-reduced (SURVEY.md 8(e)).  Default workload = BASELINE.json configs[1] (cfg2): synthetic
gwilliams2022-like MEG (208 sensors, 3 s @ 120 Hz = 360 samples, 1024-d wav2vec-like features, 27 subjects), B = 256 per
GPU, weak scaling.  The other BASELINE configurations are behind --config: cfg3 (273 sensors, 96 subjects, GLOBAL batch
512, strong scaling), cfg4 (128 sensors, 120 mel features, 19 subjects, 256 per GPU), cfg5 (4 mixed studies padded to 273
sensors, 175 subjects, GLOBAL batch 1024, strong scaling).  Prints ONE JSON line on rank 0.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    "cfg2": dict(name="cfg2 synthetic gwilliams2022 (208 sensors, 3s@120Hz, F=1024, S=27)", C=208, T=360, F=1024, S=27,
                 n_valid=(), batch_per_gpu=256, global_batch=None),
    "cfg3": dict(name="cfg3 synthetic audio_mous (273 sensors, 3s@120Hz, F=1024, S=96), global batch 512", C=273, T=360,
                 F=1024, S=96, n_valid=(), batch_per_gpu=None, global_batch=512),
    "cfg4": dict(name="cfg4 synthetic broderick2019 EEG (128 sensors, 3s@120Hz, 120 mel features, S=19)", C=128, T=360, F=120,
                 S=19, n_valid=(), batch_per_gpu=256, global_batch=None),
    "cfg5": dict(name="cfg5 mixed 4-study synthetic (273/208/128/60 valid sensors padded to 273, F=1024, S=175), global batch 1024",
                 C=273, T=360, F=1024, S=175, n_valid=(273, 208, 128, 60), batch_per_gpu=None, global_batch=1024),
}
CLIP_CONV = dict(hidden=dict(meg=320), batch_norm=True, depth=10, dilation_period=5, kernel_size=3, skip=True,
                 subject_layers=True, subject_dim=0, complex_out=True, glu=2, glu_context=1, merger=True,
                 initial_linear=270, gelu=True, merger_pos_dim=2048)       # conf/model/clip_conv.yaml:6-22
METRIC = "3s-segments/sec (training step: SimpleConv fwd + ClipLoss + bwd + Adam)"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def host_threads() -> int:
    """Threads for the CPU arm: BM_CPU_THREADS, else one per physical core (logical / 2 on these SMT-2 hosts).  Set
    EXPLICITLY with torch.set_num_threads: torchrun exports OMP_NUM_THREADS=1, which starved round 1's N>1 reference arm."""
    env = os.environ.get("BM_CPU_THREADS")
    if env:
        return max(1, int(env))
    n = os.cpu_count() or 1
    return max(1, n // 2) if n >= 4 else n


# ------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY.md 8(d)): generated on CPU, pinned, shared by the e2e and resident runs
# ------------------------------------------------------------------------------------------------------
def make_host_batch(cfg, B, seed):
    g = torch.Generator().manual_seed(seed)
    C, T, F, S = cfg["C"], cfg["T"], cfg["F"], cfg["S"]
    meg = torch.randn(B, C, T, generator=g).clamp_(-20, 20)
    feats = torch.randn(B, F, T, generator=g)
    subj = torch.randint(0, S, (B,), generator=g)
    if cfg["n_valid"]:                                  # mixed studies: sensors beyond a study's own count are zero padding
        nv = cfg["n_valid"]                             # (bm/dataset.py:353-354, 471)
        for b in range(B):
            meg[b, nv[int(subj[b]) % len(nv)]:] = 0
    return meg, feats, subj


def local_batch(cfg, world):
    if cfg["global_batch"] is not None:
        assert cfg["global_batch"] % world == 0
        return cfg["global_batch"] // world, "strong"
    return cfg["batch_per_gpu"], "weak"


def run_b200(args):
    import torch.distributed as dist
    import brainmagick_b200 as bb
    from brainmagick_b200 import _lib, distrib, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the B200 arm)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    _lib.load()

    cfg = CONFIGS[args.config]
    B, scaling = local_batch(cfg, world)
    if args.batch:
        B, scaling = args.batch, "weak"
    C, T, F, S = cfg["C"], cfg["T"], cfg["F"], cfg["S"]
    torch.manual_seed(2036)                                             # conf/config.yaml:33
    model = bb.SimpleConv(in_channels=dict(meg=C), out_channels=F, n_subjects=S,
                          **{k: (dict(v) if isinstance(v, dict) else v) for k, v in CLIP_CONV.items()}).to(dev)
    clip = bb.ClipLoss(global_negatives=world > 1, uniform_batches=True).to(dev)
    model.train()
    clip.train()
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, betas=(0.9, 0.999), fused=True)   # bm/train.py:119
    positions = synthetic.normalised_positions(S, C, n_valid=cfg["n_valid"], seed=7)
    mask = torch.ones(B, 1, T, dtype=torch.bool, device=dev)

    n_host = 2                                                          # rotate two different host batches
    host = []
    for i in range(n_host):
        meg, feats, subj = make_host_batch(cfg, B, 2036 + 1000 * rank + i)
        host.append((meg.pin_memory(), feats.pin_memory(), subj.pin_memory(), subj.tolist()))
    resident = [tuple(t.to(dev) for t in hb[:3]) for hb in host]
    recs = [synthetic.SyntheticRecording(s, positions[s]) for s in range(S)]

    diag_step = os.environ.get("BM_STEP_DIAG", "")
    last = {}                                          # --dump-outputs: the latest step's loss and estimate

    def make_batch(meg_d, subj_d, subj_h):
        return synthetic.SyntheticBatch(meg_d, subj_d, [recs[s] for s in subj_h])

    def step(meg_d, feats_d, subj_d, subj_h):
        opt.zero_grad(set_to_none=True)
        batch = make_batch(meg_d, subj_d, subj_h)
        clip.prefetch_candidates(feats_d)          # N > 1: the candidate all-gather overlaps the encoder forward
        est = model(dict(meg=meg_d), batch)
        loss = clip(est, feats_d, mask)
        loss.backward()
        if world > 1 and diag_step != "no_allreduce":      # (BM_STEP_DIAG: diagnostic only)
            distrib.sync_gradients(model.parameters())
        opt.step()
        if args.dump_outputs:
            last.update(loss=loss, estimate=est)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]
    per_step = []

    def timed(n_steps, fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        marks = []
        for i in range(n_steps):
            fn(i)
            ev = torch.cuda.Event(enable_timing=True)               # per-step boundaries (diagnostic: drift inside the region)
            ev.record()
            marks.append(ev)
            if i == 1:                     # host time to ENQUEUE a step, from the first two steps after the barrier: the launch
                host_ms[0] = (time.perf_counter() - t0) * 1e3 / 2        # queue is still far from full, so nothing blocks
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        prev = e0
        per_step.clear()
        for ev in marks:
            per_step.append(round(prev.elapsed_time(ev), 3))
            prev = ev
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- device-resident throughput (`value`) ---------------------------------------------------------
    def resident_step(i):
        meg_d, feats_d, subj_d = resident[i % n_host]
        step(meg_d, feats_d, subj_d, host[i % n_host][3])

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                 # before the warm-up steps (the same workload): nvidia-smi needs ~0.3 s to deliver its
    for i in range(args.warmup):       # first sample and a short timed region would otherwise end before it
        resident_step(i)
    launches0 = _lib.launch_count()
    ms_total = timed(args.steps, resident_step)
    launches = _lib.launch_count() - launches0
    step_ms = list(per_step)
    host_ms_value = host_ms[0]        # >= ms_per_step would mean the host, not the GPU, paces the step
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms_total / args.steps
    value = world * B / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:            # before the e2e steps below move the model on
        dump_outputs(args.dump_outputs, last["loss"], last["estimate"], model)

    # ---- end to end through the public API with HOST buffers (`e2e`) ------------------------------------
    # every step copies its inputs from pinned host memory (on a copy stream, one step ahead, like a DataLoader that
    # prefetches to the device) and reads the loss back to the host; all of it inside the timed region.
    last_loss = [0.0]
    copy_stream = torch.cuda.Stream(device=dev)
    slots = [None, None]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    # The big input (features, 377 MB) is split into chunks issued round-robin on BM_E2E_COPY_STREAMS copy streams (default 2).
    # The step's copies reach 55 GB/s alone (8.2 ms); on one box of the pool they fell to ~18 GB/s while the step's kernels
    # were running and the e2e step became copy-bound (24.8 ms against 16.4 ms of compute) -- not reproduced on other boxes,
    # where 1, 2 and 4 streams all give e2e = step + 1.2-1.5 ms (pipeline fill of the first batch + the loss read-back).
    n_cs = max(1, int(os.environ.get("BM_E2E_COPY_STREAMS", "2")))
    copy_streams = [copy_stream] + [torch.cuda.Stream(device=dev) for _ in range(n_cs - 1)]
    joined = [[torch.cuda.Event() for _ in range(n_cs)] for _ in range(2)]

    def issue_copy(i):
        meg_h, feats_h, subj_h, subj_l = host[i % n_host]
        k = i % 2
        if diag == "no_copy":                          # diagnostic only: the e2e loop without the host->device copies
            slots[k] = resident[i % n_host] + (subj_l,)
            ready[k].record(copy_stream)
            return
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k])                         # the step that used this slot has finished
            feats_d = torch.empty(feats_h.shape, device=dev, dtype=feats_h.dtype)
            meg_d = meg_h.to(dev, non_blocking=True)
            subj_d = subj_h.to(dev, non_blocking=True)
            start = torch.cuda.Event()
            start.record(copy_stream)
        rows = feats_h.shape[0]
        per = -(-rows // (2 * n_cs))
        for c, r0 in enumerate(range(0, rows, per)):
            cs = copy_streams[c % n_cs]
            with torch.cuda.stream(cs):
                if cs is not copy_stream and r0 < per * n_cs:
                    cs.wait_event(start)                                # the destination exists and its slot is free
                feats_d[r0:r0 + per].copy_(feats_h[r0:r0 + per], non_blocking=True)
        for j, cs in enumerate(copy_streams):
            joined[k][j].record(cs)
        with torch.cuda.stream(copy_stream):
            for j in range(1, n_cs):
                copy_stream.wait_event(joined[k][j])
            slots[k] = (meg_d, feats_d, subj_d, subj_l)
            ready[k].record(copy_stream)

    # device -> host read of a step's result EVERY step, pipelined by one step: the loss is copied into pinned host memory
    # right behind the step that produced it and the host waits for THAT copy's event while the next step is already queued
    # (like a training loop that logs the previous iteration's loss).  `loss.item()` would do the same copy but then
    # synchronise the whole stream -- including the step just enqueued -- and leave the GPU idle between the ~60 tiny
    # kernels at the start of the next forward pass while the host catches up (measured: +1.3-1.8 ms per step).
    diag = os.environ.get("BM_E2E_DIAG", "")
    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_run(n_steps):
        main = torch.cuda.current_stream()
        for k in range(2):
            consumed[k].record(main)
        issue_copy(0)
        for i in range(n_steps):
            if i + 1 < n_steps:
                issue_copy(i + 1)
            k = i % 2
            main.wait_event(ready[k])
            meg_d, feats_d, subj_d, subj_l = slots[k]
            if diag == "compute_on_resident":          # diagnostic only (BM_E2E_DIAG): copies still run, the step ignores them
                meg_d, feats_d, subj_d = resident[i % n_host]
            loss = step(meg_d, feats_d, subj_d, subj_l)
            consumed[k].record(main)
            loss_host[k].copy_(loss.detach().reshape(1), non_blocking=True)
            loss_ready[k].record(main)
            if i > 0 and diag != "no_readback":
                loss_ready[1 - k].synchronize()                          # step i-1's loss has landed in host memory
                last_loss[0] = float(loss_host[1 - k][0])
        k = (n_steps - 1) % 2
        loss_ready[k].synchronize()
        last_loss[0] = float(loss_host[k][0])

    e2e_run(min(2, args.warmup))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(args.steps)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    if world > 1:
        tt = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_e2e = float(tt.item())
    h2d = sum(t.numel() * t.element_size() for t in host[0][:3])
    # the same pinned -> device copies ALONE (nothing else running): the floor the interconnect puts under an e2e step
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(3):
        keep = [t.to(dev, non_blocking=True) for t in host[0][:3]]
    c1.record()
    torch.cuda.synchronize()
    h2d_ms_alone = c0.elapsed_time(c1) / 3
    del keep
    e2e = dict(value=world * B / (ms_e2e / 1e3), unit="segments/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4,
               ms_per_step=ms_e2e, h2d_ms_alone=h2d_ms_alone, h2d_gb_per_s_alone=h2d / h2d_ms_alone / 1e6,
               note="inputs copied from pinned host memory on a copy stream one step ahead; the loss of every step is copied to "
                    "pinned host memory and read by the host one step behind (event wait, not a stream synchronise); h2d_ms_alone = the step's host->device copies with nothing else running (when it approaches "
                    "ms_per_step the interconnect, not the GPU, paces the e2e step)")

    # ---- rooflines: the dominant kernel (K3 dilated conv) + the other kernels the north star names --------
    roofline = None
    cpu_baseline = None
    also = None
    if rank == 0:
        roofline, others = kernel_rooflines(dev, B, T, F, B * world)
        roofline["other_kernels"] = others
        if world == 1 and not args.lean:
            also = also_measured(cfg, model, clip, make_batch, resident, host, n_host, mask, dev, B)
        if not args.no_cpu_baseline and world == 1:
            cpu_baseline = run_cpu(cfg, steps=2, warmup=1, batch=32, threads=host_threads())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    from brainmagick_b200 import functional as BF
    BF.check_tc_status()
    if rank != 0:
        return
    act_gb = 5.0 * B / 256
    out = dict(
        metric=METRIC, value=value, unit="segments/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=ms_per_step, higher_is_better=True, scaling=scaling, vs_baseline=None, dtype="f32", data="synthetic",
        config=dict(workload=cfg["name"], batch_per_gpu=B, global_batch=B * world, sensors=C, T=T, F=F,
                    subjects=S, model="clip_conv (random init)", negatives="global (all-gather)" if world > 1 else "local",
                    arithmetic="fp32-faithful (parity 1e-4): every product = 3 tensor-core MMAs over two-piece operands, fp32 "
                               "accumulation in tensor memory -- fp16 pieces on tcgen05 kind::f16 (convs, weight gradients), "
                               "tf32 pieces on kind::tf32 (CLIP, grouped / per-sample 1x1); elementwise in fp32",
                    l2=f"per-step working set (inputs {h2d / 1e6:.0f} MB + ~{act_gb:.1f} GB saved activations) >> 126 MB L2; "
                       "two input batches rotate",
                    last_loss=last_loss[0]),
        host_enqueue_ms_per_step=host_ms_value, step_ms=step_ms,
        clocks=clocks, e2e=e2e, gpu_launches=int(launches), roofline=roofline, cpu_baseline=cpu_baseline, also=also)
    emit(json.dumps(out))


DUMP_ROWS = 8                  # segments of the estimate written by --dump-outputs
DUMP_GRAD_MAX = 1 << 20        # entries of one gradient written in full; a larger one is sampled down to this many


def dump_outputs(out_dir, loss, est, model):
    """What one training step hands its caller, as float32 .npy files under `out_dir`: `loss`, `estimate` (DUMP_ROWS
    segments of the [B, F, T] estimate) and `grad.<parameter>` (flattened; beyond DUMP_GRAD_MAX entries, that many of
    them in ascending order).  Rows and entries are drawn by generators with fixed seeds, so that the same arguments write
    the same selection and two builds can be compared file by file.  About 46 MB at cfg2, under 64 MB at every config."""
    import zlib
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rows = torch.randperm(est.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    arrays = {"loss": loss.detach().reshape(()), "estimate": est.detach()[rows.to(est.device)]}
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.detach().reshape(-1)
        if g.numel() > DUMP_GRAD_MAX:
            gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            g = g[torch.randperm(g.numel(), generator=gen)[:DUMP_GRAD_MAX].sort().values.to(g.device)]
        arrays["grad." + name] = g
    total = 0
    for name, a in arrays.items():
        a = a.float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        total += a.nbytes
    assert total <= 64 << 20, f"--dump-outputs wrote {total / 2**20:.1f} MiB"


def also_measured(cfg, model, clip, make_batch, resident, host, n_host, mask, dev, B, iters=5):
    """What SURVEY.md 8(d) asks to report beside the headline (N=1 only, after the headline has been timed; every part is
    optional and a failure is recorded instead of raised):
      * forward_only: the encoder in eval mode under no_grad (the evaluation-time cost), segments/s;
      * torch_eager_gpu: the SAME step (forward + ClipLoss + backward, no optimizer) written in plain PyTorch ops -- the
        oracle restatement of the reference modules -- run on this GPU with cuDNN / cuBLAS: the "library-kernel" bar,
        with TF32 off (fp32-faithful like this repo) and on."""
    out = {}

    def timed_ms(fn, n):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    try:
        model.eval()

        def fwd(i=0):
            meg_d, _, subj_d = resident[i % n_host]
            with torch.no_grad():
                model(dict(meg=meg_d), make_batch(meg_d, subj_d, host[i % n_host][3]))
        ms = timed_ms(fwd, iters)
        out["forward_only"] = dict(value=B / (ms / 1e3), unit="segments/s", ms_per_batch=ms, mode="eval, no_grad")
    except Exception as exc:
        out["forward_only"] = dict(error=f"{type(exc).__name__}: {exc}")
    finally:
        model.train()

    try:
        from oracle import bm_oracle
        from brainmagick_b200 import synthetic
        C, T, F, S = cfg["C"], cfg["T"], cfg["F"], cfg["S"]
        ocfg = bm_oracle.Config(in_channels=C, out_channels=F, n_subjects=S)
        params = {k: v.detach().clone() for k, v in model.state_dict().items()}
        meg_d, feats_d, subj_d = resident[0]
        pos = synthetic.normalised_positions(S, C, n_valid=cfg["n_valid"], seed=7).to(dev)
        ban = torch.tensor([0.5, 0.5], device=dev)
        saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        res = {}
        try:
            for label, tf32 in (("tf32_off", False), ("tf32_on", True)):
                torch.backends.cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = tf32

                def eager(i=0):
                    bm_oracle.training_step(params, ocfg, meg_d, pos, subj_d, subj_d, feats_d, ban_centre=ban, training=True)
                ms = timed_ms(eager, 3)
                res[label] = dict(value=B / (ms / 1e3), unit="segments/s", ms_per_step=ms)
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        res["what"] = "oracle restatement of SimpleConv + ClipLoss in PyTorch ops on this GPU: forward + loss + backward, no optimizer"
        out["torch_eager_gpu"] = res
    except Exception as exc:
        out["torch_eager_gpu"] = dict(error=f"{type(exc).__name__}: {exc}")
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------
# kernel rooflines: each kernel alone, back to back over rotating operand sets larger than L2, CUDA events on the launching stream
# ------------------------------------------------------------------------------------------------------
def ncu_traffic_bytes(pattern):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from this round's committed `ncu --set full` summary
    (profiles/r2*_ncu_<pattern>_summary.csv, made from the .ncu-rep with `ncu -i ... --page raw --csv`); None if absent."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", f"r2*_ncu_{pattern}_summary.csv")))
    if not files:
        return None
    try:
        rows = list(csv.reader(open(files[-1])))
        hdr, units, data = rows[0], rows[1], rows[2:]
        tot = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(name)
            scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[units[i]]
            tot += sum(float(v[i]) for v in data) * scale
        # one captured launch per row; the BatchNorm backward is a kernel PAIR (reduce + apply) captured once each
        return tot / (len(data) / 2.0 if pattern == "bn_bwd" else len(data))
    except Exception:
        return None


def _time_kernel(fns, flush=None, iters=24, skip=4):
    """Mean duration of one launch, the way the training step runs it: back to back on the launching stream, CUDA events
    around `iters` launches.  `fns` = the same launch over ROTATING operand sets whose combined footprint is several times
    the 126 MB L2 (timing rule: inputs larger than L2), so no launch finds its operands cached by the previous one."""
    if callable(fns):
        fns = [fns]
    for i in range(skip):
        fns[i % len(fns)]()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fns[i % len(fns)]()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_rooflines(dev, B, T, F, Bc, H=320, Kw=3):
    """The dominant kernel first (K3: Conv1d 320->320 k3 + BatchNorm statistics, half of the step with its data-gradient
    twin), then K4 (Conv1d 320->640 + GLU), K6 (CLIP scores + norms + softmax/CE), the weight-gradient kernel and the
    HBM-bound BatchNorm/GELU kernels.  Algorithmic work per SURVEY.md 8(d); the tensor pipe executes 3x the algorithmic
    FLOPs (hi*hi + lo*hi + hi*lo): at the f16 rate a tensor-bound `frac` against the measured bf16 peak tops out at 1/3, at
    the tf32 rate (= bf16 / 2) at 1/6 -- `frac_of_scheme_ceiling` is the same number against that ceiling."""
    from brainmagick_b200._lib import call, ptr, stream, load
    lib = load()
    peaks = load_peaks()
    peak_tf, peak_gb = peaks["bf16_tflops"], peaks["hbm_gbs"]
    src = peaks["source"]
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    flush = None
    st = stream()
    NSETS = 3                                               # 3 x (118 MB in + >= 118 MB out) per conv launch >> L2
    xs = [torch.randn(B, T, H, device=dev) for _ in range(NSETS)]
    x = xs[0]
    w = torch.randn(H, H, Kw, device=dev) * 0.03
    wg = torch.randn(2 * H, H, Kw, device=dev) * 0.03
    f, g = torch.empty(Kw, H, H, device=dev), torch.empty(Kw, H, H, device=dev)
    fg = torch.empty(Kw, 2 * H, H, device=dev)
    call("bm_tc_weight_split", ptr(w), H, H, Kw, ptr(f), None, ptr(g), None, st)
    call("bm_tc_weight_split", ptr(wg), 2 * H, H, Kw, ptr(fg), None, None, None, st)
    bias = torch.zeros(H, device=dev)
    ys = [torch.empty(B, T, H, device=dev) for _ in range(NSETS)]
    y = ys[0]
    h = torch.empty(B, T, 2 * H, device=dev)
    stats = torch.empty(2 * H, device=dev, dtype=torch.float64)

    def tensor_entry(kernel, ms, flops, alg_bytes, traffic, pipe="tf32"):
        """`frac` is against the measured dense bf16 peak.  An fp32-faithful product needs three MMAs (hi*hi + lo*hi + hi*lo):
        on kind::tf32 (half the bf16 rate) the ceiling of `frac` is 1/6, on kind::f16 it is 1/3 -- `frac_of_scheme_ceiling`."""
        ach = flops / (ms / 1e3) / 1e12
        ceil = peak_tf / (6 if pipe == "tf32" else 3)
        return dict(kernel=kernel, bound="tensor", achieved=ach, peak=peak_tf, unit="TFLOP/s", frac=ach / peak_tf,
                    traffic=traffic, algorithmic_bytes=alg_bytes, ms_per_launch=ms,
                    peak_source=src + " cuBLAS bf16 burst (MEASURED_PEAKS.json)", pipe="kind::" + pipe,
                    executed_tflops_bf16_equivalent=(6 if pipe == "tf32" else 3) * ach, frac_of_scheme_ceiling=ach / ceil)

    def hbm_entry(kernel, ms, alg_bytes, traffic):
        ach = alg_bytes / (ms / 1e3) / 1e9
        return dict(kernel=kernel, bound="hbm", achieved=ach, peak=peak_gb, unit="GB/s", frac=ach / peak_gb,
                    traffic=traffic, algorithmic_bytes=alg_bytes, ms_per_launch=ms,
                    peak_source=src + " copy bandwidth (MEASURED_PEAKS.json)")

    def f16_weights(w_op):
        amax = torch.empty(1, device=dev)
        call("bm_amax", ptr(w_op), w_op.numel(), ptr(amax), st)
        hi = torch.empty(w_op.shape, device=dev, dtype=torch.float16)
        lo = torch.empty(w_op.shape, device=dev, dtype=torch.float16)
        call("bm_f16_split", ptr(w_op), w_op.numel(), ptr(amax), ptr(hi), ptr(lo), st)
        return hi, lo, amax

    def amax_of(t):
        cell = torch.empty(1, device=dev)
        call("bm_amax", ptr(t), t.numel(), ptr(cell), st)
        return cell

    # the kernels the training step runs: the persistent CTA-pair conv on the F16 pipe (bm_tc_conv1d_f16)
    fh, fl, fa = f16_weights(f)
    gh, gl, ga = f16_weights(g)
    fgh, fgl, fga = f16_weights(fg)
    xa = [amax_of(x) for x in xs]
    out_amax = torch.empty(1, device=dev)
    ms = _time_kernel([lambda x=x, y=y, a=a: call("bm_tc_conv1d_f16", ptr(x), ptr(a), ptr(fh), ptr(fl), ptr(fa), ptr(bias), 0, B, T,
                                                  H, H, Kw, 4, 1, 0, 0, 0, ptr(y), None, None, ptr(stats), None, ptr(status), st)
                       for x, y, a in zip(xs, ys, xa)])
    main = tensor_entry("conv_hp_kernel via bm_tc_conv1d_f16 (K3: Conv1d 320->320 k3 d4 + BatchNorm statistics; persistent CTA "
                        "pairs, tcgen05 cta_group::2 kind::f16, fp32 operands as fp16 hi/lo pieces)", ms,
                        2.0 * H * H * Kw * T * B, 2.0 * B * T * H * 4, ncu_traffic_bytes("convh"), pipe="f16")
    main["note"] = ("achieved = ALGORITHMIC fp32 FLOPs (2*320*320*3*T*B per launch) / time; fp32-faithful parity (1e-4) takes "
                    "three MMAs per product, so the ceiling of `frac` is 1/3 on kind::f16 (1/6 on kind::tf32): see "
                    "frac_of_scheme_ceiling")
    others = []
    try:
        ms = _time_kernel([lambda x=x, y=y, a=a: call("bm_tc_conv1d_f16", ptr(x), ptr(a), ptr(fgh), ptr(fgl), ptr(fga), None, 0,
                                                      B, T, H, 2 * H, Kw, 1, 1, 1, 0, 0, ptr(h), None, ptr(y), None,
                                                      ptr(out_amax), ptr(status), st) for x, y, a in zip(xs, ys, xa)])
        others.append(tensor_entry("conv_hp_kernel GLU mode (K4: Conv1d 320->640 k3 + GLU, h saved, max |out| reported)", ms,
                                   4.0 * H * H * Kw * T * B, 4.0 * B * T * H * 4, ncu_traffic_bytes("convh_glu"), pipe="f16"))
        ms = _time_kernel([lambda x=x, y=y, a=a: call("bm_tc_conv1d_f16", ptr(x), ptr(a), ptr(gh), ptr(gl), ptr(ga), None, 1, B,
                                                      T, H, H, Kw, 4, -1, 0, 0, 0, ptr(y), None, None, None, None, ptr(status),
                                                      st) for x, y, a in zip(xs, ys, xa)])
        others.append(tensor_entry("conv_hp_kernel data gradient, y += tile (TMA reduce-add)", ms, 2.0 * H * H * Kw * T * B,
                                   3.0 * B * T * H * 4, ncu_traffic_bytes("convh_acc"), pipe="f16"))
        # the 3xTF32 variant of the same kernel (round 2's first half; still what runs where USE_CONV_F16 is off)
        ms = _time_kernel([lambda x=x, y=y: call("bm_tc_conv1d_persistent", ptr(x), ptr(f), ptr(bias), 0, B, T, H, H, Kw, 4, 1,
                                                 0, 0, 0, ptr(y), None, None, ptr(stats), ptr(status), st)
                           for x, y in zip(xs, ys)])
        others.append(tensor_entry("conv_pp_kernel via bm_tc_conv1d_persistent (K3 on kind::tf32, 3xTF32: for comparison)", ms,
                                   2.0 * H * H * Kw * T * B, 2.0 * B * T * H * 4, ncu_traffic_bytes("convp")))
        # K6: CLIP scores + candidate norms + softmax / CE / mean at the training shape (Bn = local rows, Bc = global rows)
        KT = F * T
        est = torch.randn(B, KT, device=dev) * 0.01
        cand = torch.randn(Bc, KT, device=dev)
        inv, sc, pr = torch.empty(Bc, device=dev), torch.empty(B, Bc, device=dev), torch.empty(B, Bc, device=dev)
        rl, loss = torch.empty(B, device=dev), torch.empty(1, device=dev)
        ws = torch.empty(max(int(lib.bm_clip_workspace(B, Bc, KT)), 2), device=dev)
        ms = _time_kernel(lambda: call("bm_clip_loss_fwd", ptr(est), ptr(cand), B, Bc, KT, 0, ptr(inv), ptr(sc), ptr(pr),
                                       ptr(rl), ptr(loss), ptr(ws), ws.numel(), ptr(status), st))
        e = tensor_entry(f"clip_scores_kernel + clip_finalize_kernel via bm_clip_loss_fwd (K6: {B} x {Bc} x {KT}, norms and "
                         "softmax/CE fused; split-K CTA pairs, bounded accumulation chains)", ms, 2.0 * B * Bc * KT,
                         4.0 * KT * (B + Bc), ncu_traffic_bytes("clip"))
        hbm = 4.0 * KT * (B + Bc) / (ms / 1e3) / 1e9
        e["hbm_view"] = dict(achieved=hbm, peak=peak_gb, unit="GB/s", frac=hbm / peak_gb,
                             note="arithmetic intensity B*Bc/(2(B+Bc)) FLOP/B: at 256 x 256 the kernel sits near the ridge "
                                  "of 3xTF32 (SURVEY 8d), so both views are given")
        others.append(e)
        del est, cand
        # weight gradient (K3 shape)
        dys = [torch.randn(B, T, H, device=dev) for _ in range(NSETS)]
        dy = dys[0]
        dw = torch.empty(H, H, Kw, device=dev)
        # the kernel the training step uses for this layer (functional.tc_wgrad's choice): CTA pairs, rows = (tap, x channel)
        assert lib.bm_tc_wgrad_conv_supported(T, H, H, Kw)
        wsg = torch.empty(int(lib.bm_tc_wgrad_conv_workspace(B, T, H, H, Kw)), device=dev)
        dya = [amax_of(dy) for dy in dys]
        ms = _time_kernel([lambda x=x, dy=dy, a=a, b=b: call("bm_tc_wgrad_conv_f16", ptr(dy), ptr(b), ptr(x), ptr(a), B, T, H, H, H,
                                                             Kw, 4, ptr(wsg), ptr(dw), ptr(status), st)
                           for x, dy, a, b in zip(xs, dys, xa, dya)])
        others.append(tensor_entry("wgrad_hp_kernel (+reduce) via bm_tc_wgrad_conv_f16 (weight gradient of K3, kind::f16)", ms,
                                   2.0 * H * H * Kw * T * B, 2.0 * B * T * H * 4, ncu_traffic_bytes("wgradh"), pipe="f16"))
        ms = _time_kernel([lambda x=x, dy=dy: call("bm_tc_wgrad_conv", ptr(dy), ptr(x), B, T, H, H, H, Kw, 4, ptr(wsg), ptr(dw),
                                                   ptr(status), st) for x, dy in zip(xs, dys)])
        others.append(tensor_entry("wgrad_pp_kernel (+reduce) via bm_tc_wgrad_conv (the same on kind::tf32: for comparison)", ms,
                                   2.0 * H * H * Kw * T * B, 2.0 * B * T * H * 4, ncu_traffic_bytes("wgrad")))
        del wsg
        # ... and of the GLU conv (640 x 320 x 3): the second-largest share of the step after the convs
        dy2 = torch.randn(B, T, 2 * H, device=dev)
        dy2a = amax_of(dy2)
        dw2 = torch.empty(2 * H, H, Kw, device=dev)
        wsg = torch.empty(int(lib.bm_tc_wgrad_conv_workspace(B, T, 2 * H, H, Kw)), device=dev)
        ms = _time_kernel([lambda x=x, a=a: call("bm_tc_wgrad_conv_f16", ptr(dy2), ptr(dy2a), ptr(x), ptr(a), B, T, 2 * H, H, H,
                                                 Kw, 1, ptr(wsg), ptr(dw2), ptr(status), st) for x, a in zip(xs, xa)])
        others.append(tensor_entry("wgrad_hp_kernel (+reduce) via bm_tc_wgrad_conv_f16 (weight gradient of K4)", ms,
                                   2.0 * 2 * H * H * Kw * T * B, 3.0 * B * T * H * 4, None, pipe="f16"))
        del wsg, dy2, dw2
        # HBM-bound: BatchNorm + GELU (+skip) backward and forward
        gam, bet = torch.ones(H, device=dev), torch.zeros(H, device=dev)
        mean, invstd = torch.zeros(H, device=dev), torch.ones(H, device=dev)
        sums = torch.empty(2 * H, device=dev, dtype=torch.float64)
        dgam, dbet = torch.empty(H, device=dev), torch.empty(H, device=dev)
        rows = B * T
        amax = torch.empty(1, device=dev)                     # max |output| for the F16-pipe conv downstream, as in the step
        ms = _time_kernel([lambda x=x, dy=dy, gy=gy: call("bm_bn_gelu_skip_bwd", ptr(dy), ptr(x), ptr(mean), ptr(invstd),
                                                          ptr(gam), ptr(bet), 1, rows, H, ptr(sums), ptr(gy), ptr(dgam),
                                                          ptr(dbet), ptr(amax), st) for x, dy, gy in zip(xs, dys, ys)])
        e = hbm_entry("bm_bn_gelu_skip_bwd (BatchNorm + GELU backward: reduce pass + apply pass)", ms, 3.0 * rows * H * 4,
                      ncu_traffic_bytes("bn_bwd"))
        two = 5.0 * rows * H * 4 / (ms / 1e3) / 1e9
        e["two_pass_view"] = dict(achieved=two, peak=peak_gb, unit="GB/s", frac=two / peak_gb,
                                  note="algorithmic = read dy, read x, write dx once (3 arrays); the batch statistics of the "
                                       "gradient must be complete before any dx is written and 236 MB does not stay in L2, "
                                       "so the kernel pair necessarily moves 5 arrays (2 reads for the sums, 2 reads + 1 write)")
        others.append(e)
        ms = _time_kernel([lambda x=x, dy=dy, gy=gy: call("bm_bn_gelu_skip_fwd", ptr(dy), ptr(mean), ptr(invstd), ptr(gam),
                                                          ptr(bet), ptr(x), ptr(gy), rows, H, ptr(amax), st)
                           for x, dy, gy in zip(xs, dys, ys)])
        others.append(hbm_entry("bm_bn_gelu_skip_fwd (BatchNorm apply + GELU + skip)", ms, 3.0 * rows * H * 4,
                                ncu_traffic_bytes("bn_fwd")))
    except Exception as exc:
        others.append(dict(error=f"{type(exc).__name__}: {exc}"))
    assert int(status.item()) == 0, "a tcgen05 kernel reported a pipeline timeout"
    return main, others


# ------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own modules (staged under baseline/_ref by oracle/stage_reference.py) on the host cores
# ------------------------------------------------------------------------------------------------------
def run_cpu(cfg, steps, warmup, batch, threads):
    """A bounded sample of the workload on the host: `steps` training steps of `batch` segments at the configuration's
    shapes.  kind "reference" = the VERBATIM bm.models.SimpleConv + bm.losses.ClipLoss under the step harness of
    oracle/ref_trainer.py; kind "port" (only if the staged reference is missing) = the oracle restatement."""
    from oracle import ref_loader
    torch.set_num_threads(threads)
    meg, feats, subj = make_host_batch(cfg, batch, 2036)
    if ref_loader.reference_available():
        from oracle import ref_trainer
        tr = ref_trainer.VerbatimTrainer(cfg["C"], cfg["F"], cfg["S"], n_valid=cfg["n_valid"])

        def one():
            return tr.step(meg, feats, subj)
        kind = "reference"
        what = f"verbatim bm.models.SimpleConv + bm.losses.ClipLoss ({ref_loader.REF_KIND}), fwd+loss+bwd+Adam"
    else:
        from oracle import bm_oracle
        ocfg = bm_oracle.Config(in_channels=cfg["C"], out_channels=cfg["F"], n_subjects=cfg["S"])
        tr = bm_oracle.CpuTrainer(ocfg, bm_oracle.init_state_dict(ocfg, seed=0))
        d = bm_oracle.synthetic_batch(ocfg, batch=batch, T=cfg["T"], seed=2036, n_valid=cfg["n_valid"])

        def one():
            return tr.step(d["meg"], d["rec_positions"], d["rec_of_sample"], d["subject_index"], d["candidates"], d["ban_centre"])
        kind = "port"
        what = "oracle/bm_oracle.py CpuTrainer (baseline/_ref not staged), fwd+loss+bwd+Adam"
    for _ in range(warmup):
        one()
    per = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one()
        per.append(time.perf_counter() - t0)
    dt = statistics.mean(per)
    return dict(value=batch / dt, unit="segments/s", cores=torch.get_num_threads(), kind=kind,
                sample=f"{steps} steps of B={batch} at the {cfg['name'].split()[0]} shapes ({what}); host has "
                       f"{os.cpu_count()} logical cores", s_per_step=dt, s_per_step_min=min(per), s_per_step_max=max(per))


def run_reference(args):
    """Reference arm: rank 0 alone (the other ranks exit 0 without work), threads set explicitly."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    threads = host_threads()
    batch = 64                                   # bounded sample per step; CPU seg/s is batch-insensitive (SURVEY 8d)
    res = run_cpu(cfg, steps=args.steps, warmup=min(args.warmup, 2), batch=batch, threads=threads)
    also = {}
    try:                                         # what bm/train.py:182 actually sets: ONE thread
        also["one_thread"] = run_cpu(cfg, steps=1, warmup=0, batch=8, threads=1)
        torch.set_num_threads(threads)
        if not args.lean:                        # one step at the full B=256 of the metric
            also["full_batch"] = run_cpu(cfg, steps=1, warmup=0, batch=256, threads=threads)
    except Exception as exc:
        also["error"] = f"{type(exc).__name__}: {exc}"
    out = dict(
        impl="reference", metric=METRIC, value=res["value"], unit="segments/s", n_gpus=args.gpus, steps=args.steps,
        warmup=args.warmup, ms_per_step=res["s_per_step"] * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
        dtype="f32", data="synthetic",
        config=dict(workload=cfg["name"], batch_per_step=batch, sensors=cfg["C"], T=cfg["T"], F=cfg["F"],
                    subjects=cfg["S"], model="clip_conv (random init)",
                    note="the reference's own SimpleConv + ClipLoss (unmodified files staged under baseline/_ref by "
                         "oracle/stage_reference.py) under the restated Solver step; bounded sample of B=64 per step, "
                         f"{threads} threads set with torch.set_num_threads (also under torchrun)"),
        cpu_baseline=res, also=also,
        e2e=dict(value=res["value"], unit="segments/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    emit(json.dumps(out))


_REAL_STDOUT = None


def emit(line: str) -> None:
    """The result line, on the process's ORIGINAL stdout."""
    data = (line + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line + "\n")
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # stdout carries ONE JSON line.  Libraries write there too (NCCL's version banner at communicator creation, NCCL_DEBUG
    # output): file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor.
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    # The step uses ~7 streams per rank (main, weight-gradient side stream, candidate gather, NCCL, input copies).  With
    # the default 8 hardware work queues streams alias: at N = 2 the resident loop then showed 20-50 ms stalls every few
    # steps (a spinning symmetric-memory barrier kernel ahead of an NCCL kernel in the same queue); none with 32 queues.
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="override the batch per GPU (default: the configuration's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lean", action="store_true", help="skip the `also` extras (forward-only, eager-PyTorch bar, B=256 CPU step)")
    ap.add_argument("--next-rows", action="store_true",
                    help="instead of the headline step: the SURVEY 8(f) rows (batch preparation, retrieval evaluation, "
                         "DeepMel), each beside a bounded CPU sample of its oracle; one GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last one's loss, estimate and gradients to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.next_rows):
        ap.error("--dump-outputs applies to the B200 training step")
    if args.next_rows:
        from profiles import bench_next_rows      # its CPU legs are this file's cpu_baseline leg for those rows
        bench_next_rows.main(emit=emit)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
