"""autograd.Functions that run the hot path through the C ABI (libbm_b200.so).

`encoder_forward` is SimpleConv.forward at the clip_conv configuration (bm/models/simpleconv.py:198-249) as ONE
autograd node: its backward launches the hand-written gradient kernels in reverse order, so `loss.backward()`
leaves ordinary dense `.grad` tensors on every parameter (what bm/solver.py:384-387 and
flashy.distrib.sync_model expect).  `clip_loss` / `clip_scores` are ClipLoss (bm/losses.py:77-114);
`regression_loss` is L1Loss / L2Loss (bm/losses.py:11-26).

Kernel selection is by shape only: contractions whose channel counts fit the tcgen05 tiling (K % 32 == 0 and an
N tile of 64..160 dividing N -- every layer of the real clip_conv model) run on the tensor-core kernels
(3xTF32, `bm_tc_*`); other shapes (the tiny unit-test models) run on the FP32-FMA kernels of the same library.
"""
from __future__ import annotations

import dataclasses
import typing as tp

import torch

from . import _lib
from ._lib import call, ptr, stream


@dataclasses.dataclass
class EncoderPlan:
    """Everything `encoder_forward` needs that is not a differentiable tensor."""
    dilations: tp.List[int]
    glu_after: tp.List[bool]
    kernel_size: int
    glu_kernel: int
    training: bool
    bn_eps: float
    bn_momentum: float
    rec_positions: torch.Tensor            # [R,C,2] fp32, rows = recordings present in the batch
    rec_of_sample: torch.Tensor            # [B] int32 -> row of rec_positions
    rec_order: torch.Tensor                # [B] int32 samples sorted by recording
    rec_off: torch.Tensor                  # [R+1] int32 CSR offsets
    subject: torch.Tensor                  # [B] int32
    freq: torch.Tensor                     # [sqrt(P/2)] fp32 Fourier frequencies
    ban_centre: tp.Optional[torch.Tensor]  # [2] fp32 or None
    ban_radius: float
    bn_buffers: tp.List[tp.Tuple[torch.Tensor, torch.Tensor]]   # (running_mean, running_var) per layer
    keep_for_backward: bool = True
    use_tensor_cores: bool = True
    skip: bool = True                      # ConvSequence(skip=...): residual where a layer keeps its width (common.py:146-147)
    act_code: int = 0                      # 0 = GELU (clip_conv); 1 = LeakyReLU(act_slope), i.e. simpleconv.gelu=False
    act_slope: float = 0.0
    bare_last: bool = False                # simpleconv.complex_out=False: no head, the last conv maps to out_channels and
                                           # has neither BatchNorm nor activation (simpleconv.py:190-193)
    staged: bool = False                   # a sensor-chain stage is missing (merger / initial_linear / subject_layers
                                           # ablations) or a subject embedding is appended: run the chain stage by stage
    has_sub_emb: bool = False              # the last tensor argument is the [B, E] subject-embedding rows


def _empty(shape, like, dtype=torch.float32):
    return torch.empty(shape, device=like.device, dtype=dtype)


_status: tp.Dict[torch.device, torch.Tensor] = {}


def tc_status_tensor(device) -> torch.Tensor:
    """Device int32 word the tcgen05 kernels set if their bounded pipeline waits ever time out."""
    device = torch.device(device)
    if device not in _status:
        _status[device] = torch.zeros(1, dtype=torch.int32, device=device)
    return _status[device]


def check_tc_status(device=None) -> None:
    """Synchronising check (tests, bench, end of epoch): raises if a tensor-core kernel reported a timeout."""
    for dev, t in _status.items():
        if device is None or torch.device(device) == dev:
            code = int(t.item())
            if code == 900:
                t.zero_()
                raise IndexError(f"a subject / recording index is outside the weight sets of the per-sample 1x1 layer on {dev} "
                                 "(bm/models/common.py:57 raises there too)")
            if code != 0:
                raise _lib.BmB200Error(f"a tcgen05 kernel reported a pipeline timeout (barrier code {code}) on {dev}")


OVERLAP_WGRAD = True   # weight-gradient kernels on a side stream, concurrent with the data-gradient kernels of the layer
USE_CONV_PP = True     # persistent CTA-pair kernel (tc_convp.cuh, tcgen05 cta_group::2) where its tiling fits


_side_streams: tp.Dict[torch.device, torch.cuda.Stream] = {}


def _side_stream(device) -> torch.cuda.Stream:
    device = torch.device(device)
    if device not in _side_streams:
        _side_streams[device] = torch.cuda.Stream(device=device)
    return _side_streams[device]


def _round_up(n, m):
    return (n + m - 1) // m * m


USE_CONV_F16 = True    # the persistent conv on the F16 tensor pipe (tc_convh.cuh: fp16 hi/lo pieces, twice the MMA rate of 3xTF32)
USE_WGRAD_F16 = True   # ... and the CTA-pair weight gradient (tc_wgradh.cuh)
USE_WGRAD_PP = True    # CTA-pair weight-gradient kernel (tc_wgradp.cuh) where its 256-row tiling wastes < 10 %


def tc_wgrad(dy, x, B, T, M, N, Ntrue, kw, dilation, status, dbias=None, dy_amax=None, x_amax=None):
    """dw[m][n][tap] = sum_{b,t} dy[b,t,m] x[b,t+(tap-kw//2)*dilation,n] on the tensor cores -> [M, Ntrue, kw];
    `dbias` [M] (optional) receives sum_{b,t} dy[b,t,m].  `dy_amax` / `x_amax` (F16 pipe): device floats with max |dy| /
    max |x| when their producers reported them, else a bm_amax pass here."""
    lib = _lib.load()
    dw = _empty((M, Ntrue, kw), dy)
    rows = kw * N                                       # output rows of the pair kernel, tiled in blocks of 256
    pair_ok = USE_WGRAD_PP and bool(lib.bm_tc_wgrad_conv_supported(T, M, N, kw)) and \
        rows / (-(-rows // 256) * 256) >= 0.9            # else the single-CTA kernel wastes less on padding rows
    if pair_ok:
        ws = _empty((int(lib.bm_tc_wgrad_conv_workspace(B, T, M, N, kw)),), dy)
        if USE_WGRAD_F16:
            dy_amax = tensor_amax(dy) if dy_amax is None else dy_amax
            x_amax = tensor_amax(x) if x_amax is None else x_amax
            call("bm_tc_wgrad_conv_f16", ptr(dy), ptr(dy_amax), ptr(x), ptr(x_amax), B, T, M, N, Ntrue, kw, dilation, ptr(ws),
                 ptr(dw), ptr(status), stream())
        else:
            call("bm_tc_wgrad_conv", ptr(dy), ptr(x), B, T, M, N, Ntrue, kw, dilation, ptr(ws), ptr(dw), ptr(status), stream())
        if dbias is not None:
            call("bm_col_sum", ptr(dy), B * T, M, ptr(dbias), stream())
        return dw
    ws = _empty((int(lib.bm_tc_wgrad_workspace(B, M, N, kw)),), dy)
    call("bm_tc_wgrad", ptr(dy), ptr(x), B, T, M, N, Ntrue, kw, dilation, ptr(ws), ptr(dw), ptr(dbias), ptr(status),
         stream())
    return dw


def group_layout(index: torch.Tensor, n_groups: int):
    """CSR grouping of the samples by `index` (values 0..n_groups-1): (order [B] int32, offsets [n_groups+1] int32), computed
    on the device WITHOUT a device->host synchronisation -- torch.bincount sizes its output from the data and stalls the host
    until everything queued before it has run (8.6 ms of a 17.6 ms step, measured with profiles/host_profile.py)."""
    order = torch.argsort(index, stable=True).to(torch.int32)
    groups = torch.arange(n_groups, device=index.device, dtype=index.dtype)
    counts = (index.reshape(-1, 1) == groups.reshape(1, -1)).sum(0)
    off = torch.zeros(n_groups + 1, dtype=torch.int32, device=index.device)
    off[1:] = torch.cumsum(counts, 0).to(torch.int32)
    return order, off


def tensor_amax(x: torch.Tensor) -> torch.Tensor:
    """max |x| as a device float [1] (bm_amax: one pass over x): the F16 pipe's per-tensor scale comes from it."""
    cell = _empty((1,), x)
    if x.data_ptr() % 16:                       # the kernel reads float4: a view at an odd offset goes through an aligned copy
        x = x.clone()
    call("bm_amax", ptr(x), x.numel(), ptr(cell), stream())
    return cell


def amax_cell(like: torch.Tensor) -> tp.Optional[torch.Tensor]:
    """A device float for a producer kernel to leave max |output| in (its `amax_out`), when the F16 pipe is in use."""
    return _empty((1,), like) if USE_CONV_F16 else None


class _Conv:
    """One conv layer's prepared operands + the kernel choice (tensor-core or FP32-FMA)."""

    def __init__(self, w: torch.Tensor, T: int, glu: bool, allow_tc: bool, pad_cin_to: int = 0, want_bwd=True):
        self.cout, self.cin_true, self.kw = w.shape
        self.glu = glu
        w = w.contiguous()
        if pad_cin_to and pad_cin_to != self.cin_true:
            wp = torch.zeros(self.cout, pad_cin_to, self.kw, device=w.device, dtype=w.dtype)
            wp[:, :self.cin_true] = w
            w = wp
        self.cin = w.shape[1]
        st = stream()
        lib = _lib.load()
        g = 1 if glu else 0
        # persistent CTA-pair kernel (csrc/tc_convp.cuh) where its tiling fits, else the single-CTA tensor-core kernel,
        # else FP32 FMA
        self.fwd_pp = allow_tc and USE_CONV_PP and bool(lib.bm_tc_conv1d_persistent_supported(T, self.cin, self.cout, self.kw, g))
        self.bwd_pp = allow_tc and USE_CONV_PP and bool(lib.bm_tc_conv1d_persistent_supported(T, self.cout, self.cin, self.kw, 0))
        fwd_tc = self.fwd_pp or (allow_tc and bool(lib.bm_tc_conv_supported(T, self.cin, self.cout, self.kw, g)))
        bwd_tc = self.bwd_pp or (allow_tc and bool(lib.bm_tc_conv_supported(T, self.cout, self.cin, self.kw, 0)))
        self.fwd_tc, self.bwd_tc = fwd_tc, bwd_tc
        self.wgrad_tc = allow_tc and bool(lib.bm_tc_wgrad_supported(self.cout, self.cin))
        self.f_hi = self.f_lo = self.g_hi = self.g_lo = self.wf = self.wb = None
        self.f_h16 = self.g_h16 = self.w_amax = None
        f16_f = USE_CONV_F16 and self.fwd_pp                      # operands of the F16-pipe kernel (tc_convh.cuh)
        f16_g = USE_CONV_F16 and self.bwd_pp and want_bwd
        if f16_f or f16_g:
            # fp16 hi/lo pieces of w * 2^k (k from the weights' largest magnitude), straight into the K-major layouts:
            # bm_amax + ONE re-layout-and-split launch per layer and step
            self.w_amax = _empty((1,), w)
            call("bm_amax", ptr(w), w.numel(), ptr(self.w_amax), st)
            half = dict(device=w.device, dtype=torch.float16)
            if f16_f:
                self.f_h16 = (torch.empty((self.kw, self.cout, self.cin), **half), torch.empty((self.kw, self.cout, self.cin), **half))
            if f16_g:
                self.g_h16 = (torch.empty((self.kw, self.cin, self.cout), **half), torch.empty((self.kw, self.cin, self.cout), **half))
            fh, fl = self.f_h16 if f16_f else (None, None)
            gh, gl = self.g_h16 if f16_g else (None, None)
            call("bm_tc_weight_split_f16", ptr(w), ptr(self.w_amax), self.cout, self.cin, self.kw, ptr(fh), ptr(fl), ptr(gh),
                 ptr(gl), st)
        need_f = fwd_tc and not f16_f                              # fp32 K-major operands for the TF32-pipe kernels
        need_g = bwd_tc and want_bwd and not f16_g
        if need_f or need_g:
            # RAW fp32 for the persistent kernel (it derives the tf32 lo part itself), a pre-split tf32 hi/lo pair for the
            # single-CTA kernel
            if need_f:
                self.f_hi = _empty((self.kw, self.cout, self.cin), w)
                self.f_lo = None if self.fwd_pp else _empty((self.kw, self.cout, self.cin), w)
            if need_g:
                self.g_hi = _empty((self.kw, self.cin, self.cout), w)
                self.g_lo = None if self.bwd_pp else _empty((self.kw, self.cin, self.cout), w)
            call("bm_tc_weight_split", ptr(w), self.cout, self.cin, self.kw, ptr(self.f_hi), ptr(self.f_lo),
                 ptr(self.g_hi), ptr(self.g_lo), st)
        if (not fwd_tc) or (want_bwd and not bwd_tc):
            self.wf = _empty((self.kw, self.cin, self.cout), w) if not fwd_tc else None
            self.wb = _empty((self.kw, self.cout, self.cin), w) if (want_bwd and not bwd_tc) else None
            call("bm_conv_weight_prep", ptr(w), self.cout, self.cin, self.kw, ptr(self.wf), ptr(self.wb), st)

    def run_tc(self, fwd: bool, x, bias, addend, B, T, dilation, glu, act, tmajor, y, aux, glu_out, stats, status,
               x_amax=None, out_amax=None):
        """One tensor-core conv launch: forward taps (fwd) or the data gradient; `addend` must be None or `y` itself
        (in-place accumulation) on the persistent kernel.  `x_amax` (F16 pipe): the device float holding max |x| when the
        producer of x already knows it, else one bm_amax pass here; `out_amax`: a device float that receives max |output| of a
        GLU / GELU epilogue for the conv that consumes it next (`amax_cell`)."""
        st = stream()
        if fwd:
            pp, hi, lo, cin, ntot, sign = self.fwd_pp, self.f_hi, self.f_lo, self.cin, self.cout, 1
        else:
            pp, hi, lo, cin, ntot, sign = self.bwd_pp, self.g_hi, self.g_lo, self.cout, self.cin, -1
        h16 = self.f_h16 if fwd else self.g_h16
        if pp and h16 is not None:
            assert addend is None or addend.data_ptr() == y.data_ptr(), "the persistent kernel accumulates in place only"
            if x_amax is None:
                x_amax = tensor_amax(x)
            call("bm_tc_conv1d_f16", ptr(x), ptr(x_amax), ptr(h16[0]), ptr(h16[1]), ptr(self.w_amax), ptr(bias),
                 0 if addend is None else 1, B, T, cin, ntot, self.kw, dilation, sign, glu, act, tmajor, ptr(y), ptr(aux),
                 ptr(glu_out), ptr(stats), ptr(out_amax), ptr(status), st)
            return out_amax
        elif pp:
            assert addend is None or addend.data_ptr() == y.data_ptr(), "the persistent kernel accumulates in place only"
            call("bm_tc_conv1d_persistent", ptr(x), ptr(hi), ptr(bias), 0 if addend is None else 1, B, T, cin, ntot,
                 self.kw, dilation, sign, glu, act, tmajor, ptr(y), ptr(aux), ptr(glu_out), ptr(stats), ptr(status), st)
        else:
            assert stats is None
            call("bm_tc_conv1d", ptr(x), ptr(hi), ptr(lo), ptr(bias), ptr(addend), B, T, cin, ntot, self.kw, dilation,
                 sign, glu, act, tmajor, ptr(y), ptr(aux), ptr(glu_out), None, ptr(status), st)
        return None                        # the tf32 kernels do not report max |output|

    # y = conv(x) (+bias); optionally BatchNorm statistics into `stats`
    def forward(self, x, bias, B, T, dilation, y, stats, status, x_amax=None):
        st = stream()
        if self.fwd_tc:
            fused = stats is not None and self.fwd_pp          # BatchNorm statistics out of the conv epilogue
            if self.cout > 320:
                fused = False                                   # the kernel keeps the statistics of ONE N tile in smem
            self.run_tc(True, x, bias, None, B, T, dilation, 0, 0, 0, y, None, None, stats if fused else None, status,
                        x_amax=x_amax)
            if stats is not None and not fused:
                call("bm_col_stats", ptr(y), B * T, self.cout, ptr(stats), st)
        else:
            call("bm_conv1d_fwd", ptr(x), ptr(self.wf), ptr(bias), B, T, self.cin, self.cout, self.kw, dilation,
                 ptr(y), ptr(stats), st)

    def forward_glu(self, x, bias, B, T, h, out, status, x_amax=None, out_amax=None):
        """-> the device float holding max |out| when the kernel produced it (F16 pipe), else None."""
        st = stream()
        if self.fwd_tc:
            return self.run_tc(True, x, bias, None, B, T, 1, 1, 0, 0, h, None, out, None, status, x_amax=x_amax,
                               out_amax=out_amax)
        else:
            call("bm_conv1d_glu_fwd", ptr(x), ptr(self.wf), ptr(bias), B, T, self.cin, self.cout // 2, self.kw,
                 ptr(h), ptr(out), st)

    def backward_data(self, dy, addend, B, T, dilation, dx, status, dy_amax=None):
        st = stream()
        if self.bwd_tc:
            self.run_tc(False, dy, None, addend, B, T, dilation, 0, 0, 0, dx, None, None, None, status, x_amax=dy_amax)
        else:
            call("bm_conv1d_bwd_data", ptr(dy), ptr(self.wb), ptr(addend), B, T, self.cin, self.cout, self.kw,
                 dilation, ptr(dx), st)

    def backward_weight(self, dy, x, B, T, dilation, like, status, bias_grad_is_zero=False, known_dbias=None, dy_amax=None,
                        x_amax=None):
        """`bias_grad_is_zero`: the conv feeds a training-mode BatchNorm, whose backward makes sum(dy) == 0 exactly
        (the reference's value there is rounding noise around 0); skip the reduction.  `known_dbias`: the producer of dy
        already summed it over the rows.  `dy_amax` / `x_amax`: see tc_wgrad."""
        if self.wgrad_tc:
            am = dict(dy_amax=dy_amax, x_amax=x_amax)
            if known_dbias is not None:
                return tc_wgrad(dy, x, B, T, self.cout, self.cin, self.cin_true, self.kw, dilation, status, **am), known_dbias
            if bias_grad_is_zero:
                dw = tc_wgrad(dy, x, B, T, self.cout, self.cin, self.cin_true, self.kw, dilation, status, **am)
                return dw, torch.zeros((self.cout,), device=like.device)
            db = _empty((self.cout,), like)
            dw = tc_wgrad(dy, x, B, T, self.cout, self.cin, self.cin_true, self.kw, dilation, status, dbias=db, **am)
            return dw, db
        db = _empty((self.cout,), like)
        dw = _empty((self.cout, self.cin, self.kw), like)
        call("bm_conv1d_bwd_weight", ptr(dy), ptr(x), B, T, self.cin, self.cout, self.kw, dilation, ptr(dw), ptr(db),
             stream())
        if self.cin != self.cin_true:
            dw = dw[:, :self.cin_true].contiguous()
        return dw, db


# ----------------------------------------------------------------------------------------------------
# Sensor chain in optional stages: the ablation rows merger=False / initial_linear=0 / subject_layers=False / subject_dim
# (grids/nmi/ablation_final.py:44,46,50,51; simpleconv.py:104-151, 207-233).  Each stage is the FP32-FMA stage kernel that
# the fused `bm_sensor_chain_fwd/bwd` is made of (csrc/bm_api.cu), called on its own; activations are channels-last.
# ----------------------------------------------------------------------------------------------------
def _staged_front_forward(plan: "EncoderPlan", meg, heads, il_w, il_b, subj_w, sub_emb, status):
    """-> (x [B,T,D_total] channels-last, saved dict).  meg [B,C,T]; missing stages have None parameters."""
    st = stream()
    B, C, T = meg.shape
    R = plan.rec_positions.shape[0]
    saved = dict(meg=meg, att=None, emb=None, u=None, v=None)
    width = C
    if heads is not None:                                     # ChannelMerger (common.py:334-362)
        O, P = heads.shape
        emb = _empty((R, C, P), meg)
        att = _empty((R, O, C), meg)
        call("bm_attention_weights_fwd", ptr(plan.rec_positions), ptr(plan.freq), ptr(heads.contiguous()),
             ptr(plan.ban_centre), float(plan.ban_radius), R, C, O, P, ptr(emb), ptr(att), st)
        u = _empty((B, T, O), meg)
        call("bm_sensor_mix_fwd", ptr(meg), ptr(att), ptr(plan.rec_of_sample), B, C, T, O, O, ptr(u), st)
        saved.update(att=att, emb=emb)
        width = O
    else:                                                      # raw sensors, channels-last
        u = _empty((B, T, C), meg)
        call("bm_transpose_nt", ptr(meg), B, C, T, ptr(u), st)
    saved["u"] = u
    x = u
    if il_w is not None:                                       # initial_linear (simpleconv.py:112-120)
        IL = il_w.shape[0]
        v = _empty((B, T, IL), meg)
        call("bm_initial_linear_fwd", ptr(x), width, ptr(il_w.reshape(IL, width).contiguous()), ptr(il_b.contiguous()), B, T,
             width, IL, IL, ptr(v), st)
        x, width = v, IL
    saved["v"] = x                                             # input of the subject stage
    if subj_w is not None:                                     # SubjectLayers (common.py:45-62)
        D = subj_w.shape[2]
        x0 = _empty((B, T, D), meg)
        call("bm_subject_layers_fwd", ptr(x), width, ptr(subj_w.contiguous()), ptr(plan.subject), B, T, width, D, D,
             ptr(x0), st)
        x, width = x0, D
    if sub_emb is not None:                                    # ScaledEmbedding appended as channels (simpleconv.py:231-233)
        x = torch.cat([x, sub_emb[:, None, :].expand(B, T, sub_emb.shape[1])], dim=2).contiguous()
    saved["widths"] = (C, saved["u"].shape[2], saved["v"].shape[2], width)
    return x, saved


def _staged_front_backward(plan: "EncoderPlan", saved, g, heads, il_w, subj_w, sub_emb):
    """g = dL/dx [B,T,D_total] -> (dheads, d_il_w, d_il_b, d_subj, d_sub_emb); None where the stage is absent."""
    st = stream()
    meg = saved["meg"]
    B, C, T = meg.shape
    R = plan.rec_positions.shape[0]
    _, w_u, w_v, w_x = saved["widths"]
    d_sub_emb = None
    if sub_emb is not None:
        d_sub_emb = g[:, :, w_x:].sum(dim=1)                   # the embedding is constant over time
        g = g[:, :, :w_x].contiguous()
    d_subj = None
    if subj_w is not None:
        S = subj_w.shape[0]
        subj_order, subj_off = group_layout(plan.subject, S)
        d_subj = _empty((S, w_v, w_x), meg)
        dv = _empty((B, T, w_v), meg)
        call("bm_subject_layers_bwd", ptr(g), w_x, ptr(saved["v"]), w_v, ptr(subj_w.contiguous()), ptr(plan.subject),
             ptr(subj_order), ptr(subj_off), B, T, w_v, w_x, S, w_v, ptr(dv), ptr(d_subj), st)
        g = dv
    d_il_w = d_il_b = None
    if il_w is not None:
        d_il_w = _empty((w_v, w_u), meg)
        d_il_b = _empty((w_v,), meg)
        du = _empty((B, T, w_u), meg)
        call("bm_initial_linear_bwd", ptr(g), w_v, ptr(saved["u"]), w_u, ptr(il_w.reshape(w_v, w_u).contiguous()), B, T, w_u,
             w_v, w_u, ptr(du), ptr(d_il_w), ptr(d_il_b), st)
        d_il_w = d_il_w.reshape(il_w.shape)
        g = du
    dheads = None
    if heads is not None:
        O, P = heads.shape
        d_att = _empty((R, O, C), meg)
        call("bm_sensor_mix_bwd", ptr(g), w_u, ptr(meg), ptr(plan.rec_order), ptr(plan.rec_off), B, C, T, O, R, ptr(d_att), st)
        dscores = _empty((R, O, C), meg)
        dheads = _empty((O, P), meg)
        call("bm_attention_weights_bwd", ptr(d_att), ptr(saved["att"]), ptr(saved["emb"]), R, C, O, P, ptr(dscores),
             ptr(dheads), st)
    return dheads, d_il_w, d_il_b, d_subj, d_sub_emb


class _EncoderFn(torch.autograd.Function):
    """inputs: plan, meg, heads, il_w, il_b, subj_w, w0, b0, w2, b2, then per layer k: (conv_w, conv_b, gamma, beta)
    and, appended in layer order, (glu_w, glu_b) for every layer followed by a GLU block."""

    @staticmethod
    def forward(ctx, plan: EncoderPlan, meg, heads, il_w, il_b, subj_w, w0, b0, w2, b2, *layer_params):
        depth = len(plan.dilations)
        sub_emb = None
        if plan.has_sub_emb:                     # [B, E] rows of the (scaled) subject embedding, appended by the caller
            sub_emb, layer_params = layer_params[-1], layer_params[:-1]
        conv_p = [layer_params[4 * k:4 * k + 4] for k in range(depth)]
        glu_flat = layer_params[4 * depth:]
        glu_p, gi = {}, 0
        for k in range(depth):
            if plan.glu_after[k]:
                glu_p[k] = glu_flat[2 * gi:2 * gi + 2]
                gi += 1
        st = stream()
        meg = meg.contiguous()
        B, C, T = meg.shape
        R = plan.rec_positions.shape[0]
        O, P = heads.shape if heads is not None else (0, 0)
        IL = il_w.shape[0] if il_w is not None else 0
        S, _, D = subj_w.shape if subj_w is not None else (0, 0, 0)
        H = conv_p[0][0].shape[0]
        F = conv_p[-1][0].shape[0] if plan.bare_last else w2.shape[1]
        rows = B * T
        save = plan.keep_for_backward
        tc = plan.use_tensor_cores
        status = tc_status_tensor(meg.device)

        if plan.staged:
            # sensor-side ablation rows: the chain as optional stages (see _staged_front_forward)
            x, front = _staged_front_forward(plan, meg, heads, il_w, il_b, subj_w, sub_emb, status)
            D = Dp = x.shape[2]
            conv0 = _Conv(conv_p[0][0], T, False, tc, want_bwd=save)
            emb = att = u = v = il_w2 = il_conv = subj_pad = megT = heads_conv = None
            Op = ILp = 0
        else:
            front = None
            # K1 attention weights per recording (the score contraction on the tensor cores when the widths fit)
            emb = _empty((R, C, P), meg)
            lib = _lib.load()
            Opad = _round_up(O, 64)
            heads_conv = None
            if tc and bool(lib.bm_tc_conv1d_persistent_supported(C, P, Opad, 1, 0)) and bool(lib.bm_tc_wgrad_supported(Opad, P)):
                hpad = torch.zeros((Opad, P, 1), device=meg.device)
                hpad[:O, :, 0] = heads
                heads_conv = _Conv(hpad, C, False, True, want_bwd=False)
                if not heads_conv.fwd_pp:
                    heads_conv = None
            if heads_conv is not None:
                call("bm_fourier_emb", ptr(plan.rec_positions), ptr(plan.freq), R, C, P, ptr(emb), st)
                att_full = _empty((R, Opad, C), meg)          # scores[r][o][c] = <emb[r][c], heads[o]> written channel-major
                heads_conv.run_tc(True, emb, None, None, R, C, 1, 0, 0, 1, att_full, None, None, None, status)
                call("bm_masked_softmax", ptr(att_full), ptr(plan.rec_positions), ptr(plan.ban_centre), float(plan.ban_radius),
                     R, Opad, C, st)
                att = att_full[:, :O].contiguous()
            else:
                att = _empty((R, O, C), meg)
                call("bm_attention_weights_fwd", ptr(plan.rec_positions), ptr(plan.freq), ptr(heads.contiguous()),
                     ptr(plan.ban_centre), float(plan.ban_radius), R, C, O, P, ptr(emb), ptr(att), st)
            # K2 sensor chain; x0 is kept zero-padded to a multiple of 64 channels when the tensor-core conv follows
            Dp = _round_up(D, 64)
            conv0 = _Conv(conv_p[0][0], T, False, tc, pad_cin_to=Dp, want_bwd=save)
            if not conv0.fwd_tc:
                Dp = D
                conv0 = _Conv(conv_p[0][0], T, False, False, want_bwd=save)
            il_w2 = il_w.reshape(IL, O).contiguous()
            # `initial_linear` on the tensor cores when the (64-padded) widths fit: u and v are then kept zero-padded
            Op, ILp = _round_up(O, 64), _round_up(IL, 64)
            il_conv = None
            if tc:
                wpad = torch.zeros((ILp, Op, 1), device=meg.device)
                wpad[:IL, :O, 0] = il_w2
                il_conv = _Conv(wpad, T, False, True, want_bwd=save)
                if not (il_conv.fwd_tc and il_conv.bwd_tc and il_conv.wgrad_tc):
                    il_conv = None
            # u [B,T,Op] and x [B,T,Dp] carry zero pad columns.  The tensor-core contractions write every column (their padded
            # weight rows are zero), so the buffers only need a fill when an FP32-FMA stage kernel (valid columns only) runs.
            def _padded(width_pad, width, written_in_full):
                if width_pad == width or written_in_full:
                    return _empty((B, T, width_pad), meg)
                return torch.zeros((B, T, width_pad), device=meg.device)

            lib = _lib.load()
            Cp = _round_up(C, 128)
            mix_tc = il_conv is not None and bool(lib.bm_tc_conv_supported(T, Cp, Op, 1, 0)) and \
                bool(lib.bm_tc_wgrad_supported(Op, Cp))
            subj_tc = il_conv is not None and (Dp != D or D % 64 == 0) and bool(lib.bm_tc_conv_supported(T, ILp, Dp, 1, 0)) and \
                bool(lib.bm_tc_conv_supported(T, Dp, ILp, 1, 0)) and bool(lib.bm_tc_wgrad_supported(ILp, Dp))
            x = _padded(Dp, D, subj_tc)
            if il_conv is not None:
                u = _padded(Op, O, mix_tc)
                v = _empty((B, T, ILp), meg)
                bpad = torch.zeros((ILp,), device=meg.device)
                bpad[:IL] = il_b
                # sensor mix on the tensor cores: meg transposed once to channels-last (sensor count padded to 128), then
                # u = megT @ w[rec]^T is a pointwise contraction with a per-sample weight set (one per recording)
                megT = None
                if mix_tc:
                    megT = _empty((B, T, Cp), meg)                 # the transpose writes the pad columns as zeros
                    call("bm_transpose_nt_ld", ptr(meg), B, C, T, Cp, ptr(megT), st)
                    att_pad = torch.zeros((R, Op, Cp), device=meg.device)
                    att_pad[:, :O, :C] = att
                    aw_hi, aw_lo = _empty((R * Op, Cp), meg), _empty((R * Op, Cp), meg)
                    call("bm_tc_weight_split", ptr(att_pad), R * Op, Cp, 1, ptr(aw_hi), ptr(aw_lo), None, None, st)
                    call("bm_tc_pointwise_sel", ptr(megT), ptr(aw_hi), ptr(aw_lo), ptr(plan.rec_of_sample), R, B, T, Cp, Op,
                         ptr(u), ptr(status), st)
                else:
                    call("bm_sensor_mix_fwd", ptr(meg), ptr(att), ptr(plan.rec_of_sample), B, C, T, O, Op, ptr(u), st)
                il_conv.forward(u, bpad, B, T, 1, v, None, status)
                if subj_tc:
                    # per-subject weights, zero-padded; forward operand [s][d][p] (K-major in p), tf32-split
                    subj_pad = torch.zeros((S, ILp, Dp), device=meg.device)
                    subj_pad[:, :IL, :D] = subj_w
                    mt = subj_pad.transpose(1, 2).contiguous()
                    sf_hi, sf_lo = _empty((S * Dp, ILp), meg), _empty((S * Dp, ILp), meg)
                    call("bm_tc_weight_split", ptr(mt), S * Dp, ILp, 1, ptr(sf_hi), ptr(sf_lo), None, None, st)
                    call("bm_tc_pointwise_sel", ptr(v), ptr(sf_hi), ptr(sf_lo), ptr(plan.subject), S, B, T, ILp, Dp, ptr(x),
                         ptr(status), st)
                else:
                    subj_pad = None
                    call("bm_subject_layers_fwd", ptr(v), ILp, ptr(subj_w.contiguous()), ptr(plan.subject), B, T, IL, D, Dp,
                         ptr(x), st)
            else:
                subj_pad = None
                megT = None
                Op, ILp = O, IL
                u = _empty((B, T, O), meg)
                v = _empty((B, T, IL), meg)
                call("bm_sensor_chain_fwd", ptr(meg), ptr(att), ptr(plan.rec_of_sample), ptr(il_w2),
                     ptr(il_b.contiguous()), ptr(subj_w.contiguous()), ptr(plan.subject), B, C, T, O, IL, D, Dp, ptr(u),
                     ptr(v), ptr(x), st)

        # K3/K4 ConvSequence
        stats = _empty((2 * H,), meg, torch.float64)
        saved_layers = []
        x_amax = None                                   # device float with max |x| when x's producer reported it (F16 pipe)
        for k in range(depth):
            cw, cb, gamma, beta = conv_p[k]
            conv = conv0 if k == 0 else _Conv(cw, T, False, tc, want_bwd=save)
            cout = conv.cout
            y = _empty((B, T, cout), meg)
            if plan.bare_last and k == depth - 1:
                conv.forward(x, cb.contiguous(), B, T, plan.dilations[k], y, None, status, x_amax=x_amax)
                x_amax = None
                skip = plan.skip and conv.cin_true == cout
                x_new = y
                if skip:
                    x_new = _empty((B, T, cout), meg)
                    call("bm_bn_act_skip_fwd", ptr(y), None, None, None, None, ptr(x), ptr(x_new), rows, cout, 2, 0.0, st)
                rec = dict(x_in=x, y=y, mean=None, invstd=None, conv=conv, skip=skip, x_new=x_new, bare=True)
                x = x_new
                if plan.glu_after[k]:
                    gw, gb = glu_p[k]
                    gconv = _Conv(gw, T, True, tc, want_bwd=save)
                    h = _empty((B, T, gconv.cout), meg) if save else None
                    out = _empty((B, T, gconv.cout // 2), meg)
                    x_amax = gconv.forward_glu(x, gb.contiguous(), B, T, h, out, status, x_amax=x_amax, out_amax=amax_cell(meg))
                    rec.update(h=h, gconv=gconv)
                    x = out
                saved_layers.append(rec if save else None)
                continue
            mean = _empty((cout,), meg)
            invstd = _empty((cout,), meg)
            rm, rv = plan.bn_buffers[k]
            if plan.training:
                conv.forward(x, cb.contiguous(), B, T, plan.dilations[k], y, stats, status, x_amax=x_amax)
                call("bm_bn_stats_finalize", ptr(stats), rows, float(plan.bn_eps), float(plan.bn_momentum),
                     ptr(rm), ptr(rv), ptr(mean), ptr(invstd), cout, st)
            else:
                conv.forward(x, cb.contiguous(), B, T, plan.dilations[k], y, None, status, x_amax=x_amax)
                call("bm_bn_eval_stats", ptr(rm), ptr(rv), float(plan.bn_eps), ptr(mean), ptr(invstd), cout, st)
            skip = plan.skip and conv.cin_true == cout
            x_new = _empty((B, T, cout), meg)
            x_in_amax, x_amax = x_amax, None
            if plan.act_code == 0:
                x_amax = amax_cell(meg)
                call("bm_bn_gelu_skip_fwd", ptr(y), ptr(mean), ptr(invstd), ptr(gamma.contiguous()),
                     ptr(beta.contiguous()), ptr(x) if skip else None, ptr(x_new), rows, cout, ptr(x_amax), st)
            else:
                call("bm_bn_act_skip_fwd", ptr(y), ptr(mean), ptr(invstd), ptr(gamma.contiguous()),
                     ptr(beta.contiguous()), ptr(x) if skip else None, ptr(x_new), rows, cout, plan.act_code,
                     float(plan.act_slope), st)
            rec = dict(x_in=x, y=y, mean=mean, invstd=invstd, conv=conv, skip=skip, x_new=x_new, x_in_amax=x_in_amax,
                       x_new_amax=x_amax)
            x = x_new
            if plan.glu_after[k]:
                gw, gb = glu_p[k]
                gconv = _Conv(gw, T, True, tc, want_bwd=save)
                h = _empty((B, T, gconv.cout), meg) if save else None
                out = _empty((B, T, gconv.cout // 2), meg)
                x_amax = gconv.forward_glu(x, gb.contiguous(), B, T, h, out, status, x_amax=x_amax, out_amax=amax_cell(meg))
                rec.update(h=h, gconv=gconv)
                x = out
            saved_layers.append(rec if save else None)

        if plan.bare_last:
            # no head: the sequence already ends on out_channels; hand it out channel-major
            est = _empty((B, F, T), meg)
            call("bm_transpose_nt", ptr(x), B, T, F, ptr(est), st)
            if save:
                ctx.plan = plan
                ctx.dims = (B, C, T, R, O, P, IL, S, D, Dp, H, F)
                ctx.pads = (Op, ILp)
                ctx.saved = dict(meg=meg, emb=emb, att=att, u=u, v=v, il_w2=il_w2, subj_w=None if subj_w is None else subj_w.contiguous(),
                                 il_conv=il_conv, subj_pad=subj_pad, megT=megT, heads_tc=heads_conv is not None,
                                 layers=saved_layers, conv_p=conv_p, glu_p=glu_p,
                                 il_shape=None if il_w is None else il_w.shape, front=front,
                                 params=(heads, il_w, subj_w, sub_emb))
            return est

        # K5 head
        H2 = 2 * H
        head0 = _Conv(w0, T, False, tc, want_bwd=save)                       # [2H, H, 1]
        w2_as_conv = w2.permute(1, 0, 2).contiguous()                        # ConvTranspose1d [2H,F,1] -> [F,2H,1]
        head2 = _Conv(w2_as_conv, T, False, tc, want_bwd=save)
        head_tc = head0.fwd_tc and head2.fwd_tc and head0.bwd_tc and head2.bwd_tc
        h1 = _empty((B, T, H2), meg)
        q = _empty((B, T, H2), meg)
        est = _empty((B, F, T), meg)
        w0_2 = w0.reshape(H2, H).contiguous()
        w2_2 = w2.reshape(H2, F).contiguous()
        head_generic = plan.act_code != 0
        q_amax = None
        if head_generic:
            # simpleconv.gelu=False (simpleconv.py:85-90,187): conv -> activation kernel -> conv, channels-last, then one
            # transpose to the channel-major estimate (the fused GELU epilogues below do not apply)
            head_tc = False
            head0.forward(x, b0.contiguous(), B, T, 1, h1, None, status)
            call("bm_bn_act_skip_fwd", ptr(h1), None, None, None, None, None, ptr(q), rows, H2, plan.act_code,
                 float(plan.act_slope), st)
            est_cl = _empty((B, T, F), meg)
            head2.forward(q, b2.contiguous(), B, T, 1, est_cl, None, status)
            call("bm_transpose_nt", ptr(est_cl), B, T, F, ptr(est), st)
            del est_cl
        elif head_tc:
            q_amax = head0.run_tc(True, x, b0.contiguous(), None, B, T, 1, 0, 1, 0, q, h1 if save else None, None, None, status,
                                  x_amax=x_amax, out_amax=amax_cell(meg))
            head2.run_tc(True, q, b2.contiguous(), None, B, T, 1, 0, 0, 1, est, None, None, None, status, x_amax=q_amax)
        else:
            call("bm_head_fwd", ptr(x), ptr(w0_2), ptr(b0.contiguous()), ptr(w2_2), ptr(b2.contiguous()), B, T, H, F,
                 ptr(h1), ptr(q), ptr(est), st)

        if save:
            ctx.plan = plan
            ctx.dims = (B, C, T, R, O, P, IL, S, D, Dp, H, F)
            ctx.pads = (Op, ILp)
            ctx.saved = dict(meg=meg, emb=emb, att=att, u=u, v=v, il_w2=il_w2, subj_w=None if subj_w is None else subj_w.contiguous(), il_conv=il_conv,
                             subj_pad=subj_pad, megT=megT, heads_tc=heads_conv is not None,
                             layers=saved_layers, x_last=x, w0_2=w0_2, w2_2=w2_2, h1=h1, q=q, q_amax=q_amax,
                             head0=head0, head2=head2, head_tc=head_tc, head_generic=head_generic,
                             conv_p=conv_p, glu_p=glu_p, il_shape=None if il_w is None else il_w.shape,
                             w0_shape=w0.shape, w2_shape=w2.shape, front=front, params=(heads, il_w, subj_w, sub_emb))
        return est

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dest):
        plan: EncoderPlan = ctx.plan
        s = ctx.saved
        if s is None:
            raise RuntimeError("brainmagick_b200.SimpleConv: backward through the graph a second time -- the saved activations "
                               "(~5 GB at B=256) are released by the first backward; retain_graph is not supported")
        B, C, T, R, O, P, IL, S, D, Dp, H, F = ctx.dims
        depth = len(plan.dilations)
        st = stream()
        meg = s["meg"]
        rows = B * T
        H2 = 2 * H
        dest = dest.contiguous()
        status = tc_status_tensor(meg.device)

        ctx_keep: tp.List[tp.Any] = []          # operands of side-stream kernels, released after the streams join
        # ---- head ----
        if plan.bare_last:
            g = _empty((B, T, F), meg)           # no head: the gradient of the estimate IS the sequence's output gradient
            call("bm_transpose_nt", ptr(dest), B, F, T, ptr(g), st)
            dw0 = db0 = dw2 = db2 = dq = None
        else:
            g = _empty((B, T, H), meg)
            dw0 = _empty((H2, H), meg)
            db0 = _empty((H2,), meg)
            dw2 = _empty((H2, F), meg)
            db2 = _empty((F,), meg)
            dq = _empty((B, T, H2), meg)
        if plan.bare_last:
            pass
        elif s["head_generic"]:
            head0, head2 = s["head0"], s["head2"]
            dest_t = _empty((B, T, F), meg)
            call("bm_transpose_nt", ptr(dest), B, F, T, ptr(dest_t), st)
            head2.backward_data(dest_t, None, B, T, 1, dq, status)                 # dq = dest_t @ w2^T
            dw2c, db2 = head2.backward_weight(dest_t, s["q"], B, T, 1, meg, status)    # [F, 2H, 1]
            dw2 = dw2c.permute(1, 0, 2).reshape(H2, F).contiguous()
            dh1 = _empty((B, T, H2), meg)
            call("bm_bn_act_skip_bwd", ptr(dq), ptr(s["h1"]), None, None, None, None, 0, rows, H2, plan.act_code,
                 float(plan.act_slope), None, ptr(dh1), None, None, st)
            dw0, db0 = head0.backward_weight(dh1, s["x_last"], B, T, 1, meg, status)   # [2H, H, 1]
            head0.backward_data(dh1, None, B, T, 1, g, status)
            del dest_t, dh1
        elif s["head_tc"]:
            head0, head2 = s["head0"], s["head2"]
            dest_t = _empty((B, T, F), meg)
            call("bm_transpose_nt", ptr(dest), B, F, T, ptr(dest_t), st)
            # dq = dest_t @ w2^T  (w2_as_conv [F,2H,1]: its data-gradient operand is [1][2H][F])
            dest_amax = tensor_amax(dest_t) if USE_CONV_F16 else None      # one pass serves the dgrad and the wgrad below
            head2.run_tc(False, dest_t, None, None, B, T, 1, 0, 0, 0, dq, None, None, None, status, x_amax=dest_amax)
            lib = _lib.load()
            if lib.bm_tc_wgrad_supported(H2, F) and lib.bm_tc_wgrad_supported(H2, H):
                main0 = torch.cuda.current_stream()
                side0 = _side_stream(meg.device) if OVERLAP_WGRAD else None

                def on_side(fn, *tensors):
                    """runs fn() on the side stream after everything queued so far on the main stream"""
                    if side0 is None:
                        return fn()
                    side0.wait_stream(main0)
                    with torch.cuda.stream(side0):
                        out = fn()
                    ctx_keep.append(tensors)
                    out.record_stream(main0)
                    return out

                # dW2 / db2 only need dest_t and q: they overlap the dq contraction queued just before
                dw2 = on_side(lambda: tc_wgrad(s["q"], dest_t, B, T, H2, F, F, 1, 1, status, dy_amax=s.get("q_amax"),
                                               x_amax=dest_amax), s["q"], dest_t, dest_amax).reshape(H2, F)
                call("bm_col_sum", ptr(dest_t), rows, F, ptr(db2), st)
                call("bm_gelu_bwd", ptr(dq), ptr(s["h1"]), rows * H2, ptr(dq), st)           # dq <- dh1
                dw0 = on_side(lambda: tc_wgrad(dq, s["x_last"], B, T, H2, H, H, 1, 1, status, dbias=db0), dq,
                              s["x_last"], db0).reshape(H2, H)
            else:
                call("bm_head_bwd_params", ptr(dest), ptr(s["x_last"]), ptr(s["h1"]), ptr(s["q"]), B, T, H, F,
                     ptr(dq), ptr(dw0), ptr(db0), ptr(dw2), ptr(db2), st)   # dq <- dq*GELU'(h1); dW0, db0, dW2, db2
            head0.run_tc(False, dq, None, None, B, T, 1, 0, 0, 0, g, None, None, None, status)
            del dest_t
        else:
            call("bm_head_bwd", ptr(dest), ptr(s["x_last"]), ptr(s["w0_2"]), ptr(s["w2_2"]), ptr(s["h1"]), ptr(s["q"]),
                 B, T, H, F, ptr(dq), ptr(g), ptr(dw0), ptr(db0), ptr(dw2), ptr(db2), st)
        del dq

        sums = _empty((2 * H,), meg, torch.float64)
        layer_grads: tp.List[tp.Any] = [None] * depth
        glu_grads = {}
        # The weight gradient and the data gradient of a layer are independent given dy: the weight-gradient kernels go to
        # a side stream so that their CTAs fill the SMs left idle by the partial last wave of the data-gradient kernel.
        main = torch.cuda.current_stream()
        side = _side_stream(meg.device) if (OVERLAP_WGRAD and plan.use_tensor_cores) else None
        keep_alive: tp.List[tp.Any] = ctx_keep

        def weight_grad(conv_obj, dy_t, x_t, dil, bias_zero, known_dbias=None, dy_amax=None, x_amax=None):
            if side is None:
                return conv_obj.backward_weight(dy_t, x_t, B, T, dil, meg, status, bias_grad_is_zero=bias_zero,
                                                known_dbias=known_dbias, dy_amax=dy_amax, x_amax=x_amax)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                out = conv_obj.backward_weight(dy_t, x_t, B, T, dil, meg, status, bias_grad_is_zero=bias_zero,
                                               known_dbias=known_dbias, dy_amax=dy_amax, x_amax=x_amax)
            # the big operands are kept alive until the streams join (no record_stream: with the host running steps ahead
            # it would block the allocator from reusing ~3 GB of blocks and force cudaMallocs in the timed loop)
            keep_alive.append((dy_t, x_t, dy_amax, x_amax))
            for o in out:
                o.record_stream(main)
            return out

        for k in reversed(range(depth)):
            rec = s["layers"][k]
            cw, cb, gamma, beta = s["conv_p"][k]
            conv: _Conv = rec["conv"]
            cout = conv.cout
            if plan.glu_after[k]:
                gconv: _Conv = rec["gconv"]
                dh = _empty((B, T, gconv.cout), meg)
                dgb = _empty((gconv.cout,), meg)          # the GLU conv's bias gradient, summed while dh is produced
                dh_amax = amax_cell(meg)
                call("bm_glu_bwd", ptr(g), ptr(rec["h"]), rows, gconv.cout // 2, ptr(dh), ptr(dgb), ptr(dh_amax), st)
                glu_grads[k] = weight_grad(gconv, dh, rec["x_new"], 1, False, dgb, dy_amax=dh_amax, x_amax=rec.get("x_new_amax"))
                g = _empty((B, T, gconv.cin), meg)
                gconv.backward_data(dh, None, B, T, 1, g, status, dy_amax=dh_amax)
                del dh
            if rec.get("bare"):
                # bare convolution (+ residual): dL/dy = dL/dx_new; no BatchNorm behind it, so the bias gradient is real
                dy = g.clone() if rec["skip"] else g
                dcw, dcb = weight_grad(conv, dy, rec["x_in"], plan.dilations[k], False)
                if rec["skip"]:
                    conv.backward_data(dy, g, B, T, plan.dilations[k], g, status)
                else:
                    g_in = _empty((B, T, conv.cin), meg)
                    conv.backward_data(dy, None, B, T, plan.dilations[k], g_in, status)
                    g = g_in
                layer_grads[k] = (dcw, dcb, None, None)
                del dy
                continue
            dy = _empty((B, T, cout), meg)
            dgamma = _empty((cout,), meg)
            dbeta = _empty((cout,), meg)
            dy_amax = None
            if plan.act_code == 0:
                dy_amax = amax_cell(meg)
                call("bm_bn_gelu_skip_bwd", ptr(g), ptr(rec["y"]), ptr(rec["mean"]), ptr(rec["invstd"]),
                     ptr(gamma.contiguous()), ptr(beta.contiguous()), 1 if plan.training else 0, rows, cout, ptr(sums),
                     ptr(dy), ptr(dgamma), ptr(dbeta), ptr(dy_amax), st)
            else:
                call("bm_bn_act_skip_bwd", ptr(g), ptr(rec["y"]), ptr(rec["mean"]), ptr(rec["invstd"]),
                     ptr(gamma.contiguous()), ptr(beta.contiguous()), 1 if plan.training else 0, rows, cout,
                     plan.act_code, float(plan.act_slope), ptr(sums), ptr(dy), ptr(dgamma), ptr(dbeta), st)
            dcw, dcb = weight_grad(conv, dy, rec["x_in"], plan.dilations[k], plan.training, dy_amax=dy_amax,
                                   x_amax=rec.get("x_in_amax"))
            if rec["skip"]:
                # in place: g += conv_transpose(dy) (addend == output: the pair kernel turns this into a TMA reduce-add)
                conv.backward_data(dy, g, B, T, plan.dilations[k], g, status, dy_amax=dy_amax)
            else:
                g_in = _empty((B, T, conv.cin), meg)
                conv.backward_data(dy, None, B, T, plan.dilations[k], g_in, status, dy_amax=dy_amax)
                g = g_in
            layer_grads[k] = (dcw, dcb, dgamma, dbeta)
            del dy

        if side is not None:
            main.wait_stream(side)
        keep_alive.clear()
        if plan.staged:
            heads_p, il_w_p, subj_w_p, sub_emb_p = s["params"]
            dheads, d_il_w, d_il_b, d_subj, d_sub_emb = _staged_front_backward(plan, s["front"], g, heads_p, il_w_p,
                                                                               subj_w_p, sub_emb_p)
        else:
            d_sub_emb = None
            # ---- sensor chain + attention ----
            subj_order, subj_off = group_layout(plan.subject, S)
            Op, ILp = ctx.pads
            d_subj = _empty((S, IL, D), meg)
            d_att = _empty((R, O, C), meg)
            il_conv = s["il_conv"]
            if il_conv is not None:
                if s["subj_pad"] is not None:
                    subj_pad = s["subj_pad"]                                   # [S][ILp][Dp]: data-gradient operand as is
                    sb_hi, sb_lo = _empty((S * ILp, Dp), meg), _empty((S * ILp, Dp), meg)
                    call("bm_tc_weight_split", ptr(subj_pad), S * ILp, Dp, 1, ptr(sb_hi), ptr(sb_lo), None, None, st)
                    dv = _empty((B, T, ILp), meg)
                    call("bm_tc_pointwise_sel", ptr(g), ptr(sb_hi), ptr(sb_lo), ptr(plan.subject), S, B, T, Dp, ILp, ptr(dv),
                         ptr(status), st)
                    mpad = _round_up(ILp, 128)
                    dm = _empty((S, mpad, Dp), meg)
                    call("bm_tc_wgrad_grouped", ptr(s["v"]), ptr(g), ptr(subj_order), ptr(subj_off), S, B, T, ILp, Dp,
                         ptr(dm), ptr(status), st)
                    d_subj = dm[:, :IL, :D].contiguous()
                else:
                    dv = torch.zeros((B, T, ILp), device=meg.device) if ILp != IL else _empty((B, T, IL), meg)
                    call("bm_subject_layers_bwd", ptr(g), Dp, ptr(s["v"]), ILp, ptr(s["subj_w"]), ptr(plan.subject),
                         ptr(subj_order), ptr(subj_off), B, T, IL, D, S, ILp, ptr(dv), ptr(d_subj), st)
                du = _empty((B, T, Op), meg)
                il_conv.backward_data(dv, None, B, T, 1, du, status)
                dbp = _empty((ILp,), meg)
                d_il_w = tc_wgrad(dv, s["u"], B, T, ILp, Op, O, 1, 1, status, dbias=dbp)[:IL, :, 0].contiguous()
                d_il_b = dbp[:IL].contiguous()
                if s["megT"] is not None:
                    megT = s["megT"]
                    Cp = megT.shape[2]
                    dwp = _empty((R, _round_up(Op, 128), Cp), meg)
                    call("bm_tc_wgrad_grouped", ptr(du), ptr(megT), ptr(plan.rec_order), ptr(plan.rec_off), R, B, T, Op, Cp,
                         ptr(dwp), ptr(status), st)
                    d_att = dwp[:, :O, :C].contiguous()
                else:
                    call("bm_sensor_mix_bwd", ptr(du), Op, ptr(meg), ptr(plan.rec_order), ptr(plan.rec_off), B, C, T, O, R,
                         ptr(d_att), st)
            else:
                dv = _empty((B, T, IL), meg)
                du = _empty((B, T, O), meg)
                d_il_w = _empty((IL, O), meg)
                d_il_b = _empty((IL,), meg)
                call("bm_sensor_chain_bwd", ptr(g), ptr(meg), ptr(s["il_w2"]), ptr(s["subj_w"]), ptr(plan.subject),
                     ptr(s["u"]), ptr(s["v"]), ptr(subj_order), ptr(subj_off), ptr(plan.rec_order), ptr(plan.rec_off),
                     B, C, T, O, IL, D, Dp, S, R, ptr(dv), ptr(du), ptr(d_subj), ptr(d_il_w), ptr(d_il_b), ptr(d_att), st)
            dscores = _empty((R, O, C), meg)
            if s["heads_tc"]:
                Opad = _round_up(O, 64)
                call("bm_softmax_bwd", ptr(s["att"]), ptr(d_att), R * O, C, ptr(dscores), st)
                ds_t = _empty((R, C, Opad), meg)                   # pad columns zeroed by the transpose
                call("bm_transpose_nt_ld", ptr(dscores), R, O, C, Opad, ptr(ds_t), st)
                dheads = tc_wgrad(ds_t, s["emb"], R, C, Opad, P, P, 1, 1, status)[:O, :, 0].contiguous()
            else:
                dheads = _empty((O, P), meg)
                call("bm_attention_weights_bwd", ptr(d_att), ptr(s["att"]), ptr(s["emb"]), R, C, O, P, ptr(dscores),
                     ptr(dheads), st)

        if d_il_w is not None:
            d_il_w = d_il_w.reshape(s["il_shape"])
        if plan.bare_last:
            grads = [None, None, dheads, d_il_w, d_il_b, d_subj, None, None, None, None]
        else:
            grads = [None, None, dheads, d_il_w, d_il_b, d_subj,
                     dw0.reshape(s["w0_shape"]), db0, dw2.reshape(s["w2_shape"]), db2]
        for k in range(depth):
            grads.extend(layer_grads[k])
        for k in range(depth):
            if plan.glu_after[k]:
                grads.extend(glu_grads[k])
        if plan.has_sub_emb:
            grads.append(d_sub_emb)
        ctx.saved = None
        return tuple(grads)


def encoder_forward(plan: EncoderPlan, meg, heads, il_w, il_b, subj_w, w0, b0, w2, b2, layer_params, sub_emb=None):
    """`sub_emb` [B, E]: rows of the scaled subject embedding to append as channels (plan.has_sub_emb)."""
    extra = [] if sub_emb is None else [sub_emb]
    return _EncoderFn.apply(plan, meg, heads, il_w, il_b, subj_w, w0, b0, w2, b2, *layer_params, *extra)


# ----------------------------------------------------------------------------------------------------
# ClipLoss
# ----------------------------------------------------------------------------------------------------
_clip_ws: tp.Dict[torch.device, torch.Tensor] = {}


def _clip_workspace(like: torch.Tensor, Bn: int, Bc: int, KT: int) -> torch.Tensor:
    """Scratch of the CLIP score GEMM (split-K partial tiles, partial sums of squares, finalize ticket): one buffer per
    device, grown on demand to what the library asks for (`bm_clip_workspace`), handed to every call explicitly."""
    need = max(int(_lib.load().bm_clip_workspace(Bn, Bc, KT)), 2)
    dev = like.device
    ws = _clip_ws.get(dev)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, device=dev, dtype=torch.float32)
        _clip_ws[dev] = ws
    return ws


def _check_clip_operands(est: torch.Tensor, cand: torch.Tensor) -> None:
    if est.dtype != torch.float32 or cand.dtype != torch.float32:
        raise TypeError(f"ClipLoss kernels are fp32 (bm/losses.py computes in the input dtype; the reference trains in "
                        f"fp32): got {est.dtype} / {cand.dtype}")
    if est.device != cand.device:
        raise ValueError(f"estimate on {est.device}, candidate on {cand.device}")


def clip_scores(estimates: torch.Tensor, candidates: torch.Tensor, want_probs: bool = False):
    """ClipLoss.get_scores / get_probabilities (bm/losses.py:77-102); no autograd."""
    est = estimates.detach().contiguous().float()
    cand = candidates.detach().contiguous().float()
    Bn, Bc = est.shape[0], cand.shape[0]
    KT = est[0].numel()
    assert cand[0].numel() == KT
    inv = _empty((Bc,), est)
    scores = _empty((Bn, Bc), est)
    probs = _empty((Bn, Bc), est) if want_probs else None
    ws = _clip_workspace(est, Bn, Bc, KT)
    call("bm_clip_scores", ptr(est), ptr(cand), Bn, Bc, KT, 0, ptr(inv), ptr(scores), ptr(probs), ptr(ws), ws.numel(),
         ptr(tc_status_tensor(est.device)), stream())
    return probs if want_probs else scores


def candidate_inv_norms(candidates: torch.Tensor) -> torch.Tensor:
    """inv_norm[o] = 1 / (1e-8 + ||candidate_o||) (bm/losses.py:91), for a candidate set that is scored many times."""
    cand = candidates.detach().contiguous().float()
    Bc, KT = cand.shape[0], cand[0].numel()
    ss = _empty((Bc,), cand, torch.float64)
    inv = _empty((Bc,), cand)
    call("bm_candidate_inv_norms", ptr(cand), Bc, KT, ptr(ss), ptr(inv), stream())
    return inv


def clip_scores_prenormed(estimates: torch.Tensor, candidates: torch.Tensor, inv_norms: torch.Tensor) -> torch.Tensor:
    """ClipLoss.get_scores against a candidate set whose `candidate_inv_norms` are already known (retrieval evaluation:
    the same candidates serve every query batch, so they are normed once)."""
    est = estimates.detach().contiguous().float()
    cand = candidates if (candidates.is_contiguous() and candidates.dtype == torch.float32) \
        else candidates.contiguous().float()
    Bn, Bc = est.shape[0], cand.shape[0]
    KT = est[0].numel()
    assert cand[0].numel() == KT and inv_norms.numel() == Bc
    scores = _empty((Bn, Bc), est)
    ws = _clip_workspace(est, Bn, Bc, KT)
    call("bm_clip_scores", ptr(est), ptr(cand), Bn, Bc, KT, 1, ptr(inv_norms), ptr(scores), None, ptr(ws), ws.numel(),
         ptr(tc_status_tensor(est.device)), stream())
    return scores


class _ClipLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, estimate, candidate, target_offset: int):
        _check_clip_operands(estimate, candidate)
        est = estimate.contiguous()
        cand = candidate.contiguous()
        Bn, Bc = est.shape[0], cand.shape[0]
        KT = est[0].numel()
        inv = _empty((Bc,), est)
        scores = _empty((Bn, Bc), est)
        probs = _empty((Bn, Bc), est)
        row_loss = _empty((Bn,), est)
        loss = _empty((1,), est)
        ws = _clip_workspace(est, Bn, Bc, KT)
        call("bm_clip_loss_fwd", ptr(est), ptr(cand), Bn, Bc, KT, int(target_offset), ptr(inv), ptr(scores), ptr(probs),
             ptr(row_loss), ptr(loss), ptr(ws), ws.numel(), ptr(tc_status_tensor(est.device)), stream())
        if candidate.requires_grad:      # a trainable feature model produced the candidates (solver.py:304-320)
            ctx.save_for_backward(probs, inv, cand, scores, est)
        else:
            ctx.save_for_backward(probs, inv, cand)
        ctx.meta = (Bn, Bc, KT, int(target_offset), est.shape, cand.shape)
        return loss.reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        probs, inv, cand = ctx.saved_tensors[:3]
        Bn, Bc, KT, off, shape, cand_shape = ctx.meta
        gout = gout.reshape(1).contiguous().float()
        status = tc_status_tensor(probs.device)
        dest = dcand = None
        if ctx.needs_input_grad[0]:
            G = _empty((Bn, Bc), probs)
            dest = _empty(shape, probs)
            call("bm_clip_loss_bwd", ptr(probs), ptr(inv), ptr(cand), ptr(gout), Bn, Bc, KT, off, ptr(G), ptr(dest),
                 ptr(status), stream())
        if ctx.needs_input_grad[1]:
            scores, est = ctx.saved_tensors[3:]
            G = _empty((Bn, Bc), probs)
            coef = _empty((Bc,), probs)
            dcand = _empty(cand_shape, probs)
            call("bm_clip_loss_bwd_cand", ptr(probs), ptr(scores), ptr(inv), ptr(est), ptr(cand), ptr(gout), Bn, Bc, KT,
                 off, ptr(G), ptr(coef), ptr(dcand), ptr(status), stream())
        return dest, dcand, None


def clip_loss(estimate, candidate, target_offset: int = 0):
    return _ClipLossFn.apply(estimate, candidate, target_offset)


# ----------------------------------------------------------------------------------------------------
# L1Loss / L2Loss (bm/losses.py:11-26): mean of |estimate - output|^p over mask.expand_as(estimate)
# ----------------------------------------------------------------------------------------------------
REGRESSION_WS_DOUBLES = 1186           # BM_REGRESSION_WS_DOUBLES of include/bm_b200.h


def _regression_mask(mask: torch.Tensor, estimate: torch.Tensor) -> torch.Tensor:
    """The selection the reference indexes with, `mask.expand_as(estimate)`, as contiguous bytes [B, 1, T] when it is the
    same for every feature (the solver's features_mask), else [B, F, T]."""
    full = mask.expand_as(estimate)
    if full.stride(1) == 0:
        full = full[:, :1]
    return full.contiguous().view(torch.uint8)


class _RegressionLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, estimate, output, mask, p: int):
        est = estimate.contiguous()
        out = output.contiguous()            # the solver's targets are a time-cropped view (features[..., :-offset])
        m = _regression_mask(mask, est)
        B, F, T = est.shape
        ws = _empty((REGRESSION_WS_DOUBLES,), est, torch.float64)
        loss = _empty((1,), est)
        call("bm_regression_loss_fwd", ptr(est), ptr(out), ptr(m), B, F, m.shape[1], T, p, ptr(ws), ptr(loss), stream())
        ctx.save_for_backward(est, out, m, ws)      # ws holds the selected count the backward reads
        ctx.p = p
        return loss.reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        est, out, m, ws = ctx.saved_tensors
        B, F, T = est.shape
        dest = _empty(est.shape, est) if ctx.needs_input_grad[0] else None
        dout = _empty(est.shape, est) if ctx.needs_input_grad[1] else None
        g = gout.reshape(1).contiguous().float()
        call("bm_regression_loss_bwd", ptr(est), ptr(out), ptr(m), ptr(g), ptr(ws), B, F, m.shape[1], T, ctx.p, ptr(dest),
             ptr(dout), stream())
        return dest, dout, None, None


def regression_loss(estimate: torch.Tensor, output: torch.Tensor, mask: torch.Tensor, p: int) -> torch.Tensor:
    """mean over the elements selected by `mask.expand_as(estimate)` of |estimate - output| (p = 1, nn.L1Loss) or
    (estimate - output)^2 (p = 2, nn.MSELoss), as a 0-dim tensor; no host synchronisation.  estimate, output [B, F, T]
    fp32; mask bool, broadcastable to [B, F, T] ([B, 1, T] in the solver)."""
    if p not in (1, 2):
        raise ValueError(f"p must be 1 or 2, got {p}")
    if mask is None:
        raise TypeError("a mask is required (bm/losses.py:13 expands it over the estimate)")
    if mask.dtype != torch.bool:
        raise TypeError(f"the mask selects elements and must be torch.bool, got {mask.dtype}")
    if estimate.dim() != 3 or estimate.shape != output.shape:
        raise ValueError(f"estimate {tuple(estimate.shape)} and output {tuple(output.shape)} must be the same [B, F, T]")
    if not (estimate.device == output.device == mask.device):
        raise ValueError(f"estimate on {estimate.device}, output on {output.device}, mask on {mask.device}")
    return _RegressionLossFn.apply(estimate, output, mask, p)


# ----------------------------------------------------------------------------------------------------
# Stand-alone ChannelMerger.forward / SubjectLayers.forward (bm/models/common.py:334-362, 55-58): inside SimpleConv both are
# fused into the encoder; called on their own (analysis notebooks, user code) they run the same stage kernels.  Channel-major
# tensors in and out, like the reference; gradients flow to the parameters (and to `x` for SubjectLayers), not to `meg`.
# ----------------------------------------------------------------------------------------------------
class _MergerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, meg, heads, positions, rec_of_sample, rec_order, rec_off, freq, ban_centre, radius: float):
        meg = meg.contiguous()
        B, C, T = meg.shape
        R = positions.shape[0]
        O, P = heads.shape
        st = stream()
        emb, att = _empty((R, C, P), meg), _empty((R, O, C), meg)
        call("bm_attention_weights_fwd", ptr(positions), ptr(freq), ptr(heads.contiguous()), ptr(ban_centre), float(radius),
             R, C, O, P, ptr(emb), ptr(att), st)
        u = _empty((B, T, O), meg)
        call("bm_sensor_mix_fwd", ptr(meg), ptr(att), ptr(rec_of_sample), B, C, T, O, O, ptr(u), st)
        out = _empty((B, O, T), meg)
        call("bm_transpose_nt", ptr(u), B, T, O, ptr(out), st)
        ctx.save_for_backward(meg, emb, att, rec_order, rec_off)
        ctx.dims = (B, C, T, R, O, P)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        meg, emb, att, rec_order, rec_off = ctx.saved_tensors
        B, C, T, R, O, P = ctx.dims
        st = stream()
        g = _empty((B, T, O), meg)
        call("bm_transpose_nt", ptr(gout.contiguous()), B, O, T, ptr(g), st)
        d_att, dscores, dheads = _empty((R, O, C), meg), _empty((R, O, C), meg), _empty((O, P), meg)
        call("bm_sensor_mix_bwd", ptr(g), O, ptr(meg), ptr(rec_order), ptr(rec_off), B, C, T, O, R, ptr(d_att), st)
        call("bm_attention_weights_bwd", ptr(d_att), ptr(att), ptr(emb), R, C, O, P, ptr(dscores), ptr(dheads), st)
        return None, dheads, None, None, None, None, None, None, None


def channel_merger_forward(meg, heads, positions, rec_of_sample, rec_order, rec_off, freq, ban_centre, radius):
    return _MergerFn.apply(meg, heads, positions, rec_of_sample, rec_order, rec_off, freq, ban_centre, radius)


class _SubjectLayersFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weights, subject):
        x = x.contiguous()
        B, Cin, T = x.shape
        S, _, D = weights.shape
        st = stream()
        xl = _empty((B, T, Cin), x)
        call("bm_transpose_nt", ptr(x), B, Cin, T, ptr(xl), st)
        yl = _empty((B, T, D), x)
        w = weights.contiguous()
        call("bm_subject_layers_fwd", ptr(xl), Cin, ptr(w), ptr(subject), B, T, Cin, D, D, ptr(yl), st)
        out = _empty((B, D, T), x)
        call("bm_transpose_nt", ptr(yl), B, T, D, ptr(out), st)
        ctx.save_for_backward(xl, w, subject)
        ctx.dims = (B, Cin, T, S, D)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        xl, w, subject = ctx.saved_tensors
        B, Cin, T, S, D = ctx.dims
        st = stream()
        g = _empty((B, T, D), xl)
        call("bm_transpose_nt", ptr(gout.contiguous()), B, D, T, ptr(g), st)
        order, off = group_layout(subject, S)
        dxl, dw = _empty((B, T, Cin), xl), _empty((S, Cin, D), xl)
        call("bm_subject_layers_bwd", ptr(g), D, ptr(xl), Cin, ptr(w), ptr(subject), ptr(order), ptr(off), B, T, Cin, D, S,
             Cin, ptr(dxl), ptr(dw), st)
        dx = _empty((B, Cin, T), xl)
        call("bm_transpose_nt", ptr(dxl), B, T, Cin, ptr(dx), st)
        return dx, dw, None


def subject_layers_forward(x, weights, subject):
    return _SubjectLayersFn.apply(x, weights, subject)


def library_loaded() -> bool:
    return _lib._lib is not None
