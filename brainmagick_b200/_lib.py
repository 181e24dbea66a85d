"""ctypes binding of libbm_b200.so (include/bm_b200.h).  There is no fallback: if the CUDA library is missing
or a call fails, this raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_longlong, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbm_b200.so")

P, I, L, F = c_void_p, c_int, c_longlong, c_float

# name -> argtypes, in the order of include/bm_b200.h
SIGNATURES = {
    "bm_attention_weights_fwd": [P, P, P, P, F, I, I, I, I, P, P, P],
    "bm_attention_weights_bwd": [P, P, P, I, I, I, I, P, P, P],
    "bm_fourier_emb": [P, P, I, I, I, P, P],
    "bm_masked_softmax": [P, P, P, F, I, I, I, P],
    "bm_softmax_bwd": [P, P, L, I, P, P],
    "bm_sensor_chain_fwd": [P, P, P, P, P, P, P, I, I, I, I, I, I, I, P, P, P, P],
    "bm_sensor_chain_bwd": [P, P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, P, P, P, P, P, P, P],
    "bm_sensor_mix_fwd": [P, P, P, I, I, I, I, I, P, P],
    "bm_initial_linear_fwd": [P, I, P, P, I, I, I, I, I, P, P],
    "bm_subject_layers_fwd": [P, I, P, P, I, I, I, I, I, P, P],
    "bm_subject_layers_bwd": [P, I, P, I, P, P, P, P, I, I, I, I, I, I, P, P, P],
    "bm_initial_linear_bwd": [P, I, P, I, P, I, I, I, I, I, P, P, P, P],
    "bm_sensor_mix_bwd": [P, I, P, P, P, I, I, I, I, I, P, P],
    "bm_conv_weight_prep": [P, I, I, I, P, P, P],
    "bm_conv1d_fwd": [P, P, P, I, I, I, I, I, I, P, P, P],
    "bm_bn_stats_finalize": [P, L, F, F, P, P, P, P, I, P],
    "bm_bn_eval_stats": [P, P, F, P, P, I, P],
    "bm_bn_gelu_skip_fwd": [P, P, P, P, P, P, P, L, I, P, P],
    "bm_bn_gelu_skip_bwd": [P, P, P, P, P, P, I, L, I, P, P, P, P, P, P],
    "bm_conv1d_bwd_data": [P, P, P, I, I, I, I, I, I, P, P],
    "bm_conv1d_bwd_weight": [P, P, I, I, I, I, I, I, P, P, P],
    "bm_conv1d_glu_fwd": [P, P, P, I, I, I, I, I, P, P, P],
    "bm_glu_bwd": [P, P, L, I, P, P, P, P],
    "bm_head_fwd": [P, P, P, P, P, I, I, I, I, P, P, P, P],
    "bm_head_bwd": [P, P, P, P, P, P, I, I, I, I, P, P, P, P, P, P, P],
    "bm_head_bwd_params": [P, P, P, P, I, I, I, I, P, P, P, P, P, P],
    "bm_clip_scores": [P, P, I, I, L, I, P, P, P, P, L, P, P],
    "bm_clip_loss_fwd": [P, P, I, I, L, I, P, P, P, P, P, P, L, P, P],
    "bm_clip_loss_bwd": [P, P, P, P, I, I, L, I, P, P, P, P],
    "bm_set_debug_flags": [I],
    "bm_set_debug_buffer": [P],
    "bm_tc_conv_supported": [I, I, I, I, I],
    "bm_tc_weight_split": [P, I, I, I, P, P, P, P, P],
    "bm_tc_conv1d": [P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, P, P, P, P, P, P],
    "bm_tc_conv1d_persistent_supported": [I, I, I, I, I],
    "bm_tc_conv1d_persistent": [P, P, P, I, I, I, I, I, I, I, I, I, I, I, P, P, P, P, P, P],
    "bm_amax": [P, L, P, P],
    "bm_f16_split": [P, L, P, P, P, P],
    "bm_tc_weight_split_f16": [P, P, I, I, I, P, P, P, P, P],
    "bm_tc_conv1d_f16": [P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, P, P, P, P, P, P, P],
    "bm_col_stats": [P, L, I, P, P],
    "bm_channel_mask": [P, P, I, I, I, P, P],
    "bm_transpose_nt": [P, I, I, I, P, P],
    "bm_transpose_nt_ld": [P, I, I, I, I, P, P],
    "bm_tc_wgrad_supported": [I, I],
    "bm_tc_wgrad": [P, P, I, I, I, I, I, I, I, P, P, P, P, P],
    "bm_tc_wgrad_conv_supported": [I, I, I, I],
    "bm_tc_wgrad_conv": [P, P, I, I, I, I, I, I, I, P, P, P, P],
    "bm_tc_wgrad_conv_f16": [P, P, P, P, I, I, I, I, I, I, I, P, P, P, P],
    "bm_col_sum": [P, L, I, P, P],
    "bm_tc_pointwise_sel": [P, P, P, P, I, I, I, I, I, P, P, P],
    "bm_tc_wgrad_grouped": [P, P, P, P, I, I, I, I, I, P, P, P],
    "bm_gelu_bwd": [P, P, L, P, P],
    "bm_candidate_inv_norms": [P, I, L, P, P, P],
    "bm_retrieval_topk": [P, L, I, I, P, I, I, I, P, P, P, P, P, P, P, P, P, P],
    "bm_retrieval_probs": [P, L, I, I, P, P],
    "bm_retrieval_vocab_probs": [P, L, I, P, P, P, P, P, I, P, P, P],
    "bm_rowdot_scaled": [P, P, I, L, P, P],
    "bm_scale_clamp_crop": [P, P, P, P, I, I, I, I, I, F, I, I, P, P, P],
    "bm_reject_compact": [P, P, L, F, I, P, P, P, P],
    "bm_gather_rows": [P, P, I, L, P, P],
    "bm_regression_loss_fwd": [P, P, P, I, I, I, I, I, P, P, P],
    "bm_regression_loss_bwd": [P, P, P, P, P, I, I, I, I, I, P, P, P],
    "bm_bn_act_skip_fwd": [P, P, P, P, P, P, P, L, I, I, F, P],
    "bm_bn_act_skip_bwd": [P, P, P, P, P, P, I, L, I, I, F, P, P, P, P, P],
    "bm_clip_loss_bwd_cand": [P, P, P, P, P, P, I, I, L, I, P, P, P, P, P],
}

_lib = None


class BmB200Error(RuntimeError):
    pass


def load():
    """Loads the shared library (once).  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise BmB200Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). brainmagick_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.bm_last_error.restype = ctypes.c_char_p
    lib.bm_last_error.argtypes = []
    lib.bm_abi_version.restype = c_int
    lib.bm_abi_version.argtypes = []
    lib.bm_launch_count.restype = ctypes.c_ulonglong
    lib.bm_launch_count.argtypes = []
    lib.bm_tc_wgrad_workspace.restype = c_longlong
    lib.bm_tc_wgrad_workspace.argtypes = [I, I, I, I]
    lib.bm_tc_wgrad_conv_workspace.restype = c_longlong
    lib.bm_tc_wgrad_conv_workspace.argtypes = [I, I, I, I, I]
    lib.bm_clip_workspace.restype = c_longlong
    lib.bm_clip_workspace.argtypes = [I, I, L]
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = c_int
        fn.argtypes = argtypes
    _lib = lib
    return lib


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda, "brainmagick_b200 kernels need CUDA tensors (no CPU fallback)"
    assert t.is_contiguous(), "non-contiguous tensor handed to the C ABI"
    return c_void_p(t.data_ptr())


def stream():
    """The current CUDA stream's handle (raw C accessors: torch.cuda.current_stream() builds a Stream object and resolves the
    device through several Python layers, 1.9 ms per step over the ~1 400 calls of one)."""
    return c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


def launch_count() -> int:
    return int(load().bm_launch_count())


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise BmB200Error(f"{name} failed (code {rc}): {lib.bm_last_error().decode()}")
