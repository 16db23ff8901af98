"""ctypes binding of libdeer_b200.so (declared in include/deer_b200.h).

There is NO fallback: if the library is missing or a tensor is not a CUDA tensor the call raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float as F
from ctypes import c_int as I
from ctypes import c_longlong as L
from ctypes import c_ulonglong as U
from ctypes import c_void_p as P

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DEER_B200_LIB: another build of the same library (same-box A/B of two kernel versions, tools/gpu_r2_*.sh); no fallback
LIB_PATH = os.environ.get("DEER_B200_LIB") or os.path.join(_HERE, "csrc", "libdeer_b200.so")

class GemmX3Args(ctypes.Structure):
    """deer_gemm_x3_args (include/deer_b200.h)."""
    _fields_ = [("A", P), ("B", P), ("C", P), ("bias", P), ("gate", P), ("colsum", P), ("drop_step", P),
                ("lda", L), ("ldb", L), ("ldc", L), ("ldgate", L),
                ("sA", L), ("sB", L), ("sC", L), ("sBias", L), ("sGate", L), ("sColsum", L),
                ("drop_seed", U), ("drop_offset", U), ("drop_ld", L), ("drop_batch_stride", L), ("drop_col0", I),
                ("M", I), ("N", I), ("K", I), ("batch", I), ("transA", I), ("transB", I), ("act", I),
                ("beta", F), ("drop_p", F), ("gate_mode", I), ("gate_scale", F), ("splitk", I)]


# name -> argtypes (every function returns int unless listed in _RESTYPES)
_PROTOS = {
    "deer_version": [],
    "deer_last_error": [],
    "deer_launch_count": [],
    "deer_gemm_engine_count": [I],
    "deer_timestamp": [P, I, P],
    "deer_set_option": [I, I],
    "deer_lstm_set_profile_buffer": [P],
    "deer_gemm": [P, L, I, P, L, I, P, L, I, I, I, P, I, F, I, L, L, L, L, I, P],
    "deer_gemm_rowterm": [P, L, I, P, L, I, P, L, I, I, I, P, P, I, I, I, P],
    "deer_gemm_x3": [ctypes.POINTER(GemmX3Args), P],
    "deer_chain_run": [P, P],
    "deer_chain_max_ops": None,
    "deer_chain_max_levels": None,
    "deer_gemm_h16_split": [P, P, L, I, P, P, L, I, P, L, I, I, I, P, I, P],
    "deer_cast_split16": [P, L, P, P, P, L, L, I, I, P],
    "deer_gemm_h16": [P, L, I, I, P, L, I, I, P, L, P, L, I, I, I, I, P, I, F, P],
    "deer_cast16": [P, L, P, L, L, I, I, I, P],
    "deer_gemm_h16_set_profile_buffer": [P],
    "deer_bias_act_bwd": [P, L, P, L, P, L, P, I, I, I, P],
    "deer_layernorm_fwd": [P, P, P, P, P, P, I, I, F, P],
    "deer_layernorm_bwd": [P, P, P, P, P, P, P, P, I, I, P],
    "deer_dropout": [P, P, L, F, U, U, P, P],
    "deer_dropout_cast16": [P, P, P, L, F, U, U, P, P, P],
    "deer_gemm_h16_dropmask": [P, L, I, I, P, L, I, I, P, L, I, I, I, P, F, P],
    "deer_rowdot_fwd": [P, P, P, P, L, I, P],
    "deer_rowdot_bwd": [P, P, P, P, P, P, L, I, P],
    "deer_attn_pool_fwd": [P, L, L, P, L, L, P, P, P, I, I, I, I, P],
    "deer_attn_pool_bwd": [P, P, L, L, P, L, L, P, P, P, P, I, I, I, I, I, P],
    "deer_attn_pool_len_fwd": [P, L, L, P, L, L, P, I, P, P, I, I, I, P],
    "deer_attn_pool_len_bwd": [P, P, L, L, L, L, P, I, P, P, P, I, I, I, P],
    "deer_permute_bt": [P, P, I, I, I, P],
    "deer_permute_bt_cast16": [P, P, P, I, I, I, I, P],
    "deer_permute_bt_cast16_len": [P, P, P, P, I, I, I, I, I, I, P],
    "deer_scorer_bwd": [P, P, P, P, P, P, P, P, L, I, P],
    "deer_rowscale": [P, P, P, L, I, P],
    "deer_rowscale_len": [P, P, P, I, I, I, I, P],
    "deer_im2col3": [P, P, I, I, I, P],
    "deer_col2im3": [P, P, I, I, I, P],
    "deer_rows_pad": [P, P, I, I, I, I, I, I, P],
    "deer_rows_pad_fused": [P, P, P, P, I, I, I, I, I, I, F, U, U, P, P],
    "deer_rows_pad_fused_len": [P, P, P, P, P, I, I, I, I, I, I, I, F, U, U, P, P],
    "deer_rows_pad_colsum": [P, P, P, I, I, I, P],
    "deer_conv3_weight_pack": [P, P, I, I, I, P],
    "deer_bn_stats": [P, P, L, I, P],
    "deer_bn_update_running": [P, P, P, P, L, I, F, P],
    "deer_bn_relu_fwd": [P, P, P, P, P, P, L, I, F, P],
    "deer_bn_relu_bwd": [P, P, P, P, P, P, P, P, P, P, L, I, F, I, P],
    "deer_bn_stats_len": [P, P, P, I, I, I, I, P],
    "deer_bn_update_running_len": [P, P, P, P, I, F, P],
    "deer_bn_relu_fwd_len": [P, P, P, P, P, P, P, I, I, I, I, F, P],
    "deer_bn_relu_bwd_len": [P, P, P, P, P, P, P, P, P, P, P, I, I, I, I, F, I, P],
    "deer_mha2_fwd": [P, P, P, P, P, I, I, I, P],
    "deer_mha2_bwd": [P, P, P, P, P, P, I, I, I, P],
    "deer_lstm_fwd": [P, P, P, P, P, P, I, I, I, I, P],
    "deer_lstm_bwd": [P, P, P, P, P, P, P, I, I, I, I, P],
    "deer_lstm_cluster_tile": [I],
    "deer_lstm_cluster_fwd": [P, P, P, P, P, P, P, P, I, I, I, P],
    "deer_lstm_prep": [P, P, P, P, P, P, P, P, I, I, I, I, P],
    "deer_lstm_unprep": [P, P, P, P, P, P, P, P, P, P, P, I, I, P],
    "deer_lstm_cluster_fwd_pre16": [P, P, P, P, P, P, P, P, I, I, I, P],
    "deer_lstm_cluster_bwd": [P, P, P, P, P, P, P, P, I, I, I, P],
    "deer_lstm_cluster_xin_mode": [I, I, I],
    "deer_lstm_cluster_fwd_xin": [P, I, P, P, P, P, P, P, P, P, P, I, I, I, P],
    "deer_gate_rows_interleave": [P, P, I, I, I, I, P],
    "deer_lstm_mask_pre": [P, I, P, I, I, I, I, P],
    "deer_nig_head_fwd": [P, P, P, P, P, P, P, P, L, P],
    "deer_nig_head_bwd": [P, P, P, P, P, P, P, P, P, L, P],
    "deer_nig_loss_stats": [P, P, P, P, P, P, P, P, P, L, I, I, F, P],
    "deer_nig_loss_finish": [P, P, P, P, P, P, P, P, P, F, F, F, F, F, L, L, I, I, F, P, P, P],
    "deer_nig_loss_stats_mask": [P, P, P, P, P, P, P, P, P, P, L, I, I, F, P],
    "deer_nig_loss_finish_mask": [P, P, P, P, P, P, P, P, P, P, F, F, F, F, F, L, I, I, F, P, P, P, P],
    "deer_amini_loss": [P, P, P, P, P, F, F, L, P, P, P, P],
    "deer_sumsq": [P, L, P, P],
    "deer_fill_zero": [P, L, P, L, P],
    "deer_step_increment": [P, P],
    "deer_adamw": [P, P, P, P, L, F, F, F, F, F, I, P, F, F, P, P, P],
    "deer_axpby": [P, P, P, L, F, F, P],
    "deer_mix_fwd": [P, L, P, L, P, P, P, L, I, P],
    "deer_mix_bwd": [P, P, L, P, L, P, P, P, L, P, L, P, P, L, I, P],
    "deer_gate_fwd": [P, P, P, P, L, P],
    "deer_gate_bwd": [P, P, P, P, P, P, P, L, P],
    "deer_coldiv_fwd": [P, P, P, L, I, P],
    "deer_coldiv_bwd": [P, P, P, P, P, L, I, P],
    "deer_softmax_rows_fwd": [P, P, L, I, P],
    "deer_softmax_rows_bwd": [P, P, P, L, I, P],
    "deer_linguistic_features": [P, P, P, I, I, I, P],
    "deer_metrics_moments": [P, P, L, I, P, P],
    "deer_uce_prepare": [P, P, P, L, I, P, P, P, P],
    "deer_uce_select": [P, L, P, I, P, P, L, P],
    "deer_uce_bins": [P, P, L, I, P, P, P],
}
_RESTYPES = {"deer_last_error": ctypes.c_char_p, "deer_launch_count": L, "deer_gemm_engine_count": L}

EXPORTS = tuple(_PROTOS)

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"deer_b200: {LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU or PyTorch fallback for this path.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, args in _PROTOS.items():
            fn = getattr(lib, name)
            fn.argtypes = args if args is not None else []
            fn.restype = _RESTYPES.get(name, I)
        _lib = lib
    return _lib


class DeerError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().deer_last_error()
        raise DeerError(f"deer_b200 {what} failed with status {rc}: {msg.decode() if msg else ''}")


def launch_count() -> int:
    return int(load().deer_launch_count())


ENGINE_NAMES = {1: "simt", 2: "tf32", 3: "tf32_pair", 4: "h16", 5: "tf32x3", 6: "h16_split"}


def engine_counts() -> dict:
    """{engine name: GEMM dispatches since process start} (deer_gemm_engine_count)."""
    lib = load()
    return {n: int(lib.deer_gemm_engine_count(e)) for e, n in ENGINE_NAMES.items()}


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    """Device pointer of a CUDA fp32 tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise DeerError("deer_b200 operates on CUDA tensors only; there is no CPU fallback on this path")
    return t.data_ptr()


def call(name: str, *args):
    check(getattr(load(), name)(*args, stream()), name)


_tf32_pair = [1]


def tf32_pair_on() -> bool:
    """DEER_OPT_TF32_PAIR as last set through set_option (default 1)."""
    return bool(_tf32_pair[0])


def set_option(option: int, value: int):
    check(load().deer_set_option(option, value), "deer_set_option")
    if option == 6:
        _tf32_pair[0] = int(value)
