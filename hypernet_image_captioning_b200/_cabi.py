"""ctypes binding of libcaphn_b200.so -- the C-ABI boundary (include/caphn_b200.h).

Every entry point takes raw device pointers, sizes and a cudaStream_t (as void*), and returns an int
(0 = ok, -1 = invalid argument, otherwise a cudaError_t).  There is no CPU fallback: if the library is missing or a
call fails, this module raises.
"""
import ctypes
import os
from ctypes import c_double, c_float, c_int, c_long, c_longlong, c_void_p

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libcaphn_b200.so")

P = c_void_p  # every pointer argument
I = c_int
L = c_long
LL = c_longlong
F = c_float
D = c_double

# name -> argtypes (mirrors include/caphn_b200.h)
SIGNATURES = {
    "caphn_rows_linear_fwd": [P, P, P, L, P, L, I, L, L, I, F, P],
    "caphn_rows_linear_bwd": [P, P, L, P, L, P, L, P, P, P, P, L, I, L, L, I, F, P],
    "caphn_rows_linear_fwd_bf16": [P, P, P, L, P, L, I, L, L, I, F, P],
    "caphn_rows_linear_bwd_bf16": [P, P, L, P, L, P, L, P, P, P, P, L, I, L, L, I, F, P],
    "caphn_gemm_f32": [P, L, I, P, L, I, P, L, P, I, I, I, I, I, I, P],
    "caphn_split_bf16": [P, L, L, I, P, P, L, P],
    "caphn_split_bf16_t": [P, L, I, I, P, P, L, P],
    "caphn_gemm_tc": [P, P, P, P, L, P, L, P, I, I, I, I, P],
    "caphn_gemm_tc_ex": [P, P, L, I, P, P, L, I, L, P, L, P, I, I, I, I, P],
    "caphn_transpose_pad": [P, L, P, L, I, I, P],
    "caphn_copy_pad": [P, L, P, L, L, I, P],
    "caphn_transpose_pad_batched": [P, L, L, P, L, L, I, I, I, P],
    "caphn_copy_pad_batched": [P, L, L, P, L, L, I, L, I, P],
    "caphn_gru_seq_fwd": [P, P, I, P, P, P, P, P, P, I, I, I, I, P],
    "caphn_gru_seq_bwd": [P, P, P, P, P, I, P, P, P, P, P, P, I, I, I, I, P],
    "caphn_gru_cluster_plan": [I, P],
    "caphn_gru_cluster_fwd": [P, P, P, P, P, P, I, I, I, P],
    "caphn_gru_cluster_bwd": [P, P, P, P, P, P, P, I, I, I, P],
    "caphn_gru_cluster_fwd_grouped": [P, P, P, P, P, P, I, I, I, P, I, L, L, P],
    "caphn_gru_cluster_bwd_grouped": [P, P, P, P, P, P, P, I, I, I, P, I, L, P],
    "caphn_ce_fwd": [P, L, P, L, I, I, LL, P, P, P, P],
    "caphn_ce_bwd": [P, L, P, L, I, I, LL, P, P, P, P, L, P],
    "caphn_ce_bwd_split": [P, L, P, L, I, I, LL, P, P, P, P, P, L, P, P, L, P, P],
    "caphn_softmax_argmax": [P, L, L, I, P, L, P, P],
    "caphn_gather_rows": [P, P, L, I, P, L, P],
    "caphn_build_inputs": [P, P, P, I, I, I, I, P, P],
    "caphn_embed_scatter_add": [P, P, I, I, I, I, P, P],
    "caphn_scatter_add_rows": [P, L, P, L, I, P, P],
    "caphn_colsum": [P, L, L, I, P, P],
    "caphn_lstm_seq_fwd": [P, P, I, P, P, P, P, P, P, P, P, I, I, I, I, P],
    "caphn_lstm_seq_bwd": [P, P, P, I, P, P, P, I, I, I, I, P],
    "caphn_lstm_seq_fwd_grouped": [P, P, I, P, L, P, P, P, P, I, I, I, P, I, P],
    "caphn_lstm_seq_bwd_grouped": [P, P, P, I, P, P, I, I, I, P, I, P],
    "caphn_attgru_seq_fwd": [P] * 14 + [L] + [P] * 5 + [I] * 9 + [P],
    "caphn_attgru_seq_bwd": [P] * 23 + [I] * 7 + [P],
    "caphn_attstep_pack_size": [I, I, I, I, P, P],
    "caphn_attstep_pack": [P, P, P, I, I, I, P, P],
    "caphn_attstep_fwd": [P] * 13 + [L] + [P] * 5 + [I] * 8 + [P],
    "caphn_attstep_bwd_size": [I, I, I, I, I, P, P],
    "caphn_attstep_bwd_pack": [P, P, P, I, I, I, P, P],
    "caphn_attstep_bwd": [P] * 22 + [I] * 5 + [P],
    "caphn_attn_df": [P, P, P, I, I, I, I, P],
    "caphn_gemm_tc_grouped": [P, P, L, L, L, I, P, P, L, L, L, I, P, L, P, P, P, I, I, P],
    "caphn_split_bf16_gather": [P, L, P, L, I, P, P, L, P],
    "caphn_split_bf16_batched": [P, L, L, I, I, I, P, P, L, P],
    "caphn_group_colsum": [P, L, P, I, I, I, I, P, L, P],
    "caphn_gemm_tc_amax": [P, P, L, I, P, P, L, I, L, P, L, P, I, I, P, P, I, P, P],
    "caphn_argmax_finish_gather": [P, P, I, I, L, P, I, P, P, L, P],
    "caphn_beam_step": [P] * 14 + [I] * 8 + [P],
    "caphn_leaky_relu": [P, L, F, P],
    "caphn_leaky_relu_bwd": [P, P, L, F, P],
    "caphn_attstep_pack_grouped": [P, P, P, I, I, I, I, L, P, P],
    "caphn_attstep_fwd_grouped": [P] * 13 + [L] + [P] * 5 + [I] * 8 + [P, I, I, P],
    "caphn_attstep_bwd_pack_grouped": [P, P, P, I, I, I, I, L, P, P],
    "caphn_attstep_bwd_grouped": [P] * 22 + [I] * 5 + [P, I, I, P],
    "caphn_mean_pos": [P, I, I, I, P, P],
    "caphn_mean_pos_bwd": [P, P, I, I, I, P, P],
    "caphn_relu_mask": [P, P, L, P],
    "caphn_sumsq": [P, L, P, P],
    "caphn_clip_coef": [P, F, P, P, P],
    "caphn_adam_step": [P, P, P, P, L, D, D, D, D, D, I, P, P],
    "caphn_sumsq_bf16": [P, L, P, P],
    "caphn_adam_step_bf16": [P, P, P, P, P, L, D, D, D, D, D, I, P, P],
    "caphn_gram": [P, L, I, L, P, P],
    "caphn_sumsq_lowrank": [P, P, I, P, P],
    "caphn_adam_step_lowrank": [P, P, P, P, L, P, L, I, L, L, D, D, D, D, D, I, P, P],
    "caphn_caption_compact": [P, L, I, I, LL, LL, LL, P, P, P],
    "caphn_bleu_counts": [P, P, I, P, P, I, I, I, P, P],
    "caphn_ce_fwd_split": [P, L, P, L, I, I, LL, P, P, P, P, P, L, P],
    "caphn_gemm_tc_scaled": [P, P, L, I, P, P, L, I, L, P, L, P, I, I, I, P, P, P],
    "caphn_gru_decode_step": [P, P, P, I, I, P, P, P, P, P, P, P, L, P, I, I, P],
    "caphn_gru_decode_step_tok": [P, I, P, P, P, P, P, P, P, L, I, I, P],
    "caphn_gru_resident_plan": [I, P],
    "caphn_gru_resident_fwd": [P, P, P, P, P, P, I, I, I, P],
    "caphn_gru_resident_bwd": [P, P, P, P, P, P, P, I, I, I, P],
    "caphn_launch_count": [P],
    "caphn_build_arch": [P],
}

_lib = None
_launches = 0  # number of C-ABI calls made (bench.py reports kernel launches from the per-call launch counts below)


class CaphnError(RuntimeError):
    pass


def load():
    """Load the shared library (building it first if nvcc is available and the sources changed)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:
            from . import build as _build
            _build.build()
        except Exception as e:  # no silent fallback: the product path needs the CUDA library
            raise CaphnError(f"libcaphn_b200.so is missing and could not be built: {e}") from e
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:
        raise CaphnError(f"cannot load {LIB_PATH}: {e}") from e
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header / library mismatch; must be loud
        fn.argtypes = argtypes
        fn.restype = c_int
    _lib = lib
    return lib


def call(name, *args):
    global _launches
    lib = load()
    rc = getattr(lib, name)(*args)
    _launches += 1
    if rc != 0:
        raise CaphnError(f"{name} failed with status {rc}" + (" (invalid argument)" if rc == -1 else " (cudaError_t)"))


def launches():
    """Number of CUDA kernels the library has launched since load (counted inside the library)."""
    out = ctypes.c_ulonglong(0)
    call("caphn_launch_count", ctypes.byref(out))
    return int(out.value)
