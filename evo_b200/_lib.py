"""ctypes binding of libevo_b200.so (the C ABI declared in include/evo_b200.h).

There is no CPU fallback and no other backend: if the shared library is missing or a
call fails, this module raises.  Build it with ``python -m evo_b200.build``."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libevo_b200.so")

EPI_NONE, EPI_BIAS, EPI_BIAS_RESID, EPI_RESID, EPI_GELU_GATE = range(5)
EPI_BIAS_ROPE = 6
EPI_HYENA_STEP = 7


class EvoError(RuntimeError):
    pass


class GemmParams(C.Structure):
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int64), ("W", C.c_void_p), ("C", C.c_void_p), ("ldc", C.c_int64),
                ("bias", C.c_void_p), ("residual", C.c_void_p), ("ldr", C.c_int64),
                ("M", C.c_int64), ("N", C.c_int64), ("K", C.c_int64), ("epilogue", C.c_int), ("variant", C.c_int),
                ("rope_cos", C.c_void_p), ("rope_sin", C.c_void_p), ("rope_L", C.c_int64), ("rope_cols", C.c_int64),
                ("c_peers", C.c_void_p), ("n_c_peers", C.c_int), ("peer_period", C.c_int64), ("peer_inner", C.c_int64), ("peer_row0", C.c_int64)]


class GemmSmallMParams(C.Structure):
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int64), ("W", C.c_void_p), ("C", C.c_void_p), ("ldc", C.c_int64),
                ("bias", C.c_void_p), ("residual", C.c_void_p), ("ldr", C.c_int64),
                ("M", C.c_int64), ("N", C.c_int64), ("K", C.c_int64), ("epilogue", C.c_int),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("fir_state", C.c_void_p), ("state", C.c_void_p), ("fir_w", C.c_void_p), ("fir_b", C.c_void_p), ("Dskip", C.c_void_p),
                ("poles", C.c_void_p), ("residues", C.c_void_p)]


class HyenaParams(C.Structure):
    _fields_ = [("z", C.c_void_p), ("y", C.c_void_p), ("fir_w", C.c_void_p), ("fir_b", C.c_void_p), ("Dskip", C.c_void_p),
                ("poles", C.c_void_p), ("residues", C.c_void_p),
                ("B", C.c_int), ("L", C.c_int64), ("D", C.c_int), ("S", C.c_int), ("nheads", C.c_int),
                ("halo", C.c_void_p), ("state_in", C.c_void_p), ("state_out", C.c_void_p), ("fir_state_out", C.c_void_p),
                ("force_segments", C.c_int), ("state_only", C.c_int), ("reuse_segment_states", C.c_int)]


class AttnParams(C.Structure):
    _fields_ = [("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p),
                ("q_tok_stride", C.c_int64), ("kv_tok_stride", C.c_int64),
                ("q_batch_stride", C.c_int64), ("kv_batch_stride", C.c_int64),
                ("B", C.c_int), ("Lq", C.c_int64), ("Lk", C.c_int64), ("H", C.c_int), ("hd", C.c_int),
                ("q_pos0", C.c_int64), ("softmax_scale", C.c_float),
                ("out_peers", C.c_void_p), ("n_out_peers", C.c_int), ("out_rows_per_peer", C.c_int64), ("out_row_stride", C.c_int64), ("out_col0", C.c_int64)]


class ScoreParams(C.Structure):
    _fields_ = [("x", C.c_void_p), ("W", C.c_void_p), ("targets", C.c_void_p), ("logprobs", C.c_void_p), ("entropy", C.c_void_p),
                ("M", C.c_int64), ("V", C.c_int), ("K", C.c_int64), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class LoopParams(C.Structure):
    _fields_ = [("forced", C.c_void_p), ("n_forced", C.c_int64), ("forced_stride", C.c_int64),
                ("picked", C.c_void_p), ("picked_stride", C.c_int64),
                ("kept_logits", C.c_void_p), ("n_out", C.c_int64),
                ("top_k", C.c_int32), ("top_p", C.c_float), ("temperature", C.c_float),
                ("seed", C.c_uint64), ("step0", C.c_int64)]


class RaggedLoopParams(C.Structure):
    _fields_ = [("n_forced", C.c_void_p), ("n_out", C.c_void_p), ("start", C.c_void_p),
                ("forced", C.c_void_p), ("forced_stride", C.c_int64),
                ("picked", C.c_void_p), ("kept_logits", C.c_void_p), ("out_cols", C.c_int64),
                ("top_k", C.c_int32), ("top_p", C.c_float), ("temperature", C.c_float),
                ("seed", C.c_uint64)]


# name -> (restype, argtypes); every symbol include/evo_b200.h declares
SIGNATURES = {
    "evo_last_error": (C.c_char_p, []),
    "evo_abi_version": (C.c_int, []),
    "evo_launch_count": (C.c_int64, []),
    "evo_reset_launch_count": (None, []),
    "evo_note_graph_replay": (None, [C.c_int64]),
    "evo_embed": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "evo_rmsnorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_void_p]),
    "evo_gemm": (C.c_int, [C.POINTER(GemmParams), C.c_void_p]),
    "evo_gemm_smallm_workspace": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64, C.c_int]),
    "evo_gemm_smallm": (C.c_int, [C.POINTER(GemmSmallMParams), C.c_void_p]),
    "evo_set_pdl": (C.c_int, [C.c_int]),
    "evo_hyena_fwd_workspace": (C.c_size_t, [C.POINTER(HyenaParams)]),
    "evo_hyena_fwd": (C.c_int, [C.POINTER(HyenaParams), C.c_void_p, C.c_size_t, C.c_void_p]),
    "evo_hyena_fwd_ragged_workspace": (C.c_size_t, [C.POINTER(HyenaParams)]),
    "evo_hyena_fwd_ragged": (C.c_int, [C.POINTER(HyenaParams), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "evo_hyena_step": (C.c_int, [C.c_void_p] * 9 + [C.c_int] * 4 + [C.c_void_p]),
    "evo_hyena_combine_states": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "evo_peer_publish": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "evo_peer_wait": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "evo_rope_tables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_float, C.c_void_p]),
    "evo_rotary_qk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "evo_attn_fwd_workspace": (C.c_size_t, [C.POINTER(AttnParams), C.c_int]),
    "evo_attn_fwd_ws": (C.c_int, [C.POINTER(AttnParams), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "evo_kv_append": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_void_p]),
    "evo_gelu_gate_interleaved": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "evo_decode_qkv_prep": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p]),
    "evo_decode_attn_workspace": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "evo_decode_attn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_size_t, C.c_void_p]),
    "evo_decode_qkv_prep_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p]),
    "evo_decode_attn_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_size_t, C.c_void_p]),
    "evo_advance_position": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "evo_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_uint64, C.c_uint64, C.c_void_p]),
    "evo_sample_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "evo_advance_counters": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "evo_sample_step_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "evo_ragged_advance": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "evo_unembed_score_workspace": (C.c_size_t, [C.c_int64, C.c_int]),
    "evo_unembed_score": (C.c_int, [C.POINTER(ScoreParams), C.c_void_p]),
    "evo_tokenize_pad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "evo_logprobs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
}

_lib = None


def lib():
    """The loaded library (loads on first use; raises if it is not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EvoError(f"{LIB_PATH} is missing: the CUDA extension is not built (run `python -m evo_b200.build`). "
                           "evo_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().evo_last_error()
        raise EvoError(f"{what or 'evo_b200'} failed (rc={rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
