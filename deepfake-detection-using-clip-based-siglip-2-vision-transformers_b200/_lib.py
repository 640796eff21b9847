"""ctypes binding of libdfd.so (the C ABI declared in include/dfd.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C csrc``.  There is no CPU
fallback: if the shared object is missing, or a compute entry point is called without a CUDA device,
the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = _PKG_DIR / "libdfd.so"


class DfdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libdfd error {code}: {msg}")
        self.code = code


class GemmEpilogue(C.Structure):
    _fields_ = [
        ("bias", C.c_void_p),
        ("act", C.c_int),
        ("pos", C.c_void_p),
        ("pos_rows", C.c_int),
        ("residual", C.c_void_p),
        ("ldr", C.c_int64),
        ("ln_rowstats", C.c_void_p),
        ("ln_colsum", C.c_void_p),
        ("ln_dim", C.c_int),
        ("ln_eps", C.c_float),
        ("stats_out", C.c_void_p),
        ("residual_op", C.c_int),
        ("ln_parts", C.c_int),
        ("residual_lo", C.c_void_p),
    ]


class DenseLayer(C.Structure):
    _fields_ = [("w", C.c_void_p), ("b", C.c_void_p), ("out_dim", C.c_int), ("in_dim", C.c_int), ("act", C.c_int)]


class HeadWeights(C.Structure):
    _fields_ = [
        ("kind", C.c_int),
        ("dim", C.c_int),
        ("norm_eps", C.c_float),
        ("ln_eps", C.c_float),
        ("se_w1", C.c_void_p), ("se_b1", C.c_void_p), ("se_w2", C.c_void_p), ("se_b2", C.c_void_p),
        ("ln_g", C.c_void_p), ("ln_b", C.c_void_p),
        ("n_layers", C.c_int),
        ("layers", DenseLayer * 6),
    ]


class ScoreWeights(C.Structure):
    _fields_ = [
        ("gen", C.c_int),
        ("g1_ln_w", C.c_void_p), ("g1_ln_b", C.c_void_p), ("g1_w1", C.c_void_p),
        ("g1_b1", C.c_void_p), ("g1_w2", C.c_void_p), ("g1_b2", C.c_void_p),
        ("g1_fc_w", C.c_float * 2), ("g1_fc_b", C.c_float), ("freq_temp", C.c_float),
        ("g2_mean", C.c_void_p), ("g2_std", C.c_void_p), ("g2_alpha", C.c_void_p),
        ("g2_beta", C.c_void_p), ("g2_gates", C.c_void_p),
        ("g2_blk", (C.c_void_p * 6) * 2),
        ("g2_head_w", C.c_void_p), ("g2_head_b", C.c_void_p),
        ("g2_temp", C.c_float),
        ("f2_w0", C.c_void_p), ("f2_b0", C.c_void_p), ("f2_w1", C.c_void_p), ("f2_b1", C.c_void_p),
        ("f2_temp", C.c_float),
        ("coral_cuts", C.c_float * 4),
        ("coral_temp", C.c_float),
    ]


class Scores(C.Structure):
    _fields_ = [
        ("z_freq", C.c_void_p), ("z", C.c_void_p), ("z_scaled", C.c_void_p), ("p_raw", C.c_void_p),
        ("risk_probs", C.c_void_p), ("p_coral", C.c_void_p), ("entropy", C.c_void_p),
        ("p_blend", C.c_void_p), ("risk_idx", C.c_void_p),
    ]


class EngineConfig(C.Structure):
    _fields_ = [
        ("image_size", C.c_int), ("patch", C.c_int), ("hidden", C.c_int), ("inter", C.c_int),
        ("layers", C.c_int), ("heads", C.c_int), ("gelu_tanh", C.c_int), ("ln_eps", C.c_float),
        ("fuse_ln", C.c_int),
    ]


_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_F = C.c_float

# name -> (restype, argtypes); must list every DFD_API symbol of include/dfd.h (tests check this).
SIGNATURES = {
    "dfd_last_error": (C.c_char_p, []),
    "dfd_version": (_I, []),
    "dfd_launch_count": (_L, []),
    "dfd_gemm_bf16": (_I, [_P, _L, _P, _L, _P, _L, _I, _I, _I, C.POINTER(GemmEpilogue), _P]),
    "dfd_gemm_schedule": (_I, [_I, _I, _I, _I, _I]),
    "dfd_gemm_last_variant": (_I, []),
    "dfd_gemm_variant_launches": (_L, [_I]),
    "dfd_gemm_bf16_tile": (_I, [_P, _L, _P, _L, _P, _L, _I, _I, _I, C.POINTER(GemmEpilogue), _I, _P]),
    "dfd_layernorm_bf16": (_I, [_P, _L, _P, _P, _L, _P, _P, _I, _I, _F, _P]),
    "dfd_attention_bf16": (_I, [_P, _L, _P, _L, _I, _I, _I, _I, _F, _P]),
    "dfd_attention_bf16_impl": (_I, [_P, _L, _P, _L, _I, _I, _I, _I, _F, _I, _P]),
    "dfd_patchify": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _L, _P]),
    "dfd_map_attention_bf16": (_I, [_P, _L, _P, _P, _L, _I, _I, _I, _I, _F, _P]),
    "dfd_attention_probs": (_I, [_P, _L, _I, _I, _I, _I, _F, _I, _P, _P]),
    "dfd_attention_rollout": (_I, [_P, _P, _I, _I, _I, _I, _F, _I, _I, _P, _P, _P]),
    "dfd_head_fwd": (_I, [C.POINTER(HeadWeights), _P, _L, _I, _P, _P, _P, _P, _P]),
    "dfd_freq_features": (_I, [_P, _I, _P, _F, _I, _P, _P, _P]),
    "dfd_freq_scratch_bytes": (_L, [_I]),
    "dfd_resample_ksize": (_I, [_I, _I, _I]),
    "dfd_resample_coeffs_host": (_I, [_I, _I, _I, _P, _P, _P]),
    "dfd_gray256_scratch_bytes": (_L, [_I, _I, _I]),
    "dfd_resize_u8": (_I, [_P, _L, _L, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _I, _P, _P, _P]),
    "dfd_gray256": (_I, [_P, _L, _L, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _I, _P, _P, _P]),
    "dfd_clahe_scratch_bytes": (_L, [_I, _I]),
    "dfd_clahe_u8": (_I, [_P, _I, _I, _I, _I, _P, _P, _P]),
    "dfd_score_epilogue": (_I, [C.POINTER(ScoreWeights), _P, _P, _P, _I, C.POINTER(Scores), _P]),
    "dfd_fusion_fwd_bwd": (_I, [_P, _P, _P, _P, _I, _F, _P, _P, _P, _P]),
    "dfd_dwconv3x3_bf16": (_I, [_P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _P]),
    "dfd_seg_head_upsample": (_I, [_P, _L, _P, _F, _I, _I, _I, _I, _I, _P, _P, _P]),
    "dfd_linear_small": (_I, [_P, _L, _P, _P, _P, _I, _I, _I, _P]),
    "dfd_freqmlp_fwd_bwd": (_I, [_P, _P, _P, _P, _P, _I, _F, _F, C.c_uint32, _P, _P, _P, _P]),
    "dfd_engine_create": (_I, [C.POINTER(EngineConfig), _I, _I, C.POINTER(_P)]),
    "dfd_engine_destroy": (_I, [_P]),
    "dfd_engine_set_tensor": (_I, [_P, C.c_char_p, _P, _I, _I, C.POINTER(_L), _I]),
    "dfd_engine_finalize": (_I, [_P]),
    "dfd_engine_forward": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "dfd_engine_workspace_bytes": (_L, [_P]),
    "dfd_engine_set_hidden_tap": (_I, [_P, _P]),
    "dfd_engine_set_attention_tap": (_I, [_P, _P, _I, _P]),
    "dfd_engine_set_graphs": (_I, [_P, _I]),
    "dfd_engine_set_precise_residual": (_I, [_P, _I]),
    "dfd_engine_graph_replays": (C.c_int64, [_P]),
    "dfd_engine_profile": (_I, [_P, _I]),
    "dfd_engine_profile_read": (_I, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
}

_lib = None


def load() -> C.CDLL:
    """Load libdfd.so (once).  Raises if it has not been built — there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("DFD_LIB", LIB_PATH))   # development hook: A/B a second build of the same ABI
    if not path.exists():
        raise ImportError(
            f"{path} not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            f"or `make -C {_PKG_DIR / 'csrc'}`. There is no CPU fallback."
        )
    lib = C.CDLL(os.fspath(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        msg = load().dfd_last_error()
        raise DfdError(code, msg.decode("utf-8", "replace") if msg else "")


def ptr(t) -> int:
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
