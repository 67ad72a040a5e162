"""ctypes binding of ``librllm_b200.so`` (the C ABI declared in ``include/rllm_b200.h``).

There is deliberately no Python / torch fallback: if the shared library is missing or a symbol
cannot be resolved, importing a product module that needs it raises ``NativeLibraryError``.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = _PKG_DIR / "lib" / "librllm_b200.so"
HEADER_PATH = _PKG_DIR.parent / "include" / "rllm_b200.h"

ABI_VERSION = 3
SEGMENT_PIECE = 64  # RLLM_B200_SEGMENT_PIECE: most input positions one warp of the tied-embedding fold sums

# estimator / mode ids (keep in sync with include/rllm_b200.h)
EST_GRPO, EST_REINFORCE, EST_RPP_BASELINE, EST_RLOO = 0, 1, 2, 3
AGG_TOKEN_MEAN, AGG_SEQ_MEAN_TOKEN_SUM, AGG_SEQ_MEAN_TOKEN_MEAN, AGG_SEQ_MEAN_TOKEN_SUM_NORM, AGG_SUM = 0, 1, 2, 3, 4
LOSS_NONE, LOSS_VANILLA, LOSS_TINKER_PPO, LOSS_TINKER_IS, LOSS_GPG, LOSS_CISPO, LOSS_GSPO, LOSS_DRO, LOSS_GEO_MEAN = 0, 1, 2, 3, 4, 5, 6, 7, 8
KL_OFF, KL_K1, KL_ABS, KL_MSE, KL_LOW_VAR = 0, 1, 2, 3, 4
SUM_NAMES = ("loss", "w_pg", "w_kl", "w_ent", "mask", "m_negd", "m_clip", "m_clip_lower", "m_ent", "m_logp", "m_ratio", "tokens")
N_SUMS = len(SUM_NAMES)

AGG_MODE_IDS = {
    "token-mean": AGG_TOKEN_MEAN,
    "seq-mean-token-sum": AGG_SEQ_MEAN_TOKEN_SUM,
    "seq-mean-token-mean": AGG_SEQ_MEAN_TOKEN_MEAN,
    "seq-mean-token-sum-norm": AGG_SEQ_MEAN_TOKEN_SUM_NORM,
    "sum": AGG_SUM,
}
KL_TYPE_IDS = {"kl": KL_K1, "k1": KL_K1, "abs": KL_ABS, "mse": KL_MSE, "k2": KL_MSE, "low_var_kl": KL_LOW_VAR, "k3": KL_LOW_VAR}
# clip_cov / kl_cov reuse the single-clip / unclipped importance-sampling algebra: their covariance-selected tokens enter
# through per-token weights / a per-token penalty prepared on the host side of the sweep (loss.py FusedLMHeadLoss._run_split)
LOSS_MODE_IDS = {"none": LOSS_NONE, "vanilla": LOSS_VANILLA, "ppo": LOSS_TINKER_PPO, "importance_sampling": LOSS_TINKER_IS, "gpg": LOSS_GPG, "cispo": LOSS_CISPO, "gspo": LOSS_GSPO,
                 "dro": LOSS_DRO, "geo_mean": LOSS_GEO_MEAN, "clip_cov": LOSS_TINKER_PPO, "kl_cov": LOSS_TINKER_IS}


class NativeLibraryError(RuntimeError):
    pass


class LossParams(C.Structure):
    _fields_ = [
        ("loss_mode", C.c_int32),
        ("kl_type", C.c_int32),
        ("clip_low", C.c_float),
        ("clip_high", C.c_float),
        ("clip_c", C.c_float),
        ("kl_coef", C.c_float),
        ("entropy_coef", C.c_float),
        ("inv_temperature", C.c_float),
        ("mode_coef", C.c_float),
    ]


_P = C.c_void_p
_I32, _I64, _F32, _F64 = C.c_int32, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); every symbol declared in include/rllm_b200.h must appear here.
SIGNATURES: dict[str, tuple] = {
    "rllm_b200_abi_version": (C.c_int, []),
    "rllm_b200_last_error": (C.c_char_p, []),
    "rllm_b200_device_sm_count": (C.c_int, []),
    "rllm_b200_set_tuning": (C.c_int, [_I32, _I32]),
    "rllm_b200_set_gemm_tuning": (C.c_int, [_I32]),
    "rllm_b200_get_gemm_tuning": (C.c_int, []),
    "rllm_b200_pack_prefix_merge": (
        C.c_int,
        [_I32, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    ),
    "rllm_b200_token_segments": (C.c_int, [_P, _I64, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "rllm_b200_embedding_grad_accumulate": (C.c_int, [_P, _I64, _P, _P, _P, _P, _I32, _P, _P, _I32, _P, _P, _I64, _I32, _I32, _P]),
    "rllm_b200_group_advantage": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _F64, _P, _P, _P, _P]),
    "rllm_b200_row_mask_counts": (C.c_int, [_P, _P, _P, _I32, _P, _P, _P]),
    "rllm_b200_row_loss_coef": (C.c_int, [_P, _I32, _I32, _F64, _F64, _F64, _P, _P]),
    "rllm_b200_rollout_correction": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _F32, _P, _P, _P]),
    "rllm_b200_loss_fwd_max_ctas": (C.c_int, []),
    "rllm_b200_logprob_loss_fwd": (
        C.c_int,
        [_P, _I64, _I32, _I32, _P, _P, _P, _P, _P, _P, _I32, _I64, _P, _P, _P, _P, _P, C.POINTER(LossParams), _P, _P, _P, _P, _P, _P, _P, _I32, _P],
    ),
    "rllm_b200_row_masked_mean_diff": (C.c_int, [_P, _P, _P, _P, _I32, _P, _P]),
    "rllm_b200_row_geo_mean_logratio": (C.c_int, [_P, _P, _P, _P, _P, _I32, _F32, _F32, _P, _P]),
    "rllm_b200_lm_head_gemm": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I32, _I32, _I32, _P]),
    "rllm_b200_adamw_max_partials": (C.c_int, []),
    "rllm_b200_adamw_step": (C.c_int, [_P, _P, _P, _P, _P, _I64, _F32, _F32, _F32, _F32, _F32, _I32, _F32, _F32, _I32, _P, _P, _P]),
    "rllm_b200_grad_sqnorm": (C.c_int, [_P, _I64, _P, _P, _P]),
    "rllm_b200_adamw_step_sharded": (C.c_int, [_P, _P, _P, _P, _P, _I64, _F32, _F32, _F32, _F32, _F32, _I32, _F32, _F32, _I32, _P, _P, _P]),
    "rllm_b200_debug_occupy_sms": (C.c_int, [_I32, _I64, _P]),
    "rllm_b200_gemm_bf16": (C.c_int, [_P, _I64, _I32, _P, _I64, _I32, _P, _I64, _I32, _I32, _I32, _I32, _P]),
    "rllm_b200_lm_head_fwd_stats": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I32, _I32, _I32, _P, _F32, _I32, _P, _I64, _P]),
    "rllm_b200_lm_head_fwd_exp_stats": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I32, _I32, _I32, _P, _F32, _I32, _P, _P, _I64, _P]),
    "rllm_b200_dh_from_exp": (C.c_int, [_P, _I64, _P, _I64, _P, _P, _P, _P, _F32, _F32, _I32, _I32, _I32, _P]),
    "rllm_b200_dw_exp_prepare": (C.c_int, [_P, _I64, _P, _I64, _P, _P, _P, _P, _F32, _F32, _P, _P, _I32, _P, _I64, _I32, _I32, _I32, _P]),
    "rllm_b200_lm_head_col_blocks": (C.c_int, [_I32]),
    "rllm_b200_logprob_loss_from_partials": (C.c_int, [_P, _I32, _I64, _I32, _I32, _I32] + [_P] * 6 + [_I32, _I64] + [_P] * 5 + [C.POINTER(LossParams)] + [_P] * 8),
    "rllm_b200_logprob_loss_bwd": (C.c_int, [_P, _I64, _I32, _I32, _P, _P, _P, _P, _P, _F32, _F32, _P, _I64, _I32, _P]),
}

_lib: C.CDLL | None = None


def build_hint() -> str:
    return "build it with `python -c 'import __graft_entry__ as g; g.build()'` or `make -C rllm_b200/csrc`"


def lib() -> C.CDLL:
    """Load (once) and return the native library; raises NativeLibraryError if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("RLLM_B200_LIB", LIB_PATH))
    if not path.exists():
        raise NativeLibraryError(f"native library not found at {path}; {build_hint()}")
    try:
        handle = C.CDLL(str(path))
    except OSError as e:  # e.g. libcudart missing
        raise NativeLibraryError(f"failed to load {path}: {e}") from e
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(handle, name)
        except AttributeError as e:
            raise NativeLibraryError(f"{path} does not export `{name}`; rebuild ({build_hint()})") from e
        fn.restype = restype
        fn.argtypes = argtypes
    if handle.rllm_b200_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI version mismatch: library {handle.rllm_b200_abi_version()} vs binding {ABI_VERSION}")
    _lib = handle
    return handle


def last_error() -> str:
    return lib().rllm_b200_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed: {last_error()}")


def ptr(t) -> int | None:
    """Device / host pointer of a torch tensor or numpy array (None passes NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def current_stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
