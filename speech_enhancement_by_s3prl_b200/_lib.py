"""ctypes binding of ``libse_b200.so`` (the C ABI of include/se_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc; if that is
impossible, or a call fails, a ``RuntimeError`` is raised (the reference's OOM /
RuntimeError handling at runner.py:504-508, 605-611 keeps working on top of it).
"""
import ctypes
import os
import threading

from . import build as _build

_lock = threading.Lock()
_lib = None

c_f = ctypes.c_void_p          # device pointers travel as integers
i64 = ctypes.c_int64
c_int = ctypes.c_int
c_float = ctypes.c_float
c_double = ctypes.c_double

_SIGNATURES = {
    "se_version": [],
    "se_last_error": [ctypes.c_char_p, c_int],
    "se_prepare": [c_int],
    "se_set_option": [c_int, c_int],
    "se_set_trace": [c_f],
    "se_stft": [c_f, i64, i64, i64, c_int, c_int, c_f, c_float, c_f, c_f, c_f, c_f],
    "se_stft_strided": [c_f, i64, i64, i64, c_int, c_int, c_f, c_float, c_f, c_f, c_f, i64, c_f],
    "se_istft": [c_f, c_f, i64, i64, c_int, c_int, c_f, c_f, i64, i64, c_f],
    "se_mask_istft": [c_f, c_f, i64, c_f, c_f, i64, i64, c_int, c_int, c_f, c_f, i64, i64, c_f, c_int, c_f],
    "se_mask_istft_strided": [c_f, c_f, i64, c_f, i64, c_f, i64, i64, c_int, c_int, c_f, c_f, i64, i64, c_f, c_int, c_f],
    "se_mask_istft_ex": [c_f, c_f, i64, c_f, i64, c_f, i64, i64, c_int, c_int, c_f, c_f, i64, i64, c_f, c_int, c_f],
    "se_stft_features": [c_f, i64, i64, i64, c_int, c_int, c_f, c_float, c_int, c_f, i64, c_f, i64, c_int, c_f],
    "se_stft_features2": [c_f, i64, i64, i64, c_int, c_int, c_f, c_float, c_f, c_f, i64, c_f, i64, c_int, c_f],
    "se_stft_features_pair_supported": [c_int, c_int],
    "se_stft_features_pair": [c_f, i64, i64, i64, i64, c_int, c_int, c_f, c_float, c_f, c_f, i64, c_f, i64, c_int, c_f],
    "se_linear_head_bwd_fused": [c_f, i64, c_f, i64, c_float, c_f, c_f, i64, i64, i64, i64, i64, c_int, c_f, i64, c_f, c_f, c_f],
    "se_adam_clip_step": [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_int, c_float, c_float,
                          c_float, c_float, c_float, c_float, c_f, c_f, c_f],
    "se_adam_clip_step_mirror": [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_int, c_float,
                                 c_float, c_float, c_float, c_float, c_float, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, c_int,
                                 c_f, c_f, c_f],
    "se_sisdr_mask_step": [c_f, i64, c_f, i64, c_f, i64, c_f, i64, i64, i64, i64, c_float, c_f, c_int, c_f, c_f, c_f, i64, c_f],
    "se_linear_head_bwd_sisdr_supported": [i64, i64, i64, i64, i64, i64, i64, i64],
    "se_linear_head_bwd_sisdr": [c_f, i64, c_f, i64, c_float, c_f, i64, c_f, i64, c_f, i64, c_f, i64, c_f, c_float, i64, i64, i64, i64, c_int,
                                 c_f, i64, c_f, c_f, c_f],
    "se_head_grad_embeddings_sisdr_supported": [i64, i64, i64, i64, i64, i64, i64, i64],
    "se_head_grad_embeddings_sisdr": [c_f, i64, c_f, i64, c_float, c_f, i64, c_f, i64, c_f, i64, c_f, i64, c_f, c_float, i64, i64, i64, i64,
                                      c_int, c_f, i64, c_f, c_f],
    "se_head_grad_embeddings_workspace": [i64, i64, i64, i64],
    "se_head_grad_embeddings": [c_f, i64, c_f, c_f, c_f, i64, c_float, c_f, c_f, i64, i64, i64, i64, i64, c_int, c_f, i64, c_f, c_f],
    "se_match_scores": [c_f, i64, c_f, i64, i64, c_float, c_f, c_f, c_f, c_f],
    "se_sisdr_mask_fwd": [c_f, i64, c_f, i64, c_f, i64, c_f, i64, i64, i64, c_float, c_f, c_f, c_f],
    "se_sisdr_mask_bwd": [c_f, i64, c_f, i64, c_f, i64, c_f, i64, i64, i64, c_float, c_f, c_f, c_f, i64, c_f],
    "se_feature_sums": [c_f, i64, i64, i64, i64, c_f, i64, c_f],
    "se_linear_head_fused_supported": [i64, i64, i64, i64, i64, i64, i64],
    "se_linear_head_fused": [c_f, i64, c_f, i64, c_float, c_f, i64, c_f, i64, i64, i64, i64, c_int, c_f, i64, c_f],
    "se_finalize_metrics": [c_f, c_f, i64, i64, c_float, c_f, i64, i64, c_f, c_f, c_f, c_f],
    "se_finalize_metrics_acc": [c_f, c_f, i64, i64, c_float, c_f, i64, i64, c_f, c_f, c_f, c_f, c_f],
    "se_sisdr_spec_fwd": [c_f, c_f, c_f, i64, i64, i64, c_float, c_f, c_f, c_f],
    "se_sisdr_spec_bwd": [c_f, c_f, c_f, i64, i64, i64, c_float, c_f, c_f, c_f, c_f],
    "se_l1_logspec_fwd": [c_f, c_f, c_f, i64, i64, i64, c_float, c_f, c_f],
    "se_l1_logspec_bwd": [c_f, c_f, c_f, i64, i64, i64, c_float, c_double, c_f, c_f, c_f],
    "se_mix_batch": [c_f, i64, c_f, c_f, i64, c_f, c_f, i64, i64, c_float, c_float, c_f, c_f, c_f],
    "se_wsd_fwd": [c_f, c_f, c_f, c_f, i64, i64, i64, c_float, c_float, c_float, c_f, c_f, c_f, c_f, c_f],
    "se_wsd_bwd": [c_f, c_f, c_f, c_f, i64, i64, i64, c_float, c_float, c_float, c_f, c_f, c_f, c_f, c_f],
    "se_wsd_energy": [c_f, i64, i64, i64, i64, c_f, c_f, c_f],
    "se_wsd_mask_step": [c_f, i64, c_f, i64, c_f, i64, c_f, i64, i64, i64, i64, c_float, c_float, c_float, c_f, c_f, c_f, c_int, c_f, c_f,
                         c_f, i64, c_f],
    "se_mask_istft_wsd_supported": [c_int, c_int],
    "se_mask_istft_wsd": [c_f, c_f, i64, c_f, i64, c_f, i64, i64, c_int, c_int, c_f, c_f, i64, i64, c_f, c_f, c_f, c_int, c_f],
    "se_wsd_eval_finish": [c_f, c_f, i64, i64, c_float, c_float, c_float, c_f, c_f, c_f, c_f],
    "se_linear_head_bwd_wsd_supported": [i64, i64, i64, i64, i64, i64, i64, i64],
    "se_linear_head_bwd_wsd": [c_f, i64, c_f, i64, c_float, c_f, i64, c_f, i64, c_f, i64, c_f, i64, c_f, c_f, c_float, c_float, c_float, i64,
                               i64, i64, i64, c_int, c_f, i64, c_f, c_f, c_f],
    "se_sisdr_wave": [c_f, i64, c_f, i64, c_f, i64, i64, c_float, c_f, c_f, c_f],
    "se_stoi_workspace": [i64, i64, c_int],
    "se_stoi": [c_f, i64, c_f, i64, c_f, i64, i64, c_int, c_f, i64, c_f, c_f, c_f, c_f, c_f],
    "se_masked_normalize_db": [c_f, i64, c_f, i64, i64, c_f, c_f, i64, c_float, c_f, c_f, i64, c_f],
    "se_length_masks": [c_f, i64, i64, c_f, c_f],
    "se_cmvn_stats": [c_f, i64, i64, i64, c_f, c_f, c_f],
    "se_linear_head_fwd": [c_f, c_f, c_f, c_float, c_f, c_f, i64, i64, i64, i64, c_int, c_f, c_f, c_f, c_int, c_f],
    "se_cmvn_stats_strided": [c_f, i64, i64, i64, i64, c_f, c_f, i64, c_f],
    "se_linear_head_fwd_strided": [c_f, i64, c_f, c_f, i64, c_float, c_f, i64, c_f, i64, i64, i64, i64, c_int, c_f, c_f, c_f, i64, c_int, c_f],
    "se_linear_head_bwd": [c_f, c_f, c_f, c_float, c_f, c_f, c_f, i64, i64, i64, i64, c_int, c_f, c_f, c_f],
    "se_linear_head_bwd_tc_workspace": [i64, i64, i64, i64],
    "se_linear_head_bwd_tc": [c_f, i64, c_f, c_f, i64, c_float, c_f, c_f, i64, i64, i64, i64, i64, c_int, c_f, i64, c_f, c_f, c_f],
    "se_mel": [c_f, i64, i64, c_f, i64, c_int, c_float, c_f, i64, c_f],
    "se_delta": [c_f, i64, i64, i64, c_int, c_f],
    "se_mel_features": [c_f, i64, i64, i64, i64, c_f, c_f, i64, c_int, c_float, c_int, c_f, i64, c_f, c_f],
    "se_cmvn_apply_sums": [c_f, i64, i64, i64, c_f, c_float, c_f],
    "se_cmvn_apply": [c_f, i64, i64, i64, c_f, c_f, c_float, c_f],
    "se_h2d_channels": [c_f, i64, i64, i64, i64, c_f, c_f],
    "se_h2d_channels_pcm16": [c_f, i64, i64, i64, i64, c_f, c_f, c_f],
}

EXPORTS = tuple(_SIGNATURES)


def library_path():
    return _build.LIB_PATH


def load():
    """Load (building first if stale/missing) and return the ctypes library."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            path = os.environ.get("SE_B200_LIB") or _build.LIB_PATH      # override: experiment builds
            if path == _build.LIB_PATH and _build.is_stale():
                try:
                    path = _build.build_library()
                except Exception as exc:           # a stale library may not match _SIGNATURES: never load it silently
                    raise RuntimeError(f"libse_b200.so is missing or older than csrc/ and cannot be rebuilt: {exc}") from exc
            lib = ctypes.CDLL(path)
            for name, argtypes in _SIGNATURES.items():
                fn = getattr(lib, name)            # AttributeError if the symbol is not exported
                fn.argtypes = argtypes
                fn.restype = i64 if name.endswith("_workspace") else c_int
            _lib = lib
    return _lib


def last_error():
    buf = ctypes.create_string_buffer(512)
    load().se_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"libse_b200 {what} failed (code {rc}): {last_error()}")
