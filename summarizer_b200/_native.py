"""ctypes binding of libsummarizer_b200.so (the C ABI declared in include/summarizer_b200.h).

There is no CPU fallback: if the shared library is missing, or the device is not an sm_100
part, every entry point raises.  PyTorch is used only as the device-memory container
(``tensor.data_ptr()``) and for the current stream.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsummarizer_b200.so")

SMZ_METHOD = {"knapsack": 0, "rank": 1}
SMZ_STATUS_VALUE_RANGE = 1
SMZ_STATUS_INTERVALS = 2
SMZ_STATUS_WEIGHT_RANGE = 4
FSCORE_MAX_USERS = 1024

# struct smz_video_desc (include/summarizer_b200.h) — 104 bytes
VIDEO_DESC = np.dtype([
    ("score_off", "<i8"), ("picks_off", "<i8"), ("seg_off", "<i8"), ("user_off", "<i8"),
    ("user_ld", "<i8"), ("summ_off", "<i8"), ("frame_off", "<i8"), ("mask_off", "<i8"),
    ("ucount_off", "<i8"),
    ("n_scores", "<i4"), ("n_picks", "<i4"), ("n_segs", "<i4"), ("n_users", "<i4"),
    ("n_frames", "<i4"), ("summ_len", "<i4"), ("capacity", "<i4"), ("reserved", "<i4"),
], align=True)
assert VIDEO_DESC.itemsize == 104

# struct smz_corr_desc — 48 bytes
CORR_DESC = np.dtype([("m_off", "<i8"), ("u_off", "<i8"), ("u_ld", "<i8"), ("rank_off", "<i8"),
                      ("n_frames", "<i4"), ("n_users", "<i4"), ("row0", "<i4"), ("reserved", "<i4")], align=True)
assert CORR_DESC.itemsize == 48
SMZ_METRIC = {"spearmanr": 0, "kendalltau": 1}

_P = C.c_void_p
_I = C.c_int
_L = C.c_int64

# name -> (restype, argtypes); must list every symbol the header declares
SIGNATURES = {
    "smz_version": (C.c_char_p, []),
    "smz_last_error": (C.c_char_p, []),
    "smz_device_check": (_I, []),
    "smz_profile_report": (None, []),
    "smz_select_workspace_bytes": (_I, [_I, _I, _I, _I, _I, C.POINTER(C.c_int64)]),
    "smz_select_shots": (_I, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "smz_knapsack": (_I, [_P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _L, _P]),
    "smz_fscore": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "smz_eval_batch": (_I, [_P, _I, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                            _P, _P, _P, _P, _P, _L, _P]),
    "smz_pack_summary": (_I, [_P, _I, _I, _P, _P, _P, _P]),
    "smz_upsample": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "smz_rank_correlation": (_I, [_P, _I, _I, _I, _P, _P, _I, _P, _P, _P, _P]),
    "smz_vasnet_workspace_bytes": (_I, [_P, _I, _I, _I, C.POINTER(C.c_int64)]),
    "smz_vasnet_set_exact_softmax": (None, [_I]),
    "smz_vasnet_launch_count": (_I, [_P, _I, _I, _I, C.POINTER(C.c_int64)]),
    "smz_vasnet_forward": (_I, [_P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P, _L, _P]),
    "smz_vasnet_backward": (_I, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "smz_mha_workspace_bytes": (_I, [_I, C.POINTER(C.c_int64)]),
    "smz_mha_forward": (_I, [_P, _L, _P, _I, _I, _I, _P, _L, _P, _L, _P]),
    "smz_transformer_workspace_bytes": (_I, [_P, _I, _I, C.POINTER(C.c_int64)]),
    "smz_transformer_forward": (_I, [_P, _I, _P, _I, _P, _I, _P, _P, _L, _P]),
    "smz_sumgan_att_selector_forward": (_I, [_P, _I, _P, _I, _P, _I, _P, _P, _L, _P]),
    "smz_dsn_pack_whh": (_I, [_P, _P, _P, _P, _P]),
    "smz_dsn_workspace_bytes": (_I, [_I, _I, _I, _I, C.POINTER(C.c_int64)]),
    "smz_dsn_forward": (_I, [_P, _I, _P, _I, _P, _I, _P, _P, _L, _P]),
    "smz_dsn_backward": (_I, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _L, _P]),
    "smz_dsn_reward_workspace_bytes": (_I, [_I, _I, C.POINTER(C.c_int64)]),
    "smz_dsn_reward": (_I, [_P, _I, _P, _I, _I, _I, _P, _P, _L, _P]),
    "smz_bernoulli_logprob": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "smz_bernoulli_logprob_backward": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "smz_host_pack_user_summary": (_I, [_P, _I, _P, _P, _P, _I]),
    "smz_fscore_packed": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "smz_pack_user_bits": (_I, [_P, _I, _P, _P, _P, _P]),
    "smz_kts_workspace_bytes": (_I, [_I, _I, _I, C.POINTER(C.c_int64)]),
    "smz_kts_gram": (_I, [_P, _I, _I, _I, _P, _P]),
    "smz_kts": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, C.c_double, _I, _P, _P, _P, _P, _L, _P]),
    "smz_lstm_seq_forward": (_I, [_P, _I, _P, _P]),
    "smz_lstm_seq_backward": (_I, [_P, _I, _P, _P]),
    "smz_lstm_decode_forward": (_I, [_P, _P, _P]),
    "smz_lstm_decode_backward": (_I, [_P, _P, _P]),
    "smz_cvt_bf16_multi": (_I, [_P, _P, _P, _I, _P]),
    "smz_split_bf16_multi": (_I, [_P, _P, _P, _P, _I, _P]),
    "smz_dropout_keep_masks": (_I, [_P, _P, _L, _P]),
    "smz_mse_loss": (_I, [_P, _P, _L, _P, _P, _P]),
    "smz_grad_sqnorm_workspace_floats": (_I, [_P, _I, C.POINTER(C.c_int64)]),
    "smz_grad_sqnorm": (_I, [_P, _I, _P, _P, _L, _P]),
    "smz_clip_grads": (_I, [_P, _I, _P, C.c_float, _P]),
    "smz_adam_step": (_I, [_P, _I, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _P]),
    "smz_gemm_bf16": (_I, [_I, _I, _P, _L, _P, _L, _P, _L, _I, _I, _I, C.c_float, _P, _P, _L, _I, _P]),
    "smz_gemm_bf16_split": (_I, [_I, _I, _P, _P, _L, _P, _P, _L, _P, _P, _L, _I, _I, _I, C.c_float, _P, _P, _L, _I, _P]),
    "smz_gemm_bf16_tn": (_I, [_P, _L, _P, _L, _P, _L, _I, _I, _I, C.c_float, _P, _P, _L, _I, _P]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Loads libsummarizer_b200.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C summarizer_b200/csrc).  summarizer_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().smz_last_error().decode("utf-8", "replace")
        raise NativeError(f"libsummarizer_b200 error {rc}: {msg}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_device():
    import torch
    if not torch.cuda.is_available():
        raise NativeError("summarizer_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    check(lib().smz_device_check())
