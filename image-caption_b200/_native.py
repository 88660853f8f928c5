"""ctypes binding of libicap.so (include/icap.h).  There is deliberately NO fallback: if the
library is missing or the device is not sm_100 every call raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libicap.so")

F32, BF16 = 0, 1
EPI_NONE, EPI_RELU, EPI_RELU_MASK, EPI_ROWSTATS = 0, 1, 2, 3
EPI_B_STATIC = 16      # flag: B / bias are weights the preceding kernel of the stream does not write

P, I, L, F, U = c_void_p, c_int, c_int64, c_float, c_uint64

# name -> argtypes, in the order of include/icap.h
SIGNATURES = {
    "icap_version": [],
    "icap_sm_check": [I],
    "icap_set_pdl": [I],
    "icap_gemm": [I, I, I, L, L, L, P, L, P, L, P, L, I, P, I, P, L, I, I, P],
    "icap_reload_env": [],
    "icap_set_gemm_sms": [I],
    "icap_debug_trace": [P, I],
    "icap_mha_fwd": [I, L, L, L, L, L, L, P, L, P, L, P, L, P, L, P, I, F, U, P, P, P],
    "icap_mha_bwd": [I, L, L, L, L, L, L, P, L, P, L, P, L, P, L, P, L, P, L, P, L, P, I, F, U, P, P],
    "icap_add_ln_fwd": [I, I, L, L, P, P, L, P, P, P, P, P, P, I, F, U, P, F, P],
    "icap_add_ln_bwd": [I, L, L, P, P, P, P, P, P, P, P, P, P, P, P, F, U, P, P],
    "icap_add_ln_bwd_rows": [I, L, L, P, P, P, P, P, P, P, P, P, F, U, P, P],
    "icap_add_ln_bwd_params": [I, L, L, P, P, P, P, P, P, P, P, P, P, P, P],
    "icap_gemm_ln": [L, L, L, P, L, P, L, P, P, L, P, P, P, P, L, P, L, P, P, F, F, U, P, P],
    "icap_xent": [I, L, L, P, L, P, I, P, P, I, P],
    "icap_xent_finalize": [L, P, P, I, P, P],
    "icap_argmax": [I, L, L, P, L, P, L, P, P],
    "icap_sample_tokens": [I, L, L, P, L, F, U, P, L, L, P, P, L, I, I, P],
    "icap_beam_select": [I, L, L, L, P, L, P, L, P, P, P, P, I, P, L, P],
    "icap_beam_reorder": [L, L, L, L, P, P, P, P, P, P, P],
    "icap_decode_embed_ln": [I, L, L, L, L, L, P, P, P, P, P, P, P, P, P, P, P, P, I, F, P],
    "icap_log_softmax_argmax": [L, L, P, L, P, L, P, P],
    "icap_log_softmax_bwd": [L, L, P, L, P, L, P, L, P],
    "icap_mha_decode": [I, L, L, L, L, L, P, L, P, L, P, L, L, P, L, P, L, P, L, I, P, L, P, P],
    "icap_mha_decode_self": [I, L, L, L, L, L, P, L, P, P, L, P, L, P, L, L, P, L, P, L, P, L, I, L, P],
    "icap_copy2d": [P, I, L, P, I, L, L, L, I, P],
    "icap_rows_gather_add": [I, P, L, P, L, P, L, L, L, L, L, L, P],
    "icap_rows_segsum_add": [I, P, L, P, L, L, L, L, L, L, P],
    "icap_region_valid": [P, L, L, P, P, P],
    "icap_gather_regions": [I, P, P, L, P, I, L, L, L, P, P, P, P, P],
    "icap_caption_prep": [P, I, L, L, I, P, P, P, P, P, P, P],
    "icap_embed_fwd": [I, I, P, L, L, L, P, P, P, I, P],
    "icap_embed_bwd": [I, P, L, L, I, P, P, P],
    "icap_colsum": [I, L, L, P, L, P, P],
    "icap_adam_step": [L, P, P, P, P, P, F, F, F, F, P, I, P, F, P],
    "icap_step_tick": [P, P],
    "icap_scale": [P, L, P, F, P],
    "icap_reciprocal": [P, P, F, P],
    "icap_im2col_nhwc": [I, P, L, L, L, L, I, I, I, I, P, L, P],
    "icap_bn_scale_shift": [I, P, L, L, P, P, P, P, P, F, F, I, P, P, P],
    "icap_bn_act": [I, P, L, L, P, P, P, I, P, P],
    "icap_maxpool_nhwc": [I, P, L, L, L, L, I, I, I, P, P],
    "icap_avgpool_nhwc": [I, P, L, L, L, P, P],
    "icap_p2p_barrier": [P, I, I, P, P, P],
    "icap_p2p_reduce_scatter": [P, I, I, L, L, I, P],
    "icap_p2p_all_gather": [P, I, I, L, L, I, P],
    "icap_p2p_allreduce_nvls": [P, I, I, L, L, I, P],
    "icap_caption_cook": [P, I, L, L, L, P, P, P, P, P, P],
    "icap_caption_df": [L, P, L, P, P, P, P, L, P, P],
    "icap_caption_ref_prep": [L, L, P, P, P, L, P, P, L, P, P],
    "icap_caption_score": [P, I, L, L, L, P, L, P, L, P, P, P, P, P, P, P, P, L, P, P, F, F, P, P],
}


class IcapError(RuntimeError):
    pass


_lib = None
launch_count = 0          # number of C-ABI kernel-launching calls made by this process (bench: gpu_launches)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IcapError(f"{LIB_PATH} is missing: run `python __graft_entry__.py build` "
                            "(image-caption_b200 has no CPU / PyTorch fallback)")
        l = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = c_int
        l.icap_last_error.argtypes = []
        l.icap_last_error.restype = c_char_p
        _lib = l
    return _lib


def last_error() -> str:
    return lib().icap_last_error().decode("utf-8", "replace")


call_log = None           # profiling: when a list, every call is appended as (name, args) -- see tools/step_breakdown.py


def call(name: str, *args) -> None:
    """Invoke an entry point; raise IcapError on a non-zero return code."""
    global launch_count
    if call_log is not None:
        call_log.append((name, args))
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise IcapError(f"{name} failed (rc={rc}): {last_error()}")
    launch_count += 1
