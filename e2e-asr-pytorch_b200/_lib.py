"""ctypes binding of libe2e_asr_b200.so (include/e2e_asr_b200.h).

There is NO CPU fallback: if the shared object is missing (and cannot be built)
or CUDA is unavailable, every entry point raises.
"""
import ctypes
import os

from . import build as _build

c_int, c_float, c_void_p = ctypes.c_int, ctypes.c_float, ctypes.c_void_p

# mirrors of the header's constants
CTC_LOGZERO = -100000000.0
DEC_LOG_ZERO = -10000000.0
STATUS_PREFIX_TOO_LONG = 1
STATUS_TOKEN_NOT_CAND = 2
PREFIX_FULL = 1
PREFIX_SKIP_DEAD_ROWS = 2
PREFIX_FAST_MATH = 4
PREFIX_LIBM_MATH = 8
PREFIX_ROW_COPIES = 16
PREFIX_POLY_MATH = 32
PREFIX_POLY_ESTRIN = 64
BEAM_USE_CTC = 1
BEAM_USE_LM = 2

# name -> (restype, argtypes); kept in one table so tests can check the export list
SIGNATURES = {
    "e2e_last_error": (ctypes.c_char_p, []),
    "e2e_abi_version": (c_int, []),
    "e2e_padded_vocab": (c_int, [c_int]),
    "e2e_launch_count": (ctypes.c_longlong, []),
    "e2e_add_launch_count": (None, [ctypes.c_longlong]),
    "e2e_ctc_log_softmax": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "e2e_ctc_init_state": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "e2e_ctc_prefix_score": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                     c_void_p, c_int,
                                     c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "e2e_ctc_prefix_step_supported": (c_int, [c_int, c_int, c_int]),
    "e2e_ctc_prefix_step": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                    c_void_p, c_int,
                                    c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_int, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "e2e_beam_candidates": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "e2e_emb_fuse_candidates": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                        c_void_p, c_int, c_float, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "e2e_beam_combine_prune": (c_int, [c_void_p, c_int, c_void_p,
                                       c_void_p, c_int,
                                       c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_int,
                                       c_void_p, c_void_p,
                                       c_float, c_float, c_float, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p,
                                       c_void_p,
                                       c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "e2e_attention_loc_full": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_float, c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p]),
    "e2e_attention_loc_heads_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "e2e_attention_loc_heads": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_float, c_float, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                        c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "e2e_lstm_split_rows": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_int, c_int, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p]),
    "e2e_lstm_split_rows_multi": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "e2e_lstm_cell": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                              c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p]),
    "e2e_lstm_split_rows_f16x2": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_int, c_int, c_void_p, ctypes.c_longlong, c_int, c_int,
                                          c_float, c_void_p]),
    "e2e_lstm_split_rows_multi_f16x2": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_int, c_float, c_void_p]),
    "e2e_lstm_cell_f16x2": (c_int, [c_void_p, ctypes.c_longlong, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_float, c_void_p]),
    "e2e_gru_cell": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                             c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p]),
    "e2e_gru_cell_f16x2": (c_int, [c_void_p, ctypes.c_longlong, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                   c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_float, c_void_p]),
    "e2e_conv3x3_unfold_split": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_longlong, c_int, c_void_p, c_void_p]),
    "e2e_conv_bias_relu_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_longlong,
                                        ctypes.c_longlong, c_void_p]),
    "e2e_conv3x3_igemm_supported": (c_int, [c_int, c_int]),
    "e2e_conv3x3_igemm": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "e2e_lstm_sequence": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int,
                                  c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "e2e_gru_sequence": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_int, c_int, c_int, c_int,
                                 c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "e2e_packed_subsample_ln": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p,
                                        c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p]),
    "e2e_conv1_direct": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p, c_void_p]),
    "e2e_conv_bias_relu_mask_pool": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "e2e_conv1_direct_amax": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                      c_void_p, c_void_p, c_void_p]),
    "e2e_conv3x3_unfold_split_f16x2": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_longlong, c_int, c_void_p,
                                               c_void_p, c_void_p]),
    "e2e_conv_bias_relu_mask_scaled": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_longlong,
                                               ctypes.c_longlong, c_void_p, c_float, c_void_p, c_void_p]),
    "e2e_conv_bias_relu_mask_pool_scaled": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float,
                                                    c_void_p, c_void_p]),
    "e2e_nbest_pack_ragged": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "e2e_copy_rows_h2d": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "e2e_beam_finalize": (c_int, [c_int, c_int, c_void_p,
                                  c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_int,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_void_p]),
}

_lib = None


class E2EError(RuntimeError):
    pass


def load():
    """Load (building first if needed) the shared object; never falls back."""
    global _lib
    if _lib is None:
        path = os.environ.get("E2E_ASR_B200_LIB")          # tuning builds (tools/): an explicit library, never a fallback
        if not path:
            path = _build.LIB_PATH
            if _build.stale():
                path = _build.build()
        lib = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if a declared symbol is missing
            fn.restype, fn.argtypes = res, args
        if lib.e2e_abi_version() != 1:
            raise E2EError("libe2e_asr_b200.so ABI version mismatch")
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise E2EError("libe2e_asr_b200: rc=%d: %s" % (rc, load().e2e_last_error().decode()))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise E2EError("libe2e_asr_b200 has no CPU path: tensor on %s" % t.device)
