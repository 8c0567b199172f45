"""ctypes binding of libsn100.so (the C ABI declared in include/sn100.h).

There is NO fallback: if the library is missing or the device is not sm_100 every op raises.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int32, c_int64, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsn100.so")

OP_NT, OP_NN, OP_TN = 0, 1, 2
CELL_FACTORED, CELL_LSTM = 0, 1

_P = c_void_p
_I32, _I64, _F, _D = c_int32, c_int64, c_float, c_double

# name -> (restype, argtypes); must list EVERY symbol include/sn100.h declares
SIGNATURES = {
    "sn_version": (_I32, []),
    "sn_last_error": (c_char_p, []),
    "sn_device_info": (_I32, [_P, _P, _P, _P]),
    "sn_gather_pack_fwd": (_I32, [_P, _I64, _P, _I64, _P, _I64, _I32, _P, _P, _P, _I64, _P, _I64, _F, c_uint64, _P, _P, _I64, _P]),
    "sn_gather_pack_bwd": (_I32, [_P, _I64, _P, _I64, _P, _I64, _I32, _P, _P, _P, _I64, _P, _I64, _F, c_uint64, _P, _I64, _P, _P, _P]),
    "sn_gemm": (_I32, [_I32, _I64, _I64, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _F, _I32, _I64, _I64, _I64, _I64, _P]),
    "sn_gemm_bf16": (_I32, [_I32, _I64, _I64, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _F, _I32, _I64, _I64, _I64, _I64, _I64, _P]),
    "sn_gemm_bf16_splitk": (_I32, [_I32, _I64, _I64, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _F, _I32, _I64, _I64, _I64, _I64, _I64, _I32, _P]),
    "sn_gemm2_ws_bytes": (_I64, [_I64, _I64, _I32, _I32]),
    "sn_gemm2_bf16": (_I32, [_I32, _I64, _I64, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _F, _I32, _I64, _I64, _I64, _I64, _I64, _I32, _P, _I64, _I32, _P]),
    "sn_vocab_ws_bytes": (_I64, [_I64, _I64]),
    "sn_vocab_nll_fwd": (_I32, [_I64, _I64, _I64, _P, _I64, _P, _I64, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "sn_vocab_nll_bwd": (_I32, [_I64, _I64, _I64, _P, _I64, _P, _I64, _P, _P, _P, _P, _F, _P, _P, _I64, _P, _P, _P]),
    "sn_cast_bf16": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _I64, _P]),
    "sn_cast_bf16_ex": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _I64, _I32, _P]),
    "sn_colsum": (_I32, [_P, _I64, _I64, _I64, _P, _F, _P]),
    "sn_colsum_ex": (_I32, [_P, _I64, _I64, _I64, _P, _F, _I32, _P]),
    "sn_colsum_bf16_ex": (_I32, [_P, _I64, _I64, _I64, _P, _F, _I32, _P]),
    "sn_embed_plan": (_I32, [_P, _I64, _I32, _P, _P, _P, _I64, _I64, _P, _P]),
    "sn_embed_grad": (_I32, [_P, _I64, _P, _I64, _I32, _P, _P, _P, _I64, _P, _I64, _F, c_uint64, _P, _I64, _P, _P, _I32, _P]),
    "sn_adam_clamp_dev_ex": (_I32, [_P, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _F, _F, _F, _F, _I32, _P]),
    "sn_recur_ws_bytes": (_I64, [_I64, _I64]),
    "sn_recur_fwd": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sn_recur_bwd": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sn_recur_fwd_bf16": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _I32] + [_P] * 12),
    "sn_recur_bwd_bf16": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _I32] + [_P] * 11),
    "sn_recur_cl_max_clusters": (_I32, [_I64]),
    "sn_recur_fwd_cl": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _I32] + [_P] * 11),
    "sn_recur_bwd_cl": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _I32] + [_P] * 11),
    "sn_gate_wait": (_I32, [_P, _I64, _P]),
    "sn_cast_bf16_gate_interleave": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _P]),
    "sn_recur_fwd_gemm": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sn_recur_hprev": (_I32, [_P, _P, _P, _P, _I64, _I64, _P, _P]),
    "sn_recur_bwd_gemm": (_I32, [_I32, _I64, _I64, _P, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sn_softmax_nll": (_I32, [_P, _I64, _I64, _I64, _P, _P, _P, _I64, _F, _P, _P, _P, _P, _I64, _P]),
    "sn_colsum_bf16": (_I32, [_P, _I64, _I64, _I64, _P, _F, _P]),
    "sn_reduce_sum": (_I32, [_P, _I64, _F, _P, _P, _I32, _P]),
    "sn_adam_clamp": (_I32, [_P, _P, _P, _P, _I32, _P, _P, _P, _F, _F, _F, _F, _P]),
    "sn_adam_clamp_dev": (_I32, [_P, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _F, _F, _F, _F, _P]),
    "sn_enable_peer_access": (_I32, [_I32]),
    "sn_ipc_export": (_I32, [_P, _P, _P]),
    "sn_ipc_open": (_I32, [_P, _P]),
    "sn_ipc_close": (_I32, [_P]),
    "sn_dp_adam_fused": (_I32, [_I32, _I32, _P, _P, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _F, _F, _F, _F, _P]),
    "sn_dp_slot_elems": (_I64, [_I64, _I32]),
    "sn_dp_push": (_I32, [_I32, _I32, _P, _P, _I64, _I32, _P, _I32, _P, _I32, _P]),
    "sn_dp_adam_recv": (_I32, [_I32, _I32, _P, _P, _P, _I64, _I32, _P, _P, _I32, _P, _P, _I32, _P, _P, _P, _P, _P, _F, _F, _F, _F, _I32, _P]),
    "sn_att_step_fwd": (_I32, [_P, _P, _P, _P, _F, _P, _I64, _I64, _I64, _I64, _P, _I64, _P, _I64, _P]),
    "sn_att_step_bwd": (_I32, [_P, _P, _P, _P, _F, _P, _P, _I64, _P, _I64, _P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P]),
    "sn_att_step_fwd_b16": (_I32, [_P, _P, _P, _P, _F, _P, _I64, _I64, _I64, _I64, _P, _I64, _P, _I64, _P]),
    "sn_att_step_bwd_b16": (_I32, [_P, _P, _P, _P, _P, _P, _I64, _P, _I64, _P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _P]),
    "sn_mean_pixels": (_I32, [_P, _I64, _I64, _I64, _P, _P]),
    "sn_beam_split_ws_floats": (_I64, [_I32, _I32, _I32]),
    "sn_beam_step_split": (_I32, [_P, _I64, _I64, _I32, _I32, _I32, _I32, _I32] + [_P] * 14 + [_I32, _P, _I32, _P]),
    "sn_split_limbs_cols": (_I32, [_P, _I64, _I64, _I64, _I64, _P, _I64, _I32, _P]),
    "sn_split_limbs_rows": (_I32, [_P, _I64, _I64, _I64, _I64, _P, _I64, _I64, _I32, _P]),
    "sn_skinny_max_rows": (_I32, []),
    "sn_skinny_linear": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _I64, _I64, _I64, _P, _P, _I64, _P, _P]),
    "sn_decode_cell": (_I32, [_I32, _I64, _I64, _P, _I64, _I64, _P, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sn_decode_cell_groups": (_I32, [_I32, _I64, _I64, _P, _I64, _P, _I64, _I64, _I64, _P, _I64, _I64, _P, _I64, _P, _P,
                                     _P, _P, _P, _P, _P, _P, _P]),
    "sn_pool_nhwc_fwd": (_I32, [_P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P]),
    "sn_pool_nhwc_bwd": (_I32, [_P, _I64, _I64, _I64, _I64, _I64, _P, _P]),
    "sn_bn1d_fwd": (_I32, [_P, _I64, _I64, _P, _P, _P, _P, _F, _F, _I32, _P, _P, _P, _P]),
    "sn_bn1d_bwd": (_I32, [_P, _P, _I64, _I64, _P, _P, _P, _I32, _P, _P, _P, _P]),
    "sn_beam_step": (_I32, [_P, _I64, _I64, _I32, _I32, _I32, _I32, _I32] + [_P] * 15),
    "sn_bleu_counts": (_I32, [_P, _P, _I64, _P, _P, _P, _I32, _I64, _P, _P]),
    "sn_cider_df": (_I32, [_P, _P, _P, _I64, _I32, _I32, _I64, _P, _P, _I64, _P, _P]),
    "sn_cider_scores": (_I32, [_P, _P, _I64, _P, _P, _P, _I32, _D, _I32, _I64, _P, _P, _I64, _P, _P, _P]),
    "sn_cider_scores_rows": (_I32, [_P, _I64, _P, _I64, _I32, _P, _I64, _P, _P, _P, _I32, _D, _I32, _I64, _P, _P, _I64,
                                    _P, _P]),
    "sn_rouge_l": (_I32, [_P, _P, _I64, _P, _P, _P, _I32, _D, _P, _P]),
    "sn_rouge_l_rows": (_I32, [_P, _I64, _P, _I64, _I32, _P, _I64, _P, _P, _P, _I32, _D, _P, _P]),
    "sn_sample_step": (_I32, [_P, _I64, _I64, _I32, _I32, _I32, _D, _I32] + [_P] * 9),
}

_lib = None


def load():
    """Load libsn100.so and bind every exported symbol.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libsn100.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU or PyTorch fallback for this path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class SnError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        msg = load().sn_last_error()
        raise SnError("%s failed (rc=%d): %s" % (what or "libsn100 call", rc, msg.decode() if msg else "?"))


_dev_ok = {}


def require_device(device_index):
    """Hard error unless the current device is sm_100 (no multi-backend dispatch)."""
    if _dev_ok.get(device_index):
        return
    lib = load()
    sm = c_int32(); sh = c_int32(); ma = c_int32(); mi = c_int32()
    check(lib.sn_device_info(ctypes.byref(sm), ctypes.byref(sh), ctypes.byref(ma), ctypes.byref(mi)), "sn_device_info")
    _dev_ok[device_index] = (sm.value, sh.value, ma.value, mi.value)
