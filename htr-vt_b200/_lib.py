"""ctypes loader for the C-ABI CUDA library (include/htrvt.h).

There is NO CPU fallback: if libhtrvt_b200.so is missing or a call returns a negative status the
caller gets an exception.  Build with `python htr-vt_b200/build.py` (or __graft_entry__.build()).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhtrvt_b200.so")
_lib = None

ERRORS = {-1: "bad shape", -2: "bad alignment", -3: "wrong architecture (sm_100a only)",
          -4: "kernel launch failed", -5: "workspace missing or too small", -6: "CUDA driver entry point failed"}


class HtrvtError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HtrvtError(
                "htr-vt_b200: %s not found. The CUDA extension is mandatory (no CPU fallback); build it with "
                "`python htr-vt_b200/build.py`." % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        raise HtrvtError("%s failed: %s (status %d)" % (what, ERRORS.get(status, "unknown"), status))


_P, _I, _L, _F, _Z = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_size_t

SIGNATURES = {
    # name: (restype, argtypes)
    "htrvt_version": (_I, []),
    "htrvt_ctc_set_mode": (_I, [_I]),
    "htrvt_ctc_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "htrvt_ctc_loss_grad": (_I, [_P, _L, _L, _I, _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _L, _L, _P, _F, _P, _Z, _P]),
    "htrvt_ctc_fallback_count": (_L, []),
    "htrvt_ctc_flagged_count": (_L, []),
    "htrvt_line_prep_u8": (_I, [_P, _L, _I, _P, _I, _I, _I, _P, _P, _P, _F, _P]),
    "htrvt_edit_distance": (_I, [_P, _P, _I, _P, _P, _P, _I, _P, _I, _I, _P, _P]),
    "htrvt_greedy_decode": (_I, [_P, _L, _L, _I, _I, _I, _P, _I, _P, _P, _P, _P]),
    "htrvt_ctc_collapse": (_I, [_P, _I, _P, _P, _I, _I, _I, _P, _P, _P]),
    "htrvt_ctc_kbest_paths": (_I, [_P, _L, _L, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "htrvt_augment_lines": (_I, [_P, _L, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "htrvt_ctc_prefix_beam": (_I, [_P, _L, _L, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "htrvt_ctc_prefix_beam_lm": (_I, [_P, _L, _L, _P, _I, _I, _I, _I, _P, _L, _I, _P, _I, ctypes.c_double,
                                      ctypes.c_double, _P, _P, _P, _P, _P]),
    "htrvt_ctc_prefix_beam_lex": (_I, [_P, _L, _L, _P, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P, _L, _I, _P, _I,
                                       ctypes.c_double, ctypes.c_double, _P, _P, _P, _P, _P]),
    "htrvt_ctc_prefix_beam_lex_wlm": (_I, [_P, _L, _L, _P, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P, _L, _I, _P,
                                           _P, ctypes.c_double, ctypes.c_double, _P, _P, _P, _P, _P]),
    "htrvt_ctc_align_workspace_bytes": (_Z, [_I, _I, _I]),
    "htrvt_ctc_align": (_I, [_P, _L, _L, _I, _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _Z, _P]),
    "htrvt_set_pdl": (_I, [_I]),
    "htrvt_gemm_tn": (_I, [_P, _L, _P, _L, _I, _I, _I, _I, _P, _P, _L, _F, _P, _L, _P]),
    "htrvt_gemm_nn": (_I, [_P, _L, _P, _L, _I, _I, _I, _I, _P, _L, _F, _P, _P, _P]),
    "htrvt_wgrad_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "htrvt_linear_wgrad": (_I, [_P, _L, _P, _L, _I, _I, _I, _P, _I, _P, _Z, _P]),
    "htrvt_conv_fwd": (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P]),
    "htrvt_conv_fwd_stats_rows": (_I, [_I, _I, _I, _I, _I, _I]),
    "htrvt_conv_dgrad": (_I, [_P, _I, _I, _I, _I, _P, _P, _I, _I, _I, _I, _P, _I, _P]),
    "htrvt_transpose_px": (_I, [_P, _P, _L, _I, _I, _P]),
    "htrvt_conv_wgrad": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _I, _P, _Z, _P]),
    "htrvt_conv_wgrad_acc": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "htrvt_conv_wgrad_acc_t": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "htrvt_conv_wgrad_acc_w": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "htrvt_unpack_conv_grads": (_I, [_I, _P, _P, _P, _P, _P, _P]),
    "htrvt_sample_ln_fwd": (_I, [_P, _P, _I, _P, _P, _I, _I, _F, _P]),
    "htrvt_sample_ln_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "htrvt_row_ln_fwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _F, _P]),
    "htrvt_gelu_fwd": (_I, [_P, _P, _L, _P]),
    "htrvt_row_ln_bwd_ctas": (_I, [_I]),
    "htrvt_row_ln_bwd": (_I, [_P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _P]),
    "htrvt_tokens_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "htrvt_tokens_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "htrvt_gelu_bwd": (_I, [_P, _P, _P, _L, _P]),
    "htrvt_mul_bf16": (_I, [_P, _P, _P, _L, _P]),
    "htrvt_colsum_rows": (_I, [_I]),
    "htrvt_colsum_bf16": (_I, [_P, _L, _I, _I, _P, _I, _P, _P]),
    "htrvt_cast_bf16": (_I, [_P, _P, _L, _P]),
    "htrvt_cast_colsum_bf16": (_I, [_P, _P, _P, _I, _I, _P]),
    "htrvt_dropout_bf16": (_I, [_P, _L, _L, _F, ctypes.c_ulonglong, ctypes.c_uint, _P, _P]),
    "htrvt_pack_weights": (_I, [_I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "htrvt_pack_conv_weight": (_I, [_P, _P, _I, _I, _I, _P]),
    "htrvt_conv1_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "htrvt_bn_finalize": (_I, [_P, _I, ctypes.c_double, _P, _P, _P, _P, _P, _F, _F, _I, _P, _P, _P, _P, _I, _P]),
    "htrvt_bn_act_fwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _P]),
    "htrvt_pool_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "htrvt_pool_bwd": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "htrvt_bn_bwd_ctas": (_I, [_L]),
    "htrvt_conv_dgrad_bn": (_I, [_P, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P]),
    "htrvt_bn_bwd_apply": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P, _I, _P]),
    "htrvt_bn_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P, _P, _I, _P]),
    "htrvt_conv1_wgrad_ctas": (_I, []),
    "htrvt_conv1_wgrad": (_I, [_P, _P, _P, _I, _P, _I, _I, _I, _I, _P]),
    "htrvt_stem_head_moment_ctas": (_I, []),
    "htrvt_stem_head_bwd_ctas": (_I, []),
    "htrvt_stem_head_moments": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "htrvt_stem_head_set_mode": (_I, [_I]),
    "htrvt_stem_head_fwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "htrvt_stem_head_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "htrvt_mt_sqnorm": (_I, [_I, _P, _P, _P, _I, _P, _P]),
    "htrvt_mt_sam_first": (_I, [_I, _P, _P, _P, _P, _P, _F, _I, _P]),
    "htrvt_mt_adamw": (_I, [_I, _P, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _I, _P]),
    "htrvt_mt_ema": (_I, [_I, _P, _P, _P, _F, _P]),
    "htrvt_attention_fwd": (_I, [_P, _I, _I, _I, _I, _F, _P, _P, _P]),
    "htrvt_attention2_fwd": (_I, [_P, _I, _I, _I, _I, _F, _P, _I, _I, _I, _F, ctypes.c_ulonglong, _P, _P, _P]),
    "htrvt_attention2_bwd_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "htrvt_attention2_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _F, _P, _I, _I, _I, _F, ctypes.c_ulonglong, _P, _P, _P,
                                  _Z, _P]),
    "htrvt_attention_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _F, _P, _P]),
    # fp32-parity mode (csrc/exact.cu)
    "htrvt_split3": (_I, [_P, _P, _L, _P]),
    "htrvt_bn_act_f32": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _P]),
    "htrvt_maxpool_f32": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "htrvt_tokens_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "htrvt_row_ln_f32": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _F, _P]),
    "htrvt_gelu_split": (_I, [_P, _P, _L, _P]),
    "htrvt_attention_f32": (_I, [_P, _I, _I, _I, _I, _F, _P, _P]),
    "htrvt_attention2_f32": (_I, [_P, _I, _I, _I, _I, _F, _P, _I, _I, _I, _P, _P]),
}


def _declare(l: ctypes.CDLL) -> None:
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(l, name)          # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
