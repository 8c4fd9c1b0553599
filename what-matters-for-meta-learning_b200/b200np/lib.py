"""ctypes binding of libb200np.so -- the C ABI declared in include/b200np.h.

This is exactly the stub a maintainer of the reference would add to call the B200 path
(INTEGRATION.md).  There is no fallback: if the library is missing the import raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200NP_LIB") or os.path.join(os.path.dirname(_HERE), "csrc", "libb200np.so")

PREC_FP32_SIMT, PREC_TF32X3, PREC_TF32 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2

_p, _i, _ll, _f, _sz = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_size_t


class GemmDesc(C.Structure):
    """struct b200np_gemm_desc (include/b200np.h)."""
    _fields_ = [("A", _p * 8), ("B", _p * 8), ("C", _p * 8), ("bias", _p * 8), ("groups", _i),
                ("M", _i), ("N", _i), ("K", _i), ("a_rs", _ll), ("a_cs", _ll), ("b_rs", _ll),
                ("b_cs", _ll), ("ldc", _ll), ("alpha", _f), ("beta", _f), ("act", _i),
                ("row_scale", _p), ("addend", _p), ("ld_add", _ll), ("precision", _i),
                ("workspace", _p), ("workspace_bytes", _sz), ("sum_groups", _i),
                ("conv_operand", _i), ("conv_H", _i), ("conv_W", _i), ("conv_C", _i)]


# name: (restype, [argtypes])  -- one entry per symbol in include/b200np.h
SIGNATURES = {
    "b200np_strerror": (C.c_char_p, [_i]),
    "b200np_version": (_i, []),
    "b200np_device_ok": (_i, []),
    "b200np_launch_count": (_ll, []),
    "b200np_conv_small_fwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "b200np_conv_small_wgrad_workspace": (_sz, [_i] * 9),
    "b200np_conv_small_wgrad": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "b200np_packed_weight_floats": (_sz, [_i, _i, _i]),
    "b200np_pack_conv_weight": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "b200np_conv_fwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "b200np_conv_dgrad": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _i, _i, _i, _p]),
    "b200np_conv_wgrad_workspace": (_sz, [_i] * 7),
    "b200np_conv_wgrad": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _i, _i, _p, _sz, _p]),
    "b200np_adaptive_maxpool2x2_flatten_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_adaptive_maxpool2x2_flatten_bwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_nhwc_to_nchw_flat": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "b200np_nchw_flat_to_nhwc": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_maxpool2x2_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_maxpool2x2_bwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_gather_images_u8": (_i, [_p, _p, _p, _ll, _i, _i, _i, _p]),
    "b200np_multi_copy": (_i, [_p, _p, _p, _i, _p, _p]),
    "b200np_multi_accumulate": (_i, [_p, _p, _p, _i, _p, _p]),
    "b200np_gemm_workspace": (_sz, [C.POINTER(GemmDesc)]),
    "b200np_gemm": (_i, [C.POINTER(GemmDesc), _p]),
    "b200np_act_bwd": (_i, [_p, _p, _p, _ll, _i, _p]),
    "b200np_colsum_workspace": (_sz, [_ll, _i]),
    "b200np_colsum": (_i, [_p, _p, _ll, _i, _ll, _p, _sz, _p]),
    "b200np_fill": (_i, [_p, _ll, _f, _p]),
    "b200np_axpy": (_i, [_p, _p, _ll, _f, _p]),
    "b200np_repeat_rows": (_i, [_p, _p, _ll, _i, _i, _p]),
    "b200np_repeat_rows_bwd": (_i, [_p, _p, _ll, _i, _i, _p]),
    "b200np_scale_by_device_scalar": (_i, [_p, _p, _p, _ll, _p]),
    "b200np_ctx_aggregate_fwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_ctx_aggregate_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_baco_fwd": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "b200np_baco_bwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "b200np_favor_rowstats": (_i, [_p, _p, _p, _p, _p, _ll, _i, _i, _ll, _p]),
    "b200np_reduce": (_i, [_p, _ll, _p, _i, _p]),
    "b200np_favor_attn_fwd": (_i, [_p] * 11 + [_i] * 6 + [_ll, _p]),
    "b200np_favor_attn_bwd": (_i, [_p] * 18 + [_i] * 6 + [_ll, _p]),
    "b200np_favor_key_fixup": (_i, [_p, _p, _p, _p, _p, _ll, _i, _ll, _p]),
    "b200np_loss_fwd_bwd": (_i, [_p, _p, _p, _p, _ll, _i, _i, _i, _p]),
    "b200np_adam_step": (_i, [_p, _p, _p, _p, _ll, _f, _f, _f, _f, _f, _i, _f, _p]),
    "b200np_adam_step_dev": (_i, [_p, _p, _p, _p, _ll, _f, _f, _f, _f, _f, _p, _f, _p]),
    "b200np_grad_norm_workspace": (_sz, [_ll]),
    "b200np_grad_norm": (_i, [_p, _ll, _f, _p, _p, _sz, _p]),
    "b200np_adam_step_ctrl": (_i, [_p, _p, _p, _p, _ll, _p, _f, _f, _f, _f, _p, _f, _p, _p, _p, _p]),
    "b200np_adam_step_groups": (_i, [_p, _p, _p, _p, _ll, _p, _i, _p, _p, _i, _p, _f, _p, _p, _p, _p]),
    "b200np_im2col3x3s2": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "b200np_col2im3x3s2": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_im2col_small": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p]),
    "b200np_conv_weight_tapmajor": (_i, [_p, _p, _i, _i, _i, _p]),
    "b200np_col2im3x3s2_tapmajor": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "b200np_bn_workspace": (_sz, [_ll, _i]),
    "b200np_bn_act_fwd": (_i, [_p, _p, _p, _f, _f, _p, _p, _p, _p, _p, _f, _ll, _i, _i, _p, _sz, _p]),
    "b200np_bn_act_bwd": (_i, [_p, _p, _p, _p, _p, _p, _f, _p, _p, _p, _ll, _i, _i, _p, _sz, _p]),
    "b200np_bn_workspace2": (_sz, [_ll, _i]),
    "b200np_bn_act_bwd2": (_i, [_p, _p, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p, _ll, _i, _i, _p, _sz, _p]),
    "b200np_mul3": (_i, [_p, _p, _p, _f, _p, _ll, _p]),
    "b200np_bbb_kl_blocks": (_i, [_ll]),
    "b200np_bbb_sample_kl_fwd": (_i, [_p, _p, _p, _f, _f, _p, _p, _p, _ll, _p]),
    "b200np_bbb_sample_kl_bwd": (_i, [_p, _p, _p, _p, _p, _p, _f, _f, _p, _p, _ll, _p]),
    "b200np_debug_set_wgrad_waves": (None, [_i]),
}


class B200NPError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing -- build it with `make -C {os.path.dirname(LIB_PATH)}` or "
            "`python -c 'import __graft_entry__ as g; g.build()'`.  There is no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


LIB = _load()


def check(rc, what):
    if rc != 0:
        raise B200NPError(f"{what}: {LIB.b200np_strerror(rc).decode()} (code {rc})")
