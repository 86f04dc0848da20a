"""ctypes binding of libvlbert_b200.so (the C ABI in include/vlbert_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a RuntimeError
is raised (the reference's native op raises RuntimeError through AT_ASSERTM / THCudaCheck,
common/lib/roi_pooling/cuda/ROIAlign_cuda.cu:262-264,297).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvlbert_b200.so")

_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_float = ctypes.c_float
c_int64 = ctypes.c_int64
c_uint32 = ctypes.c_uint32


def _declare(lib):
    lib.vlb_abi_version.restype = c_int
    lib.vlb_abi_version.argtypes = []
    lib.vlb_last_error_string.restype = ctypes.c_char_p
    lib.vlb_last_error_string.argtypes = []
    lib.vlb_launch_count.restype = c_int64
    lib.vlb_launch_count.argtypes = []
    lib.vlb_gemm_bf16.restype = c_int
    lib.vlb_gemm_bf16.argtypes = [c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int,
                                  c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                  c_void_p, c_int, c_float, c_int, c_int, c_void_p]
    lib.vlb_debug_gemm_desc.restype = None
    lib.vlb_debug_gemm_desc.argtypes = [c_uint32, c_uint32, c_uint32]
    lib.vlb_debug_gemm_trace.restype = None
    lib.vlb_debug_gemm_trace.argtypes = [c_void_p]

    P, I, F, L = c_void_p, c_int, c_float, c_int64

    def decl(name, args, res=c_int):
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args

    decl("vlb_gemm_grouped_tn", [P, P, I, I, I, I, P])
    decl("vlb_set_sm_limit", [I], None)
    decl("vlb_streamk_compiled", [])
    decl("vlb_profile_enable", [I], None)
    decl("vlb_profile_collect", [P, P, P])
    decl("vlb_mhsa_forward", [P, P, P, P, I, I, I, I, P])
    decl("vlb_mhsa_backward", [P, P, P, P, P, P, P, I, I, I, I, P])
    decl("vlb_layernorm_forward", [P, I, P, P, P, P, P, P, I, I, F, P])
    decl("vlb_layernorm_backward", [P, P, P, I, P, P, P, P, P, I, P, P, P, I, I, P])
    decl("vlb_colsum_bf16", [P, I, P, I, I, P])
    decl("vlb_cast_f32_to_bf16", [P, P, L, P])
    decl("vlb_cast_bf16_to_f32", [P, P, L, P])
    decl("vlb_multi_cast", [P, I, I, P])
    decl("vlb_pack_index", [P, P, P, I, I, I, I, I, P, P, P, P, P, P, P, P, P])
    decl("vlb_pack_forward", [P, P, P, P, P, P, P, P, P, P, P, P, I, I, P, I, I, I, I, I, I, I, P, P])
    decl("vlb_pack_backward", [P, P, P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, P])
    decl("vlb_gather_rows", [P, I, I, P, P, I, I, I, I, P])
    decl("vlb_scatter_rows_add", [P, I, I, P, P, I, I, I, P])
    decl("vlb_roi_align_forward", [P, P, P, I, I, I, I, I, I, F, I, P])
    decl("vlb_roi_align_backward", [P, P, P, I, I, I, I, I, I, I, F, I, P])
    decl("vlb_region_operand", [P, I, P, P, I, P, P, P, P, I, I, I, P])
    decl("vlb_im2col_nhwc", [P, P] + [I] * 12 + [P])
    decl("vlb_col2im_nhwc", [P, P, P] + [I] * 12 + [P])
    decl("vlb_conv_gemm", [P, I, P, I, P, I, I, I, P, P, P, I, P])
    decl("vlb_dropout_mask", [P, L, ctypes.c_float, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, P])
    decl("vlb_dropout", [P, P, L, I, ctypes.c_float, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, P])
    decl("vlb_grad_sqnorm", [P, I, P, P])
    decl("vlb_adamw_step", [P, P, I, ctypes.c_double, ctypes.c_double, ctypes.c_double, P, ctypes.c_float, P])
    decl("vlb_conv_fprop", [P, P, P, I, P, I, P, P, P, I, P])
    decl("vlb_conv_wgrad", [P, P, P, I, P, I, I, P])
    decl("vlb_relu_bn_backward", [P, P, P, P, P, P, L, I, P])
    decl("vlb_maxpool3x3s2_nhwc", [P, P, I, I, I, I, P])
    decl("vlb_avgpool_forward", [P, P, I, I, I, P])
    decl("vlb_avgpool_backward", [P, P, I, I, I, P])
    decl("vlb_nchw_f32_to_nhwc_bf16", [P, P, I, I, I, I, P])
    decl("vlb_nhwc_bf16_to_nchw_f32", [P, P, I, I, I, I, P])
    decl("vlb_roi_align_nhwc_forward", [P, P, P, I, I, I, I, I, I, F, I, P])
    decl("vlb_roi_align_nhwc_backward", [P, P, P, I, I, I, I, I, I, I, F, I, P])
    decl("vlb_bert_layer_forward", [P, P, P, P, P, I, I, I, I, I, F, P, P])
    decl("vlb_bert_layer_backward_workspace", [I, I, I], L)
    decl("vlb_bert_layer_backward", [P, P, P, P, P, P, P, P, P, P, L, I, I, I, I, I, P, P])
    decl("vlb_label_compact", [P, I, L, P, P, I, P, P])
    decl("vlb_mlm_ce_forward", [P, I, I, P, P, I, P, P, P, P])
    decl("vlb_mlm_ce_backward", [P, I, I, P, P, I, P, P, P])
    decl("vlb_soft_target_rows", [P, I, I, I, P, P])
    decl("vlb_soft_ce_forward", [P, I, I, P, I, P, P, P, I, P, P, P, P])
    decl("vlb_soft_ce_backward", [P, I, I, P, I, P, P, I, P, P, P])
    decl("vlb_layer_dropout_bits", [P, I, I, I, I, P, P])
    decl("vlb_gemm_bias_residual_f32", [I, I, I, P, I, P, I, P, I, P, P, P, I, P])
    decl("vlb_dropout_bits_words", [L, I], L)
    decl("vlb_dropout_bits", [P, L, I, P, P])
    # dropout-aware forms (ABI version 2): trailing VlbDropout* before the stream
    decl("vlb_gemm_bf16_dropout", [c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p,
                                   c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_float, c_int, c_int, P, P])
    decl("vlb_mhsa_forward_dropout", [P, P, P, P, I, I, I, I, P, P])
    decl("vlb_mhsa_backward_dropout", [P, P, P, P, P, P, P, I, I, I, I, P, P, P])
    decl("vlb_layernorm_forward_dropout", [P, I, P, P, P, P, P, P, I, I, F, P, P])
    decl("vlb_layernorm_backward_dropout", [P, P, P, I, P, P, P, P, P, I, P, P, P, I, I, P, P, P, P])
    decl("vlb_region_operand_dropout", [P, I, P, P, I, P, P, P, P, I, I, I, P, P])
    decl("vlb_dropout_mask_2d", [P, L, I, ctypes.c_float, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, P])
    decl("vlb_dropout_2d", [P, I, P, I, L, I, I, I, I, P, P])


class LayerWeights(ctypes.Structure):
    """VlbLayerWeights (include/vlbert_b200.h)"""
    _fields_ = [(n, c_void_p) for n in ("w_qkv", "b_qkv", "w_o", "b_o", "ln1_g", "ln1_b", "w_1", "b_1", "w_2", "b_2",
                                        "ln2_g", "ln2_b")]


class LayerActs(ctypes.Structure):
    """VlbLayerActs"""
    _fields_ = [(n, c_void_p) for n in ("qkv", "ctx", "lse", "a", "ln1_mean", "ln1_rstd", "h", "z", "u", "y0", "ln2_mean",
                                        "ln2_rstd", "y", "y_f32", "keep_attn", "keep_self_out", "keep_out")]


class LayerGrads(ctypes.Structure):
    """VlbLayerGrads"""
    _fields_ = [(n, c_void_p) for n in ("dw_qkv", "db_qkv", "dw_o", "db_o", "dln1_g", "dln1_b", "dw_1", "db_1", "dw_2",
                                        "db_2", "dln2_g", "dln2_b")]


class Dropout(ctypes.Structure):
    """VlbDropout"""
    _fields_ = [("p", c_float), ("site", c_uint32), ("rng", c_void_p), ("keep_bits", c_void_p)]


class Residual(ctypes.Structure):
    """VlbResidual"""
    _fields_ = [(n, c_void_p) for n in ("x_f32", "mean", "rstd", "gamma", "beta")]


class LayerDropout(ctypes.Structure):
    """VlbLayerDropout"""
    _fields_ = [("p_attn", c_float), ("p_hidden", c_float), ("site_attn", c_uint32), ("site_self_out", c_uint32),
                ("site_out", c_uint32), ("rng", c_void_p), ("keep_bits_ready", c_int)]


class GroupedProblem(ctypes.Structure):
    """VlbGroupedProblem"""
    _fields_ = [("M", c_int), ("N", c_int), ("A", c_void_p), ("lda", c_int), ("B", c_void_p), ("ldb", c_int),
                ("out", c_void_p), ("ldo", c_int)]


class ConvGeom(ctypes.Structure):
    """VlbConvGeom"""
    _fields_ = [(n, ctypes.c_int) for n in ("N", "H", "W", "C", "Ho", "Wo", "kh", "kw", "stride", "pad", "dil")]


class AdamWTensor(ctypes.Structure):
    """VlbAdamWTensor"""
    _fields_ = [("param", c_void_p), ("grad", c_void_p), ("exp_avg", c_void_p), ("exp_avg_sq", c_void_p), ("n", c_int64)]


class CastDesc(ctypes.Structure):
    """VlbCastDesc"""
    _fields_ = [("src", c_void_p), ("dst", c_void_p), ("n", c_int64), ("dst_is_bf16", c_int64)]


def lib():
    """Load (once) and return the ctypes handle; raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "vlbert_b200: %s not found -- run `python vl-bert_b200/build.py` (there is no CPU "
                "fallback)" % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        _declare(handle)
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().vlb_last_error_string().decode("utf-8", "replace")
        raise RuntimeError("vlbert_b200 error %d: %s" % (rc, msg))


def last_error():
    return lib().vlb_last_error_string().decode("utf-8", "replace")


def launch_count():
    return int(lib().vlb_launch_count())
