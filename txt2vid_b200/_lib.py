"""ctypes binding of libt2v_b200.so (the C ABI declared in include/t2v.h).

There is no CPU fallback: importing this module without the built library, or calling a kernel
without a CUDA device, raises.  Build with `python -c "import __graft_entry__ as g; g.build()"`
(or `make -C txt2vid_b200/csrc`).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libt2v_b200.so")

T2V_OK = 0
ALGO_AUTO, ALGO_TC, ALGO_SIMT, ALGO_TC_GENERIC, ALGO_SIMT_F32 = 0, 1, 2, 3, 4
EPI_RELU, EPI_OUT_F32, EPI_RELU_MASK, EPI_IN_F32 = 1, 2, 4, 16


class ConvGeom(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("N", "D", "H", "W", "Cin", "Cout", "kd", "kh", "kw")]


class GconvGeom(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("N", "Di", "Hi", "Wi", "Do", "Ho", "Wo", "Cin", "Cout", "kd", "kh", "kw",
                                              "sd", "sh", "sw", "pd", "ph", "pw")]


class T2VError(RuntimeError):
    pass


_lib = None


def lib():
    """Load the shared library once; fail loudly when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise T2VError(
                "libt2v_b200.so is not built (%s). Run __graft_entry__.build(); there is no fallback path."
                % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


c_void_p, c_int, c_i64, c_u32, c_float = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint32,
                                          ctypes.c_float)
_P = c_void_p
c_i32 = ctypes.c_int32
_I32P = ctypes.POINTER(ctypes.c_int32)
_PP = ctypes.POINTER(ctypes.c_void_p)

# name -> argtypes (restype is int unless listed in _RESTYPES); kept in one table so the CPU test
# can check that every symbol of include/t2v.h is exported.
SIGNATURES = {
    "t2v_version": [],
    "t2v_launch_count": [],
    "t2v_profile_enable": [c_int],
    "t2v_profile_read": [ctypes.POINTER(ctypes.c_double)],
    "t2v_profile_read4": [ctypes.POINTER(ctypes.c_double)],
    "t2v_profile_read6": [ctypes.POINTER(ctypes.c_double)],
    "t2v_profile_next_scale": [ctypes.c_double],
    "t2v_conv_fprop": [ctypes.POINTER(ConvGeom), _P, _P, _P, _P, _P, c_u32, c_int, _P],
    "t2v_conv_lstm_step": [ctypes.POINTER(ConvGeom), _P, _P, _P, _P, _P, _P, _P, _P, c_i32, c_i32, _P],
    "t2v_conv_fprop_skip": [ctypes.POINTER(ConvGeom), _P, _P, _P, _P, _P, c_i32, _P, c_u32, _P],
    "t2v_conv_dgrad": [ctypes.POINTER(ConvGeom), _P, _P, _P, _P, c_u32, c_int, _P],
    "t2v_conv_wgrad": [ctypes.POINTER(ConvGeom), _P, _P, _P, c_int, c_int, _P],
    "t2v_conv_sd2_supported": [ctypes.POINTER(ConvGeom)],
    "t2v_conv_fprop_sd2": [ctypes.POINTER(ConvGeom), _P, _P, _P, _P, c_u32, _P],
    "t2v_conv_dgrad_sd2": [ctypes.POINTER(ConvGeom), _P, _P, _P, _P, c_u32, _P],
    "t2v_conv_wgrad_sd2": [ctypes.POINTER(ConvGeom), _P, _P, _P, c_int, _P],
    "t2v_stem_fprop": [_P, c_i32, _P, _P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_stem_wgrad": [_P, _P, c_i32, _P, c_i64, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_rgb_to_cl": [_P, _P, _P, c_i64, c_i64, _P],
    "t2v_wgrad_fold_pairs": [_P, _P, c_i32, c_i32, c_i32, _P],
    "t2v_gconv_fprop": [ctypes.POINTER(GconvGeom), _P, _P, _P, _P, c_i32, _P],
    "t2v_gconv_dgrad": [ctypes.POINTER(GconvGeom), _P, _P, _P, _P, c_i32, _P],
    "t2v_gconv_wgrad": [ctypes.POINTER(GconvGeom), _P, _P, _P, c_i32, _P],
    "t2v_moving_digits": [_P, _P, _P, _P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_grammar_tokens": [_P, _P, _P, _P, c_i32, _P],
    "t2v_u8_normalize": [_P, _P, c_i64, _P],
    "t2v_s2d_shift": [_P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_d2s_shift": [_P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_s2d_embed_weight": [_P, _P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_s2d_extract_wgrad": [_P, _P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_transpose_flip_bf16": [_P, _P, c_i32, c_i32, c_i32, _P],
    "t2v_window_rows": [_P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_s2d_tile_bias": [_P, _P, c_i32, c_i32, c_i32, _P],
    "t2v_conv_fprop_win": [ctypes.POINTER(ConvGeom), _I32P, _P, _P, _P, _P, c_u32, _P],
    "t2v_conv_wgrad_win": [ctypes.POINTER(ConvGeom), _I32P, _P, _P, _P, c_int, _P],
    "t2v_cast_f32_to_bf16": [_P, _P, c_i64, _P],
    "t2v_cast_bf16_to_f32": [_P, _P, c_i64, _P],
    "t2v_pack_dgrad_weight": [_P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P],
    "t2v_pack_weight_padded": [_P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P],
    "t2v_unpack_wgrad_padded": [_P, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _P],
    "t2v_relu_fwd": [_P, _P, c_i64, _P],
    "t2v_relu_bwd": [_P, _P, _P, c_i64, _P],
    "t2v_leaky_relu_fwd": [_P, _P, c_i64, c_float, _P],
    "t2v_leaky_relu_bwd": [_P, _P, _P, c_i64, c_float, _P],
    "t2v_tanh_fwd": [_P, _P, c_i64, _P],
    "t2v_tanh_bwd": [_P, _P, _P, c_i64, _P],
    "t2v_avgpool_fwd": [_P, _P, _P, _I32P, _I32P, _I32P, _I32P, _P],
    "t2v_avgpool_bwd": [_P, _P, _I32P, _I32P, _I32P, _I32P, _P],
    "t2v_upsample2x_fwd": [_P, _P, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_upsample2x_bwd": [_P, _P, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_nchw_to_cl": [_P, _P, c_i64, c_i32, c_i64, c_i32, _P],
    "t2v_cl_to_nchw": [_P, _P, c_i64, c_i32, c_i64, c_i32, _P],
    "t2v_im2col3": [_P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_col2im3": [_P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_sum_rows": [_P, _P, c_i64, c_i32, _P],
    "t2v_sum_rows_acc": [_P, _P, c_i64, c_i32, _P],
    "t2v_sum_spatial": [_P, _P, c_i64, c_i64, c_i32, _P],
    "t2v_broadcast_spatial": [_P, _P, c_i64, c_i64, c_i32, _P],
    "t2v_bn_stats": [_P, _P, c_i64, c_i32, _P],
    "t2v_bn_finalize": [_P, _P, _P, _P, _P, _P, _P, c_i32, c_i64, c_float, c_float, _P],
    "t2v_bn_apply": [_P, _P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_bn_bwd": [_P, _P, _P, _P, _P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_bn_bwd_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_i64, c_i32, c_i32, c_i32, _P],
    "t2v_attention_fwd": [_P, _P, _P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_attention_bwd": [_P, _P, _P, _P, _P, _P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_attention_bwd_large": [_P, _P, _P, _P, _P, _P, _P, _P, c_i64, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32,
                                _P],
    "t2v_render_fwd": [_P, _P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_render_bwd": [_P, _P, _P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_gather_frames": [_P, _P, c_i32, c_i32, c_i64, c_i32, c_i32, c_i32, _P, c_i32, _P],
    "t2v_pyramid_level": [_P, _P, _I32P, c_i32, c_i32, c_i32, c_i32, c_i32, _P, _P],
    "t2v_lstm_cell_fwd": [_P, _P, _P, _P, _P, c_i64, c_i32, _P],
    "t2v_lstm_cell_bwd": [_P, _P, _P, _P, _P, _P, _P, c_i64, c_i32, _P],
    "t2v_multi_copy": [c_i32, _PP, _PP, ctypes.POINTER(c_i64), _P],
    "t2v_adam_step": [c_i32, _PP, _PP, _PP, _PP, ctypes.POINTER(c_i64), c_float, c_float, c_float, c_float, c_i32,
                      c_float, _P, _P],
}

# fp32 activation storage: every storage-typed entry point has an _f32 twin with the same signature
_TYPED = ["t2v_relu_fwd", "t2v_relu_bwd", "t2v_leaky_relu_fwd", "t2v_leaky_relu_bwd", "t2v_tanh_fwd", "t2v_tanh_bwd",
          "t2v_avgpool_fwd", "t2v_avgpool_bwd", "t2v_upsample2x_fwd", "t2v_upsample2x_bwd", "t2v_nchw_to_cl",
          "t2v_cl_to_nchw", "t2v_im2col3", "t2v_col2im3", "t2v_sum_rows", "t2v_sum_rows_acc", "t2v_sum_spatial",
          "t2v_broadcast_spatial", "t2v_bn_stats", "t2v_bn_apply", "t2v_bn_bwd", "t2v_bn_bwd_bwd", "t2v_render_fwd",
          "t2v_render_bwd",
          "t2v_lstm_cell_fwd", "t2v_lstm_cell_bwd", "t2v_gconv_fprop", "t2v_gconv_dgrad", "t2v_gconv_wgrad",
          "t2v_scale", "t2v_scale_add", "t2v_dot", "t2v_cl_slice_f32", "t2v_f32_pad_cl", "t2v_lstm_seq_fwd",
          "t2v_lstm_seq_bwd", "t2v_embedding_fwd", "t2v_embedding_bwd"]
_F32P = ctypes.POINTER(ctypes.c_float)
SIGNATURES.update({
    "t2v_scale": [_P, _P, _P, c_i64, _P],
    "t2v_scale_add": [_P, _P, _P, _P, c_i64, _P],
    "t2v_dot": [_P, _P, _P, c_i64, _P],
    "t2v_cl_slice_f32": [_P, _P, c_i64, c_i32, c_i32, _P],
    "t2v_f32_pad_cl": [_P, _P, c_i64, c_i32, c_i32, _P],
    "t2v_maxpool122_fwd": [_P, _P, _P, c_i64, c_i32, c_i32, c_i32, _P],
    "t2v_pool122_gather": [_P, _P, _P, c_i64, c_i32, c_i32, c_i32, _P],
    "t2v_pool122_scatter": [_P, _P, _P, c_i64, c_i32, c_i32, c_i32, _P],
    "t2v_bmm_f32": [_P, _P, _P, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_softmax_fwd": [_P, _P, c_i64, c_i32, _P],
    "t2v_softmax_bwd": [_P, _P, _P, c_i64, c_i32, _P],
    "t2v_softmax_bwd_bwd": [_P, _P, _P, _P, _P, c_i64, c_i32, _P],
    "t2v_head_fwd": [_P, _P, _P, _P, _P, c_i32, c_i32, c_i32, _P],
    "t2v_head_bwd_data": [_P, _P, _P, _P, c_i32, c_i32, c_i32, _P],
    "t2v_head_bwd_weight": [_P, _P, _P, _P, _P, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_rel_loss_fwd": [c_i32, _PP, _PP, _I32P, _F32P, c_i32, _P, _P],
    "t2v_rel_loss_bwd": [c_i32, _PP, _PP, _PP, _PP, _I32P, _F32P, c_i32, _P, _P],
    "t2v_lerp_rows": [_P, _P, _P, _P, c_i64, c_i64, _P],
    "t2v_gp_norm_fwd": [_P, _P, _P, _P, c_i64, c_i64, c_i32, _P],
    "t2v_gp_norm_bwd": [_P, _P, _P, _P, c_i64, c_i64, _P],
    "t2v_lstm_pack_whh": [_P, _P, c_i32, c_i32, _P],
    "t2v_lstm_seq_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_lstm_seq_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_i32, c_i32, c_i32, c_i32, _P],
    "t2v_embedding_fwd": [_P, _P, _P, c_i64, c_i32, _P],
    "t2v_embedding_bwd": [_P, _P, _P, c_i64, c_i32, c_i64, _P],
})
for _n in _TYPED:
    SIGNATURES[_n + "_f32"] = SIGNATURES[_n]
_RESTYPES = {"t2v_launch_count": ctypes.c_ulonglong}


def _declare(l):
    for name, argtypes in SIGNATURES.items():
        fn = getattr(l, name)
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, c_int)


def typed(name, t):
    """entry point for the storage type of tensor t: `name` (bf16) or its fp32 twin `name_f32`"""
    return getattr(lib(), name + "_f32" if t.dtype == torch.float32 else name)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def check(rc, what):
    if rc != T2V_OK:
        raise T2VError("%s failed with T2V error %d" % (what, rc))


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise T2VError("txt2vid_b200 kernels need CUDA tensors (got %s); there is no CPU path" % t.device)
