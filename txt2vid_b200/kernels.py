"""Raw kernel calls: torch tensors in, torch tensors out, one C-ABI call each.

Tensors here are in the kernels' native layouts ("CL" = contiguous (N, D, H, W, C) bf16; 2-D
feature maps use D = 1).  Everything above this file (ops.py autograd formulas, the module mirrors)
only talks to the GPU through these functions.  There is no CPU path: every function raises on
non-CUDA tensors (tests/cpu_kernels.py is a test-only stand-in used to check the autograd formulas).
"""
import ctypes

import torch

from . import _lib
from ._lib import ConvGeom, GconvGeom, check, lib, ptr, require_cuda, stream

BF16 = torch.bfloat16
F32 = torch.float32

# Activation storage type of the tensors the wrappers CREATE at fp32 boundaries (layout conversion, operand packs,
# broadcast / render / LSTM outputs).  bf16 is the product; fp32 is the parity mode of BASELINE's north_star (1e-3 on
# losses and gradients): same kernels instantiated for float storage, and the convolutions on exact fp32 FMAs on the
# CUDA cores (see conv_fprop).  Elementwise wrappers follow the dtype of their input.
STORE = BF16


def set_store_dtype(dt):
    global STORE
    assert dt in (BF16, F32)
    STORE = dt


PROFILING = [False]


def profile_enable(on):
    """per-launch CUDA-event timing of the conv engine (bench.py roofline pass)"""
    PROFILING[0] = bool(on)
    lib().t2v_profile_enable(1 if on else 0)


def prof_real_fraction(real, padded):
    """tell the profiler which fraction of the next conv launch's channel products is real (not zero padding)"""
    if PROFILING[0] and padded > 0 and real != padded:
        lib().t2v_profile_next_scale(float(real) / float(padded))


def _act(*ts):
    for t in ts:
        assert t is None or (t.dtype in (BF16, F32) and t.is_contiguous()), (None if t is None else (t.dtype, t.shape))


# fp32 storage mode, convolution engine: fp32 operands, exact fp32 FMAs on the CUDA cores (gconv.cu, selected by
# T2V_EPI_IN_F32 / T2V_ALGO_SIMT_F32): the reference's own numerics, ~1e-6 per layer -- what the 1e-3 bar on
# GRADIENTS needs on this network (a forward deviation of 5e-5 already moves the generator's gradients by 5e-3 through
# ReLU / BatchNorm, measured).  The tensor pipe on bf16 part splits of the fp32 operands does not reach it: its fp32
# accumulator truncates on every MMA (7e-6 relative at K = 1024, 3e-5 at K = 9216;
# profiles/r02_fp32_engine_accuracy.txt).


def _geom(N, D, H, W, Cin, Cout, k):
    kd, kh, kw = k
    return ConvGeom(N, D, H, W, Cin, Cout, kd, kh, kw)


def _i32(*vals):
    return (ctypes.c_int32 * len(vals))(*vals)


# ------------------------------------------------------------------------------------- conv engine
def conv_fprop(x, w, bias=None, residual=None, k=(3, 3, 3), relu=False, out_f32=False, algo=0):
    """x (N,D,H,W,Cin) bf16, w (Cout,taps,Cin) bf16 -> y (N,D,H,W,Cout) bf16|f32.
    fp32 storage: x, w (and residual) fp32 -> y fp32."""
    require_cuda(x, w, bias, residual)
    N, D, H, W, Cin = x.shape
    Cout = w.shape[0]
    f32 = x.dtype == F32                          # fp32 parity mode on exact fp32 FMAs
    if f32:
        out_f32, algo = True, _lib.ALGO_SIMT
    assert w.shape[1] == k[0] * k[1] * k[2] and w.shape[2] == Cin, (w.shape, k, Cin)
    assert x.is_contiguous() and w.is_contiguous() and w.dtype == x.dtype
    assert bias is None or (bias.dtype == F32 and bias.numel() == Cout)
    assert residual is None or (residual.dtype == (F32 if f32 else BF16) and residual.is_contiguous())
    y = torch.empty((N, D, H, W, Cout), device=x.device, dtype=F32 if out_f32 else BF16)
    g = _geom(N, D, H, W, Cin, Cout, k)
    flags = (_lib.EPI_RELU if relu else 0) | (_lib.EPI_OUT_F32 if out_f32 else 0) | (_lib.EPI_IN_F32 if f32 else 0)
    check(lib().t2v_conv_fprop(ctypes.byref(g), ptr(x), ptr(w), ptr(bias), ptr(residual), ptr(y), flags, algo,
                               stream()), "t2v_conv_fprop")
    return y


def lstm_gate_interleave(hidden, device):
    """row permutation of a [i|f|g|o]-stacked (4*hidden, ...) operand for t2v_conv_lstm_step: new row
    blk * 128 + gate * 32 + j  <-  old row gate * hidden + blk * 32 + j"""
    assert hidden % 32 == 0
    return torch.arange(4 * hidden, device=device).view(4, hidden // 32, 32).permute(1, 0, 2).reshape(-1)


def conv_lstm_step(x, w_il, bias_il, c_prev, k, merged, t, steps):
    """One ConvLSTM step with the cell update in the gate GEMM's epilogue (bf16 storage only).
    x (B,1,fh,fw,Cin) bf16; w_il (4H,taps,Cin) bf16 / bias_il (4H,) fp32 gate-interleaved (lstm_gate_interleave);
    c_prev fp32 (B,1,fh,fw,H) or None; merged (B*steps,1,fh,fw,H) bf16: h_t is also written into its (b, t) slot.
    -> (gates fp32 (B,1,fh,fw,4H) in [i|f|g|o] order, c fp32, h bf16)"""
    require_cuda(x, w_il, bias_il, c_prev, merged)
    N, D, H, W, Cin = x.shape
    C4 = w_il.shape[0]
    Hd = C4 // 4
    assert x.dtype == BF16 and w_il.dtype == BF16 and x.is_contiguous() and w_il.is_contiguous() and C4 % 128 == 0
    assert w_il.shape[1] == k[0] * k[1] * k[2] and w_il.shape[2] == Cin and bias_il.dtype == F32 and bias_il.numel() == C4
    assert merged.dtype == BF16 and merged.is_contiguous() and merged.numel() == N * steps * D * H * W * Hd
    assert c_prev is None or (c_prev.dtype == F32 and c_prev.is_contiguous() and c_prev.numel() == N * D * H * W * Hd)
    gates = torch.empty((N, D, H, W, C4), device=x.device, dtype=F32)
    c = torch.empty((N, D, H, W, Hd), device=x.device, dtype=F32)
    h = torch.empty((N, D, H, W, Hd), device=x.device, dtype=BF16)
    g = _geom(N, D, H, W, Cin, C4, k)
    check(lib().t2v_conv_lstm_step(ctypes.byref(g), ptr(x), ptr(w_il), ptr(bias_il), ptr(c_prev), ptr(gates), ptr(c),
                                   ptr(h), ptr(merged), t, steps, stream()), "t2v_conv_lstm_step")
    return gates, c, h


def conv_fprop_skip(x, w, bias, x2, w2, k=(3, 3, 3), relu=False):
    """y = conv(x, w) + conv1x1x1(x2, w2) + bias in one implicit GEMM (the 1x1x1 convolution is extra K).
    x (N,D,H,W,Cin), x2 (N,D,H,W,Cin2) bf16; w (Cout,taps,Cin), w2 (Cout,1,Cin2) bf16; Cin, Cin2 multiples of 64."""
    require_cuda(x, w, bias, x2, w2)
    N, D, H, W, Cin = x.shape
    Cout, Cin2 = w.shape[0], x2.shape[-1]
    assert w.shape[1] == k[0] * k[1] * k[2] and w.shape[2] == Cin and tuple(x2.shape[:4]) == (N, D, H, W)
    assert w2.shape[0] == Cout and w2.numel() == Cout * Cin2 and Cin % 64 == 0 and Cin2 % 64 == 0
    assert all(t.is_contiguous() and t.dtype == BF16 for t in (x, w, x2, w2))
    assert bias is None or (bias.dtype == F32 and bias.numel() == Cout)
    y = torch.empty((N, D, H, W, Cout), device=x.device, dtype=BF16)
    g = _geom(N, D, H, W, Cin, Cout, k)
    check(lib().t2v_conv_fprop_skip(ctypes.byref(g), ptr(x), ptr(w), ptr(bias), ptr(x2), ptr(w2), Cin2, ptr(y),
                                    _lib.EPI_RELU if relu else 0, stream()), "t2v_conv_fprop_skip")
    return y


def conv_dgrad(dy, wT, k=(3, 3, 3), residual=None, relu=False, out_f32=False, algo=0, relu_ref=None):
    """dy (N,D,H,W,Cout) bf16, wT (Cin,taps,Cout) bf16 (from pack_dgrad_weight) -> dx (N,D,H,W,Cin).
    relu_ref (dx-shaped): dx is zeroed where relu_ref <= 0 (the ReLU in front of the convolution, fused).
    fp32 storage: dy, wT fp32 -> dx fp32."""
    require_cuda(dy, wT, residual, relu_ref)
    f32 = dy.dtype == F32                         # fp32 parity mode on exact fp32 FMAs
    if relu_ref is not None:
        assert residual is None and relu_ref.is_contiguous() and relu_ref.dtype == dy.dtype
        assert tuple(relu_ref.shape) == tuple(dy.shape[:4]) + (wT.shape[0],)
        residual = relu_ref
    N, D, H, W, Cout = dy.shape
    Cin = wT.shape[0]
    if f32:
        out_f32, algo = True, _lib.ALGO_SIMT
    assert wT.shape[2] == Cout and dy.is_contiguous() and wT.is_contiguous() and wT.dtype == dy.dtype
    dx = torch.empty((N, D, H, W, Cin), device=dy.device, dtype=F32 if out_f32 else BF16)
    g = _geom(N, D, H, W, Cin, Cout, k)
    flags = (_lib.EPI_RELU if relu else 0) | (_lib.EPI_OUT_F32 if out_f32 else 0) | \
        (_lib.EPI_RELU_MASK if relu_ref is not None else 0) | (_lib.EPI_IN_F32 if f32 else 0)
    check(lib().t2v_conv_dgrad(ctypes.byref(g), ptr(dy), ptr(wT), ptr(residual), ptr(dx), flags, algo, stream()),
          "t2v_conv_dgrad")
    return dx


def conv_wgrad(dy, x, k=(3, 3, 3), out=None, accumulate=False, algo=0):
    """dw (Cout,taps,Cin) fp32 = sum_pos dy[pos,co] x[pos+tap,ci]."""
    require_cuda(dy, x)
    N, D, H, W, Cout = dy.shape
    Cin = x.shape[-1]
    if dy.dtype == F32:                           # fp32 parity mode on exact fp32 FMAs
        algo = _lib.ALGO_SIMT_F32
    if (algo == 0 and tuple(k) == (1, 3, 3) and D == 1 and Cin == 32 and Cout in (16, 32)
            and W % 2 == 0 and W >= 16 and H >= 4 and dy.is_contiguous() and x.is_contiguous()):
        # 32-channel rows are 64 bytes: TMA and the MMA tiles run half empty.  Pair adjacent w voxels (a free view):
        # 64-channel rows on the halo-resident kernel, then fold the pair products into the 3 real w taps.
        dw2 = conv_wgrad(dy.view(N, 1, H, W // 2, 2 * Cout), x.view(N, 1, H, W // 2, 2 * Cin), k)
        if out is None:
            out = torch.empty((Cout, 9, Cin), device=x.device, dtype=F32)
            accumulate = False
        check(lib().t2v_wgrad_fold_pairs(ptr(dw2), ptr(out), Cout, Cin, 1 if accumulate else 0, stream()),
              "t2v_wgrad_fold_pairs")
        return out
    assert x.shape[:4] == dy.shape[:4] and dy.is_contiguous() and x.is_contiguous()
    assert x.dtype == dy.dtype and dy.dtype in (BF16, F32)
    taps = k[0] * k[1] * k[2]
    if out is None:
        assert not accumulate
        out = torch.empty((Cout, taps, Cin), device=x.device, dtype=F32)
    g = _geom(N, D, H, W, Cin, Cout, k)
    check(lib().t2v_conv_wgrad(ctypes.byref(g), ptr(dy), ptr(x), ptr(out), 1 if accumulate else 0, algo, stream()),
          "t2v_conv_wgrad")
    return out


def conv_sd2_supported(shape, Cin, Cout, k=(3, 3, 3)):
    """Can the stride-(2,1,1) kernels take an input of CL shape (N, D, H, W, C)?  (no GPU work)"""
    N, D, H, W = [int(v) for v in shape[:4]]
    g = _geom(N, D, H, W, Cin, Cout, k)
    return bool(lib().t2v_conv_sd2_supported(ctypes.byref(g)))


def conv_fprop_sd2(x, w, bias=None, relu=False):
    """Conv3d(64 -> 64, 3, stride (2,1,1), padding 1): x (N,D,H,W,64) bf16 -> y (N,D/2,H,W,64) bf16
    (= the even output planes of the stride-1 convolution)."""
    require_cuda(x, w, bias)
    N, D, H, W, Cin = x.shape
    Cout = w.shape[0]
    assert w.shape[1] == 27 and w.shape[2] == Cin and x.is_contiguous() and w.is_contiguous()
    assert x.dtype == BF16 and w.dtype == BF16 and (bias is None or (bias.dtype == F32 and bias.numel() == Cout))
    y = torch.empty((N, D // 2, H, W, Cout), device=x.device, dtype=BF16)
    g = _geom(N, D, H, W, Cin, Cout, (3, 3, 3))
    check(lib().t2v_conv_fprop_sd2(ctypes.byref(g), ptr(x), ptr(w), ptr(bias), ptr(y),
                                   _lib.EPI_RELU if relu else 0, stream()), "t2v_conv_fprop_sd2")
    return y


def conv_dgrad_sd2(dy, wT, relu_ref=None):
    """dy (N,D/2,H,W,Cout) bf16, wT (Cin,27,Cout) flipped pack -> dx (N,D,H,W,Cin) bf16 (zeroed where the dx-shaped
    relu_ref <= 0, if given)."""
    require_cuda(dy, wT, relu_ref)
    assert relu_ref is None or (relu_ref.is_contiguous() and relu_ref.dtype == BF16)
    N, Dj, H, W, Cout = dy.shape
    Cin = wT.shape[0]
    assert wT.shape[2] == Cout and dy.is_contiguous() and wT.is_contiguous() and dy.dtype == BF16
    dx = torch.empty((N, 2 * Dj, H, W, Cin), device=dy.device, dtype=BF16)
    g = _geom(N, 2 * Dj, H, W, Cin, Cout, (3, 3, 3))
    assert relu_ref is None or tuple(relu_ref.shape) == tuple(dx.shape)
    check(lib().t2v_conv_dgrad_sd2(ctypes.byref(g), ptr(dy), ptr(wT), ptr(relu_ref), ptr(dx), 0, stream()),
          "t2v_conv_dgrad_sd2")
    return dx


def conv_wgrad_sd2(dy, x, out=None, accumulate=False):
    """dw (Cout,27,Cin) fp32 = sum over the even output planes of dy[pos,co] x[pos+tap,ci]."""
    require_cuda(dy, x)
    N, D, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    assert tuple(dy.shape[:4]) == (N, D // 2, H, W) and dy.is_contiguous() and x.is_contiguous()
    assert dy.dtype == BF16 and x.dtype == BF16
    if out is None:
        assert not accumulate
        out = torch.empty((Cout, 27, Cin), device=x.device, dtype=F32)
    g = _geom(N, D, H, W, Cin, Cout, (3, 3, 3))
    check(lib().t2v_conv_wgrad_sd2(ctypes.byref(g), ptr(dy), ptr(x), ptr(out), 1 if accumulate else 0, stream()),
          "t2v_conv_wgrad_sd2")
    return out


def stem_pack_weight(w3):
    """fp32 (64, 27, 3) -> bf16 (64, 128) operand of t2v_stem_fprop: k = tap * 4 + c, zero padded (once per weight
    version, ~16 KB: plain tensor ops)."""
    require_cuda(w3)
    wp = torch.zeros((64, 32, 4), device=w3.device, dtype=F32)
    wp[:, :27, :3] = w3
    return wp.reshape(64, 128).to(BF16).contiguous()


def stem_fprop(xc, wp, bias=None, relu=True):
    """RGB stem conv on the tensor cores: xc (N,D,H,W,16) bf16 (RGB in 0..2), wp (64,128) bf16 (k = tap*4 + c)
    -> y (N,D,H,W,64) bf16 = [relu](conv3d(x, w, padding 1) + bias)."""
    require_cuda(xc, wp, bias)
    N, D, H, W, C = xc.shape
    assert C in (4, 16) and xc.dtype == BF16 and xc.is_contiguous() and tuple(wp.shape) == (64, 128)
    assert wp.dtype == BF16 and wp.is_contiguous() and (bias is None or (bias.dtype == F32 and bias.numel() == 64))
    y = torch.empty((N, D, H, W, 64), device=xc.device, dtype=BF16)
    check(lib().t2v_stem_fprop(ptr(xc), C, ptr(wp), ptr(bias), ptr(y), N, D, H, W, 1 if relu else 0, stream()),
          "t2v_stem_fprop")
    return y


def stem_wgrad(dy, xc, out=None, accumulate=False):
    """dw (64,27,3) fp32 = sum_pos dy[pos,co] x[pos+tap,c] for the RGB stem conv."""
    require_cuda(dy, xc)
    N, D, H, W, C = xc.shape
    assert C in (4, 16) and tuple(dy.shape) == (N, D, H, W, 64) and dy.dtype == BF16 and xc.dtype == BF16
    assert dy.is_contiguous() and xc.is_contiguous()
    if out is None:
        assert not accumulate
        out = torch.empty((64, 27, 3), device=xc.device, dtype=F32)
    check(lib().t2v_stem_wgrad(ptr(dy), ptr(xc), C, ptr(out), N, D, H, W, 1 if accumulate else 0, stream()),
          "t2v_stem_wgrad")
    return out


def cast_bf16(src):
    require_cuda(src)
    assert src.dtype == F32 and src.is_contiguous()
    dst = torch.empty(src.shape, device=src.device, dtype=BF16)
    check(lib().t2v_cast_f32_to_bf16(ptr(src), ptr(dst), src.numel(), stream()), "t2v_cast_f32_to_bf16")
    return dst


def cast_f32(src):
    require_cuda(src)
    assert src.dtype == BF16 and src.is_contiguous()
    dst = torch.empty(src.shape, device=src.device, dtype=F32)
    check(lib().t2v_cast_bf16_to_f32(ptr(src), ptr(dst), src.numel(), stream()), "t2v_cast_bf16_to_f32")
    return dst


def _pack_weight_bf16(w, CoutP, CinP):
    Cout, taps, Cin = w.shape
    if CoutP == Cout and CinP == Cin:
        return cast_bf16(w)
    dst = torch.zeros((CoutP, taps, CinP), device=w.device, dtype=BF16)
    check(lib().t2v_pack_weight_padded(ptr(w), ptr(dst), Cout, taps, Cin, CinP, stream()), "t2v_pack_weight_padded")
    return dst


def _pack_dgrad_bf16(w, CoutP, CinP):
    Cout, taps, Cin = w.shape
    alloc = torch.empty if (CoutP == Cout and CinP == Cin) else torch.zeros
    wT = alloc((CinP, taps, CoutP), device=w.device, dtype=BF16)
    check(lib().t2v_pack_dgrad_weight(ptr(w), ptr(wT), Cout, taps, Cin, CoutP, stream()), "t2v_pack_dgrad_weight")
    return wT


def pack_weight(w, CoutP=None, CinP=None):
    """w (Cout,taps,Cin) fp32 -> bf16 (CoutP,taps,CinP), zero padded (plain cast when unpadded).
    fp32 storage mode: fp32 (CoutP,taps,CinP)."""
    require_cuda(w)
    assert w.dtype == F32 and w.is_contiguous() and w.dim() == 3
    Cout, taps, Cin = w.shape
    CoutP, CinP = CoutP or Cout, CinP or Cin
    if STORE == F32:
        if (CoutP, CinP) == (Cout, Cin):
            return w.clone()
        wp = torch.zeros((CoutP, taps, CinP), device=w.device, dtype=F32)
        wp[:Cout, :, :Cin] = w
        return wp
    return _pack_weight_bf16(w, CoutP, CinP)


def pack_dgrad_weight(w, CoutP=None, CinP=None):
    """w (Cout,taps,Cin) fp32 -> (CinP,taps,CoutP) bf16 with the tap order reversed
    (fp32 storage mode: fp32 (CinP,taps,CoutP))."""
    require_cuda(w)
    assert w.dtype == F32 and w.is_contiguous() and w.dim() == 3
    Cout, taps, Cin = w.shape
    CoutP, CinP = CoutP or Cout, CinP or Cin
    if STORE == F32:
        wp = torch.zeros((CinP, taps, CoutP), device=w.device, dtype=F32)
        wp[:Cin, :, :Cout] = w.flip(1).permute(2, 1, 0)           # tap order reversed, channels transposed
        return wp
    return _pack_dgrad_bf16(w, CoutP, CinP)


def unpack_wgrad(dwp, Cout, Cin):
    """(CoutP,taps,CinP) fp32 -> (Cout,taps,Cin) fp32 (crop of the channel padding)."""
    require_cuda(dwp)
    CoutP, taps, CinP = dwp.shape
    if CoutP == Cout and CinP == Cin:
        return dwp
    dst = torch.empty((Cout, taps, Cin), device=dwp.device, dtype=F32)
    check(lib().t2v_unpack_wgrad_padded(ptr(dwp), ptr(dst), Cout, taps, Cin, CinP, stream()),
          "t2v_unpack_wgrad_padded")
    return dst


# ------------------------------------------------------------------------------------- general conv (TGAN / TCWYT)
def gconv_out_extent(i, k, s, p):
    return (i + 2 * p - k) // s + 1


def _ggeom(N, in_sp, Cin, Cout, k, s, p):
    out_sp = [gconv_out_extent(i, kk, ss, pp) for i, kk, ss, pp in zip(in_sp, k, s, p)]
    return GconvGeom(N, in_sp[0], in_sp[1], in_sp[2], out_sp[0], out_sp[1], out_sp[2], Cin, Cout, k[0], k[1], k[2],
                     s[0], s[1], s[2], p[0], p[1], p[2]), out_sp


def gconv_pack(w3):
    """operand of the general convolution kernels: bf16 cast of the fp32 (Cout,taps,Cin) weight, or the fp32 weight
    itself in the fp32 storage mode (CUDA-core FMA: exact)"""
    require_cuda(w3)
    return w3.contiguous() if STORE == F32 else cast_bf16(w3.contiguous())


# --- kernel-4 / stride-2 / padding-1 layers on the tcgen05 engine (csrc/s2d.cu: shifted space-to-depth blocks) --------
GCONV_TC = True          # False: every general convolution on the CUDA-core kernels (the reference of the tests)


def round16(c):
    return (c + 15) // 16 * 16


def s2d_modes(k, s, p, in_sp):
    """per-axis mode of the block formulation: 2 = kernel 4 / stride 2 / padding 1 on an even extent, 1 = kernel 1 /
    stride 1 / padding 0; None when the layer is of another kind (it stays on the CUDA-core general convolution)"""
    modes = []
    for kk, ss, pp, e in zip(k, s, p, in_sp):
        if (kk, ss, pp) == (4, 2, 1) and e % 2 == 0:
            modes.append(2)
        elif (kk, ss, pp) == (1, 1, 0):
            modes.append(1)
        else:
            return None
    return tuple(modes) if 2 in modes else None


def _s2d_phases(modes):
    return 2 ** sum(1 for m in modes if m == 2)


def s2d_block_extents(sp, modes):
    return tuple(e // 2 + 1 if m == 2 else e for e, m in zip(sp, modes))


def s2d_shift(x, modes, creal=None):
    """x (N,D,H,W,C) -> block tensor (N,D',H',W',round16(P*creal)): block b of a strided axis = samples (2b-1, 2b)"""
    require_cuda(x)
    N, D, H, W, C = x.shape
    creal = C if creal is None else creal
    Cp = round16(_s2d_phases(modes) * creal)
    Db, Hb, Wb = s2d_block_extents((D, H, W), modes)
    assert x.is_contiguous()
    xs = torch.empty((N, Db, Hb, Wb, Cp), device=x.device, dtype=x.dtype)
    check(lib().t2v_s2d_shift(ptr(x), ptr(xs), N, D, H, W, C, creal, modes[0], modes[1], modes[2], Cp,
                              x.element_size(), stream()), "t2v_s2d_shift")
    return xs


def d2s_shift(xs, modes, sp, C, creal=None):
    """inverse of s2d_shift: block tensor -> (N,D,H,W,C) (channels >= creal zero)"""
    require_cuda(xs)
    N, Cp = xs.shape[0], xs.shape[-1]
    creal = C if creal is None else creal
    assert xs.is_contiguous() and tuple(xs.shape[1:4]) == s2d_block_extents(sp, modes), (xs.shape, sp, modes)
    x = torch.empty((N, sp[0], sp[1], sp[2], C), device=xs.device, dtype=xs.dtype)
    check(lib().t2v_d2s_shift(ptr(xs), ptr(x), N, sp[0], sp[1], sp[2], C, creal, modes[0], modes[1], modes[2], Cp,
                              xs.element_size(), stream()), "t2v_d2s_shift")
    return x


def s2d_embed_weight(w, modes, creal=None, transposed=False):
    """w bf16 (Co, k taps, Ci) -> bf16 (Co, 3^s, Cp) | transposed (Cp, 3^s reversed, Co); cached on the pack tensor"""
    require_cuda(w)
    Co, taps, Ci = w.shape
    creal = Ci if creal is None else creal
    key = (modes, creal, transposed)
    cache = getattr(w, "_t2v_s2d", None)
    if cache is None:
        cache = {}
        w._t2v_s2d = cache
    if key in cache:
        return cache[key]
    assert w.dtype == BF16 and w.is_contiguous() and taps == 4 ** sum(1 for m in modes if m == 2)
    Cp = round16(_s2d_phases(modes) * creal)
    ntap = 3 ** sum(1 for m in modes if m == 2)
    we = torch.empty((Cp, ntap, Co) if transposed else (Co, ntap, Cp), device=w.device, dtype=BF16)
    check(lib().t2v_s2d_embed_weight(ptr(w), ptr(we), Co, Ci, creal, Cp, modes[0], modes[1], modes[2],
                                     1 if transposed else 0, stream()), "t2v_s2d_embed_weight")
    cache[key] = we
    return we


def s2d_extract_wgrad(dwe, modes, Ci, creal=None):
    """dwe fp32 (Co, 3^s, Cp) -> dw fp32 (Co, k taps, Ci)"""
    require_cuda(dwe)
    Co, ntap, Cp = dwe.shape
    creal = Ci if creal is None else creal
    taps = 4 ** sum(1 for m in modes if m == 2)
    assert dwe.dtype == F32 and dwe.is_contiguous()
    dw = torch.empty((Co, taps, Ci), device=dwe.device, dtype=F32)
    check(lib().t2v_s2d_extract_wgrad(ptr(dwe), ptr(dw), Co, Ci, creal, Cp, modes[0], modes[1], modes[2], stream()),
          "t2v_s2d_extract_wgrad")
    return dw


def s2d_tile_bias(bias, creal, phases, Cp):
    """fp32 (>= creal,) -> fp32 (Cp,): out[ph * creal + c] = bias[c] (the bias of a transposed convolution in block form)"""
    require_cuda(bias)
    out = torch.empty((Cp,), device=bias.device, dtype=F32)
    check(lib().t2v_s2d_tile_bias(ptr(bias), ptr(out), creal, phases, Cp, stream()), "t2v_s2d_tile_bias")
    return out


def _win9(in_sp, lo_hi):
    return _i32(in_sp[0], in_sp[1], in_sp[2], lo_hi[0][0], lo_hi[0][1], lo_hi[1][0], lo_hi[1][1], lo_hi[2][0],
                lo_hi[2][1])


def conv_fprop_win(x, w, bias, out_sp, k, lo_hi, relu=False, out_f32=False):
    """windowed implicit GEMM: x (N,iD,iH,iW,Cin) bf16, w (Cout, kd*kh*kw, Cin) bf16 -> y (N,*out_sp,Cout); tap t of an
    axis reads x at o + t - k/2 (zero outside x), only taps lo <= t < hi are live"""
    require_cuda(x, w, bias)
    N, Cin = x.shape[0], x.shape[-1]
    Cout = w.shape[0]
    assert x.dtype == BF16 and w.dtype == BF16 and x.is_contiguous() and w.is_contiguous()
    assert w.shape[1] == k[0] * k[1] * k[2] and w.shape[2] == Cin, (w.shape, k, Cin)
    assert bias is None or (bias.dtype == F32 and bias.numel() == Cout)
    y = torch.empty((N, out_sp[0], out_sp[1], out_sp[2], Cout), device=x.device, dtype=F32 if out_f32 else BF16)
    g = _geom(N, out_sp[0], out_sp[1], out_sp[2], Cin, Cout, k)
    flags = (_lib.EPI_RELU if relu else 0) | (_lib.EPI_OUT_F32 if out_f32 else 0)
    check(lib().t2v_conv_fprop_win(ctypes.byref(g), _win9(x.shape[1:4], lo_hi), ptr(x), ptr(w), ptr(bias), ptr(y), flags,
                                   stream()), "t2v_conv_fprop_win")
    return y


def conv_wgrad_win(dy, x, k, lo_hi):
    """dw (Cout, kd*kh*kw, Cin) fp32 = sum_pos dy[pos, co] x[pos + t - k/2, ci] over the live taps (others zero)"""
    require_cuda(dy, x)
    N, Cout, Cin = dy.shape[0], dy.shape[-1], x.shape[-1]
    assert dy.dtype == BF16 and x.dtype == BF16 and dy.is_contiguous() and x.is_contiguous() and x.shape[0] == N
    dw = torch.empty((Cout, k[0] * k[1] * k[2], Cin), device=x.device, dtype=F32)
    g = _geom(N, dy.shape[1], dy.shape[2], dy.shape[3], Cin, Cout, k)
    check(lib().t2v_conv_wgrad_win(ctypes.byref(g), _win9(x.shape[1:4], lo_hi), ptr(dy), ptr(x), ptr(dw), 0, stream()),
          "t2v_conv_wgrad_win")
    return dw


def _s2d_engine_args(modes, dgrad=False):
    ke = tuple(3 if m == 2 else 1 for m in modes)
    live = (0, 2) if dgrad else (1, 3)
    return ke, tuple(live if m == 2 else (0, 1) for m in modes)


def _s2d_route(t, k, s, p, in_sp):
    return s2d_modes(k, s, p, in_sp) if (GCONV_TC and t.dtype == BF16) else None


def transpose_flip(w, flat=False):
    """bf16 (Co, taps, Ci) -> bf16 (Ci, taps reversed, Co), or with flat=True the plain matrix transpose
    (taps * Ci, 1, Co) of the pack read as (Co, taps * Ci); cached on the pack tensor"""
    require_cuda(w)
    cache = getattr(w, "_t2v_wT", None)
    if cache is None:
        cache = {}
        w._t2v_wT = cache
    if flat in cache:
        return cache[flat]
    Co, taps, Ci = w.shape
    if flat:
        taps, Ci = 1, taps * Ci
    assert w.dtype == BF16 and w.is_contiguous()
    wT = torch.empty((Ci, taps, Co), device=w.device, dtype=BF16)
    check(lib().t2v_transpose_flip_bf16(ptr(w), ptr(wT), Co, taps, Ci, stream()), "t2v_transpose_flip_bf16")
    cache[flat] = wT
    return wT


def window_rows(x, k):
    """x (N,D,H,W,C) -> (N, kd*kh*kw*C): the corner window x[:, :kd, :kh, :kw]"""
    require_cuda(x)
    N, D, H, W, C = x.shape
    assert x.is_contiguous()
    rows = torch.empty((N, k[0] * k[1] * k[2] * C), device=x.device, dtype=x.dtype)
    check(lib().t2v_window_rows(ptr(x), ptr(rows), N, D, H, W, C, k[0], k[1], k[2], x.element_size(), 0, stream()),
          "t2v_window_rows")
    return rows


def window_rows_scatter(rows, sp, C, k):
    """adjoint of window_rows: zeros (N,*sp,C) with the corner window filled from rows"""
    require_cuda(rows)
    N = rows.shape[0]
    assert rows.is_contiguous() and rows.shape[1] == k[0] * k[1] * k[2] * C
    x = torch.empty((N, sp[0], sp[1], sp[2], C), device=rows.device, dtype=rows.dtype)
    check(lib().t2v_window_rows(ptr(x), ptr(rows), N, sp[0], sp[1], sp[2], C, k[0], k[1], k[2], rows.element_size(), 1,
                                stream()), "t2v_window_rows")
    return x


def _engine_route(t, k, s, p, in_sp):
    """'same': every axis kernel 1 / padding 0 or kernel 3 / padding 1 at stride 1 (the engine's own domain);
    'full': the kernel covers the whole input (padding 0, one output position): a Linear layer over taps * Cin;
    'window': one output position whose kernel covers a corner window of the input: gather the window, then 'full'"""
    if not (GCONV_TC and t.dtype == BF16):
        return None
    if all(ss == 1 and (kk, pp) in ((1, 0), (3, 1)) for kk, ss, pp in zip(k, s, p)):
        return "same"
    if tuple(k) == tuple(in_sp) and all(pp == 0 for pp in p):
        return "full"
    if all(pp == 0 for pp in p) and all((i - kk) // ss == 0 for i, kk, ss in zip(in_sp, k, s)):
        return "window"                          # one output position reading the corner window of the input
    return None


def gconv_fprop(x, w, bias, k, s, p, out_f32=False, cin_real=None):
    """Strided convolution: x (N,Di,Hi,Wi,Cin), w (Cout,taps,Cin) (both bf16, or both fp32) -> y (N,Do,Ho,Wo,Cout)."""
    require_cuda(x, w, bias)
    N, Di, Hi, Wi, Cin = x.shape
    Cout = w.shape[0]
    _act(x, w)
    assert x.dtype == w.dtype
    assert w.shape[1] == k[0] * k[1] * k[2] and w.shape[2] == Cin, (w.shape, k, Cin)
    g, osp = _ggeom(N, (Di, Hi, Wi), Cin, Cout, k, s, p)
    modes = _s2d_route(x, k, s, p, (Di, Hi, Wi))
    if modes is not None:                       # k4 s2 p1: dense kernel-2 implicit GEMM over the shifted block tensor
        ke, live = _s2d_engine_args(modes)
        return conv_fprop_win(s2d_shift(x, modes, cin_real), s2d_embed_weight(w, modes, cin_real), bias, osp, ke, live,
                              out_f32=out_f32)
    route = _engine_route(x, k, s, p, (Di, Hi, Wi))
    if route == "same":
        return conv_fprop(x, w, bias, k=tuple(k), out_f32=out_f32)
    if route == "window":
        x, route = window_rows(x, k), "full"
    if route == "full":
        return conv_fprop(x.view(N, 1, 1, 1, -1), w.view(Cout, 1, -1), bias, k=(1, 1, 1), out_f32=out_f32)
    out_f32 = out_f32 or x.dtype == F32
    y = torch.empty((N, osp[0], osp[1], osp[2], Cout), device=x.device, dtype=F32 if out_f32 else BF16)
    check(_lib.typed("t2v_gconv_fprop", x)(ctypes.byref(g), ptr(x), ptr(w), ptr(bias), ptr(y), 1 if out_f32 else 0,
                                           stream()), "t2v_gconv_fprop")
    return y


def gconv_dgrad(dy, w, bias, in_sp, k, s, p, out_f32=False, cin_real=None):
    """Data gradient of gconv_fprop == forward of a transposed convolution: dy (N,Do,Ho,Wo,Cout),
    w (Cout,taps,Cin) -> dx (N,Di,Hi,Wi,Cin); in_sp = (Di,Hi,Wi); bias fp32 (Cin,) or None."""
    require_cuda(dy, w, bias)
    N, Cout = dy.shape[0], dy.shape[-1]
    Cin = w.shape[2]
    _act(dy, w)
    assert dy.dtype == w.dtype and w.shape[0] == Cout
    g, osp = _ggeom(N, tuple(in_sp), Cin, Cout, k, s, p)
    assert tuple(osp) == tuple(dy.shape[1:4]), (osp, dy.shape)
    modes = _s2d_route(dy, k, s, p, tuple(in_sp))
    if modes is not None:                       # the same GEMM with the transposed pack, then the inverse block permute
        ke, live = _s2d_engine_args(modes, dgrad=True)
        creal = Cin if cin_real is None else cin_real
        weT = s2d_embed_weight(w, modes, creal, transposed=True)
        be = None if bias is None else s2d_tile_bias(bias, creal, _s2d_phases(modes), weT.shape[0])
        dxs = conv_fprop_win(dy, weT, be, s2d_block_extents(tuple(in_sp), modes), ke, live, out_f32=out_f32)
        return d2s_shift(dxs, modes, tuple(in_sp), Cin, creal)
    route = _engine_route(dy, k, s, p, tuple(in_sp))
    if route == "window" and bias is not None:
        route = None             # a transposed convolution's bias also covers the positions outside the window
    if route == "same":
        return conv_fprop(dy, transpose_flip(w), bias, k=tuple(k), out_f32=out_f32)
    if route in ("full", "window"):
        taps = w.shape[1]
        be = None if bias is None else s2d_tile_bias(bias, Cin, taps, taps * Cin)
        dx = conv_fprop(dy.view(N, 1, 1, 1, Cout), transpose_flip(w, flat=True), be, k=(1, 1, 1),
                        out_f32=out_f32)
        if route == "window":
            return window_rows_scatter(dx.view(N, taps * Cin), tuple(in_sp), Cin, k)
        return dx.view(N, in_sp[0], in_sp[1], in_sp[2], Cin)
    out_f32 = out_f32 or dy.dtype == F32
    dx = torch.empty((N, in_sp[0], in_sp[1], in_sp[2], Cin), device=dy.device, dtype=F32 if out_f32 else BF16)
    check(_lib.typed("t2v_gconv_dgrad", dy)(ctypes.byref(g), ptr(dy), ptr(w), ptr(bias), ptr(dx), 1 if out_f32 else 0,
                                            stream()), "t2v_gconv_dgrad")
    return dx


def gconv_wgrad(dy, x, k, s, p, cin_real=None):
    """dw (Cout,taps,Cin) fp32 = sum_pos dy[pos,co] * x[in(pos,tap),ci]."""
    require_cuda(dy, x)
    N, Di, Hi, Wi, Cin = x.shape
    Cout = dy.shape[-1]
    _act(dy, x)
    assert dy.dtype == x.dtype
    g, osp = _ggeom(N, (Di, Hi, Wi), Cin, Cout, k, s, p)
    assert tuple(osp) == tuple(dy.shape[1:4]), (osp, dy.shape)
    modes = _s2d_route(x, k, s, p, (Di, Hi, Wi))
    if modes is not None:
        ke, live = _s2d_engine_args(modes)
        dwe = conv_wgrad_win(dy, s2d_shift(x, modes, cin_real), ke, live)
        return s2d_extract_wgrad(dwe, modes, Cin, cin_real)
    route = _engine_route(x, k, s, p, (Di, Hi, Wi))
    if route == "same":
        return conv_wgrad(dy, x, k=tuple(k))
    if route == "window":
        x, route = window_rows(x, k), "full"
    if route == "full":
        taps = k[0] * k[1] * k[2]
        return conv_wgrad(dy.view(N, 1, 1, 1, Cout), x.view(N, 1, 1, 1, taps * Cin), k=(1, 1, 1)).view(Cout, taps, Cin)
    dw = torch.empty((Cout, k[0] * k[1] * k[2], Cin), device=x.device, dtype=F32)
    check(_lib.typed("t2v_gconv_wgrad", dy)(ctypes.byref(g), ptr(dy), ptr(x), ptr(dw), 0, stream()), "t2v_gconv_wgrad")
    return dw


def _unary(name, x, *extra):
    require_cuda(x)
    _act(x)
    y = torch.empty_like(x)
    check(_lib.typed(name, x)(ptr(x), ptr(y), x.numel(), *extra, stream()), name)
    return y


def _binary(name, a, b, *extra):
    require_cuda(a, b)
    _act(a, b)
    assert a.dtype == b.dtype and a.numel() == b.numel(), (a.dtype, b.dtype, a.shape, b.shape)
    y = torch.empty_like(a)
    check(_lib.typed(name, a)(ptr(a), ptr(b), ptr(y), a.numel(), *extra, stream()), name)
    return y


def leaky_relu_fwd(x, slope):
    return _unary("t2v_leaky_relu_fwd", x, float(slope))


def leaky_relu_bwd(dy, ref, slope):
    return _binary("t2v_leaky_relu_bwd", dy, ref, float(slope))


def tanh_fwd(x):
    return _unary("t2v_tanh_fwd", x)


def tanh_bwd(dy, y):
    return _binary("t2v_tanh_bwd", dy, y)


# ------------------------------------------------------------------------------------- pointwise / pooling
def relu_fwd(x):
    return _unary("t2v_relu_fwd", x)


def relu_bwd(dy, ref):
    return _binary("t2v_relu_bwd", dy, ref)


def scale(x, s):
    """y = s * x; s: 0-d / 1-element fp32 CUDA tensor"""
    require_cuda(x, s)
    _act(x)
    assert s.dtype == F32 and s.numel() == 1
    y = torch.empty_like(x)
    check(_lib.typed("t2v_scale", x)(ptr(x), ptr(s), ptr(y), x.numel(), stream()), "t2v_scale")
    return y


def scale_add(o, x, s=None):
    """y = s * o + x (s None: y = o + x)"""
    require_cuda(o, x, s)
    _act(o, x)
    assert o.dtype == x.dtype and o.numel() == x.numel() and (s is None or (s.dtype == F32 and s.numel() == 1))
    y = torch.empty_like(x)
    check(_lib.typed("t2v_scale_add", x)(ptr(o), ptr(x), ptr(s), ptr(y), x.numel(), stream()), "t2v_scale_add")
    return y


def dot(a, b):
    """0-d fp32 = sum a * b"""
    require_cuda(a, b)
    _act(a, b)
    assert a.dtype == b.dtype and a.numel() == b.numel()
    out = torch.empty((), device=a.device, dtype=F32)
    check(_lib.typed("t2v_dot", a)(ptr(a), ptr(b), ptr(out), a.numel(), stream()), "t2v_dot")
    return out


def cl_slice_f32(x, c):
    """CL (..., Cp) -> fp32 (..., c): the first c channels"""
    require_cuda(x)
    _act(x)
    Cp = x.shape[-1]
    y = torch.empty(tuple(x.shape[:-1]) + (c,), device=x.device, dtype=F32)
    check(_lib.typed("t2v_cl_slice_f32", x)(ptr(x), ptr(y), x.numel() // Cp, Cp, c, stream()), "t2v_cl_slice_f32")
    return y


def f32_pad_cl(x, Cp, dtype=None):
    """fp32 (..., c) -> CL storage (..., Cp), zero channel padding"""
    require_cuda(x)
    assert x.dtype == F32 and x.is_contiguous()
    c = x.shape[-1]
    y = torch.empty(tuple(x.shape[:-1]) + (Cp,), device=x.device, dtype=dtype or STORE)
    check(_lib.typed("t2v_f32_pad_cl", y)(ptr(x), ptr(y), x.numel() // c, Cp, c, stream()), "t2v_f32_pad_cl")
    return y


def pool_out_shape(in_shape, kernel, stride, pad):
    N, D, H, W, C = in_shape
    o = [(s + 2 * p - k) // st + 1 for s, k, st, p in zip((D, H, W), kernel, stride, pad)]
    return (N, o[0], o[1], o[2], C)


def avgpool_fwd(x, kernel, stride, pad, residual=None):
    require_cuda(x, residual)
    _act(x, residual)
    y = torch.empty(pool_out_shape(x.shape, kernel, stride, pad), device=x.device, dtype=x.dtype)
    assert residual is None or (residual.shape == y.shape and residual.dtype == x.dtype)
    check(_lib.typed("t2v_avgpool_fwd", x)(ptr(x), ptr(residual), ptr(y), _i32(*x.shape), _i32(*kernel),
                                           _i32(*stride), _i32(*pad), stream()), "t2v_avgpool_fwd")
    return y


def avgpool_bwd(dy, in_shape, kernel, stride, pad):
    require_cuda(dy)
    _act(dy)
    assert tuple(dy.shape) == tuple(pool_out_shape(in_shape, kernel, stride, pad))
    dx = torch.empty(tuple(in_shape), device=dy.device, dtype=dy.dtype)
    check(_lib.typed("t2v_avgpool_bwd", dy)(ptr(dy), ptr(dx), _i32(*in_shape), _i32(*kernel), _i32(*stride),
                                            _i32(*pad), stream()), "t2v_avgpool_bwd")
    return dx


def upsample2x_fwd(x):
    require_cuda(x)
    N, D, H, W, C = x.shape
    _act(x)
    assert D == 1
    y = torch.empty((N, 1, 2 * H, 2 * W, C), device=x.device, dtype=x.dtype)
    check(_lib.typed("t2v_upsample2x_fwd", x)(ptr(x), ptr(y), N, H, W, C, stream()), "t2v_upsample2x_fwd")
    return y


def upsample2x_bwd(dy):
    require_cuda(dy)
    N, D, H2, W2, C = dy.shape
    _act(dy)
    assert D == 1
    dx = torch.empty((N, 1, H2 // 2, W2 // 2, C), device=dy.device, dtype=dy.dtype)
    check(_lib.typed("t2v_upsample2x_bwd", dy)(ptr(dy), ptr(dx), N, H2 // 2, W2 // 2, C, stream()),
          "t2v_upsample2x_bwd")
    return dx


def nchw_to_cl(x, Cp):
    """fp32 (N,C,D,H,W) -> CL storage (N,D,H,W,Cp), padded channels zero."""
    require_cuda(x)
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 5
    N, C, D, H, W = x.shape
    y = torch.empty((N, D, H, W, Cp), device=x.device, dtype=STORE)
    check(_lib.typed("t2v_nchw_to_cl", y)(ptr(x), ptr(y), N, C, D * H * W, Cp, stream()), "t2v_nchw_to_cl")
    return y


def rgb_to_cl(x, want4=True):
    """fp32 (N,3,D,H,W) -> bf16 (N,D,H,W,16) and (optionally) bf16 (N,D,H,W,4), zero padded, in one pass
    (bf16 storage only: the direct stem kernels read the 4-channel copy)."""
    require_cuda(x)
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 5 and x.shape[1] == 3 and STORE == BF16
    N, C, D, H, W = x.shape
    y16 = torch.empty((N, D, H, W, 16), device=x.device, dtype=BF16)
    y4 = torch.empty((N, D, H, W, 4), device=x.device, dtype=BF16) if want4 else None
    check(lib().t2v_rgb_to_cl(ptr(x), ptr(y16), ptr(y4), N, D * H * W, stream()), "t2v_rgb_to_cl")
    return y16, y4


def cl_to_nchw(x, C):
    """CL (N,D,H,W,Cp) -> fp32 (N,C,D,H,W) (first C channels)."""
    require_cuda(x)
    _act(x)
    assert x.dim() == 5
    N, D, H, W, Cp = x.shape
    y = torch.empty((N, C, D, H, W), device=x.device, dtype=F32)
    check(_lib.typed("t2v_cl_to_nchw", x)(ptr(x), ptr(y), N, C, D * H * W, Cp, stream()), "t2v_cl_to_nchw")
    return y


def im2col3(x, Kp):
    """fp32 (N,C,D,H,W) -> CL storage (N,D,H,W,Kp), col[..., tap*C + c] = x[c] shifted by tap (3^3, zero padded)."""
    require_cuda(x)
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 5
    N, C, D, H, W = x.shape
    col = torch.empty((N, D, H, W, Kp), device=x.device, dtype=STORE)
    check(_lib.typed("t2v_im2col3", col)(ptr(x), ptr(col), N, C, D, H, W, Kp, stream()), "t2v_im2col3")
    return col


def col2im3(dcol, C):
    """adjoint of im2col3: CL (N,D,H,W,Kp) -> fp32 (N,C,D,H,W)."""
    require_cuda(dcol)
    _act(dcol)
    assert dcol.dim() == 5
    N, D, H, W, Kp = dcol.shape
    dx = torch.empty((N, C, D, H, W), device=dcol.device, dtype=F32)
    check(_lib.typed("t2v_col2im3", dcol)(ptr(dcol), ptr(dx), N, C, D, H, W, Kp, stream()), "t2v_col2im3")
    return dx


def sum_rows(x, out=None):
    """CL (..., C) -> fp32 (C,) sum over all leading dims; with `out` (fp32 (C,)): out += the sums."""
    require_cuda(x, out)
    _act(x)
    C = x.shape[-1]
    if out is not None:
        assert out.dtype == F32 and out.numel() == C and out.is_contiguous()
        check(_lib.typed("t2v_sum_rows_acc", x)(ptr(x), ptr(out), x.numel() // C, C, stream()), "t2v_sum_rows_acc")
        return out
    out = torch.empty((C,), device=x.device, dtype=F32)
    check(_lib.typed("t2v_sum_rows", x)(ptr(x), ptr(out), x.numel() // C, C, stream()), "t2v_sum_rows")
    return out


def sum_spatial(x):
    """CL (N,D,H,W,C) -> fp32 (N,C)."""
    require_cuda(x)
    _act(x)
    N, C = x.shape[0], x.shape[-1]
    out = torch.empty((N, C), device=x.device, dtype=F32)
    check(_lib.typed("t2v_sum_spatial", x)(ptr(x), ptr(out), N, x.numel() // (N * C), C, stream()), "t2v_sum_spatial")
    return out


def broadcast_spatial(g, shape):
    """fp32 (N,C) -> CL storage `shape` = (N,D,H,W,C)."""
    require_cuda(g)
    assert g.dtype == F32 and g.is_contiguous()
    N, C = g.shape
    y = torch.empty(tuple(shape), device=g.device, dtype=STORE)
    check(_lib.typed("t2v_broadcast_spatial", y)(ptr(g), ptr(y), N, y.numel() // (N * C), C, stream()),
          "t2v_broadcast_spatial")
    return y


# ------------------------------------------------------------------------------------- BatchNorm (train)
def bn_forward(x, gamma, beta, running_mean, running_var, relu, up, eps=1e-5, momentum=0.1, training=True):
    """x (N,1,H,W,C) CL -> y (N,1,up*H,up*W,C), plus (mean_invstd, scale_shift) fp32 [2C] for backward.
    training=False normalises with the running statistics (no update).  `relu` is the fused activation code:
    0/False none, 1/True ReLU, 2 LeakyReLU(0.2).  With up == 1 any CL shape is accepted (statistics over all
    leading dims: BatchNorm1d/2d/3d)."""
    require_cuda(x, gamma, beta)
    shape0 = tuple(x.shape)
    if up == 1 and x.shape[1] != 1:
        x = x.reshape(-1, 1, 1, 1, x.shape[-1])
    N, D, H, W, C = x.shape
    _act(x)
    assert D == 1
    dev = x.device
    mean_invstd = torch.empty((2 * C,), device=dev, dtype=F32)
    scale_shift = torch.empty((2 * C,), device=dev, dtype=F32)
    if training:
        stats = torch.empty((2 * C,), device=dev, dtype=F32)
        P = N * H * W
        check(_lib.typed("t2v_bn_stats", x)(ptr(x), ptr(stats), P, C, stream()), "t2v_bn_stats")
        check(lib().t2v_bn_finalize(ptr(stats), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
                                    ptr(mean_invstd), ptr(scale_shift), C, P, eps, momentum, stream()),
              "t2v_bn_finalize")
    else:
        # stats := {P*mean, P*(var+mean^2)} with P = 1 reproduces mean / var in the finalize kernel
        stats = torch.cat((running_mean, running_var + running_mean * running_mean)).contiguous()
        check(lib().t2v_bn_finalize(ptr(stats), ptr(gamma), ptr(beta), None, None, ptr(mean_invstd),
                                    ptr(scale_shift), C, 1, eps, momentum, stream()), "t2v_bn_finalize")
    y = torch.empty((N, 1, up * H, up * W, C), device=dev, dtype=x.dtype)
    check(_lib.typed("t2v_bn_apply", x)(ptr(x), ptr(scale_shift), ptr(y), N, H, W, C, int(relu), up, stream()),
          "t2v_bn_apply")
    if up == 1:
        y = y.view(shape0)
    return y, mean_invstd, scale_shift


def bn_backward(dy, x, mean_invstd, scale_shift, relu, up):
    """-> dx (x-shaped CL), dgamma fp32 [C], dbeta fp32 [C]."""
    require_cuda(dy, x)
    shape0 = tuple(x.shape)
    if up == 1 and x.shape[1] != 1:
        x = x.reshape(-1, 1, 1, 1, x.shape[-1])
        dy = dy.reshape(x.shape)
    N, D, H, W, C = x.shape
    _act(dy, x)
    assert dy.dtype == x.dtype and tuple(dy.shape) == (N, 1, up * H, up * W, C)
    red = torch.empty((2 * C,), device=x.device, dtype=F32)
    dx = torch.empty_like(x)
    check(_lib.typed("t2v_bn_bwd", x)(ptr(dy), ptr(x), ptr(scale_shift), ptr(mean_invstd), ptr(red), ptr(dx), N, H, W,
                                      C, int(relu), up, stream()), "t2v_bn_bwd")
    return dx.view(shape0), red[C:], red[:C]


def bn_backward_backward(dy, x, mean_invstd, scale_shift, ggx, ggamma, ggbeta, relu, up):
    """Double backward of bn_backward (up == 1): upstream ggx (x-shaped CL, w.r.t. dx) and ggamma / ggbeta (fp32 [C]
    w.r.t. dgamma / dbeta, None = zero) -> gx (w.r.t. x), gdy (w.r.t. dy), both x-shaped CL, and dgamma fp32 [C]
    (w.r.t. gamma)."""
    require_cuda(dy, x, ggx, ggamma, ggbeta)
    _act(dy, x, ggx)
    assert up == 1, "the double backward has no upsampling form"
    C = x.shape[-1]
    P = x.numel() // C
    assert dy.dtype == x.dtype == ggx.dtype and dy.numel() == ggx.numel() == x.numel()
    for t in (ggamma, ggbeta):
        assert t is None or (t.dtype == F32 and t.is_contiguous() and t.numel() == C)
    red = torch.empty((5 * C,), device=x.device, dtype=F32)
    gx, gdy = torch.empty_like(x), torch.empty_like(x)
    dgamma = torch.empty((C,), device=x.device, dtype=F32)
    check(_lib.typed("t2v_bn_bwd_bwd", x)(ptr(dy), ptr(x), ptr(ggx), ptr(ggamma), ptr(ggbeta), ptr(scale_shift),
                                          ptr(mean_invstd), ptr(red), ptr(gx), ptr(gdy), ptr(dgamma), P, C, int(relu),
                                          up, stream()), "t2v_bn_bwd_bwd")
    return gx, gdy, dgamma


# ------------------------------------------------------------------------------------- non-local attention core
def attention_fwd(theta, phi, g, c8, c2):
    """theta/phi (N,D,H,W,C8p), g (N,D,H,W,C2p) bf16 -> o (N,D,H,W,C2p): softmax(theta . maxpool(phi)^T) . maxpool(g)."""
    require_cuda(theta, phi, g)
    N, D, H, W, C8p = theta.shape
    C2p = g.shape[-1]
    assert theta.dtype == BF16 and theta.is_contiguous() and phi.is_contiguous() and g.is_contiguous()
    o = torch.empty((N, D, H, W, C2p), device=theta.device, dtype=BF16)
    check(lib().t2v_attention_fwd(ptr(theta), ptr(phi), ptr(g), ptr(o), N, D, H, W, c8, c2, C8p, C2p, stream()),
          "t2v_attention_fwd")
    return o


def attention_bwd(theta, phi, g, dout, c8, c2):
    require_cuda(theta, phi, g, dout)
    N, D, H, W, C8p = theta.shape
    C2p = g.shape[-1]
    assert dout.dtype == BF16 and dout.is_contiguous()
    dtheta, dphi, dg = torch.empty_like(theta), torch.empty_like(phi), torch.empty_like(g)
    if attention_is_large(D, H, W):            # beyond one CTA per map: the two-launch form with a statistics workspace
        stats = torch.empty((N * D * H * W * 3,), device=theta.device, dtype=F32)
        check(lib().t2v_attention_bwd_large(ptr(theta), ptr(phi), ptr(g), ptr(dout), ptr(dtheta), ptr(dphi), ptr(dg),
                                            ptr(stats), N, D, H, W, c8, c2, C8p, C2p, stream()),
              "t2v_attention_bwd_large")
        return dtheta, dphi, dg
    check(lib().t2v_attention_bwd(ptr(theta), ptr(phi), ptr(g), ptr(dout), ptr(dtheta), ptr(dphi), ptr(dg), N, D, H, W,
                                  c8, c2, C8p, C2p, stream()), "t2v_attention_bwd")
    return dtheta, dphi, dg


def attention_is_large(D, H, W):
    """pooled keys of a map beyond the one-CTA backward kernel (2 * Kp > 512)"""
    return 2 * D * (H // 2) * (W // 2) > 512


def attention_fused_ok(D, H, W, c8, c2):
    """shapes the fused generator-attention kernels take: any map of <= 1024 voxels with c8 <= 8, c2 <= 16; larger maps
    (up to 2560 pooled keys: shared memory) in the compile-time configuration c8 = 4, c2 = 16"""
    if c8 > 8 or c2 > 16:
        return False
    if D * H * W <= 1024:
        return True
    return c8 == 4 and c2 == 16 and D * (H // 2) * (W // 2) <= 2560


# ------------------------------------------------------------------------------------- render / index
def render_fwd(pre, B, T, C):
    """pre (B*T,1,H,W,Cp) bf16 -> tanh -> fp32 (B,C,T,H,W)."""
    require_cuda(pre)
    BT, D, H, W, Cp = pre.shape
    _act(pre)
    assert BT == B * T and D == 1
    y = torch.empty((B, C, T, H, W), device=pre.device, dtype=F32)
    check(_lib.typed("t2v_render_fwd", pre)(ptr(pre), ptr(y), B, T, H, W, C, Cp, stream()), "t2v_render_fwd")
    return y


def render_bwd(dy, y, Cp):
    require_cuda(dy, y)
    B, C, T, H, W = y.shape
    assert dy.dtype == F32 and dy.is_contiguous() and y.is_contiguous()
    dpre = torch.empty((B * T, 1, H, W, Cp), device=y.device, dtype=STORE)
    check(_lib.typed("t2v_render_bwd", dpre)(ptr(dy), ptr(y), ptr(dpre), B, T, H, W, C, Cp, stream()), "t2v_render_bwd")
    return dpre


def _bt_args(bt, T, st):
    """bt: python int, or a device int32 tensor (CUDA-graph replays).  With a tensor the frame count must not
    depend on its value: T divisible by st."""
    if isinstance(bt, torch.Tensor):
        assert bt.is_cuda and bt.dtype == torch.int32 and T % st == 0, "device-side bt needs T % st == 0"
        return 0, bt
    return int(bt), None


def gather_frames(x, B, T, bt, sn=2, st=2):
    """x (B*T,1,H,W,C) merged-frame map -> frames (b*sn, bt + t*st): (Bo*To,1,H,W,C)."""
    require_cuda(x)
    assert x.is_contiguous() and x.shape[0] == B * T
    bt, bt_dev = _bt_args(bt, T, st)
    Bo = (B + sn - 1) // sn
    To = (T - bt + st - 1) // st if T > bt else 0
    y = torch.empty((Bo * To,) + tuple(x.shape[1:]), device=x.device, dtype=x.dtype)
    fb = x[0].numel() * x.element_size()
    check(lib().t2v_gather_frames(ptr(x), ptr(y), B, T, fb, sn, st, bt, ptr(bt_dev), 0, stream()),
          "t2v_gather_frames")
    return y


def scatter_frames(dy, B, T, bt, sn=2, st=2):
    """adjoint of gather_frames: zero-filled (B*T, ...) with the gathered frames written back."""
    require_cuda(dy)
    assert dy.is_contiguous()
    bt, bt_dev = _bt_args(bt, T, st)
    dx = torch.empty((B * T,) + tuple(dy.shape[1:]), device=dy.device, dtype=dy.dtype)
    fb = dx[0].numel() * dx.element_size()
    check(lib().t2v_gather_frames(ptr(dy), ptr(dx), B, T, fb, sn, st, bt, ptr(bt_dev), 1, stream()),
          "t2v_gather_frames")
    return dx


def pyramid_level(x, Ho, Wo, sn=1, st=1, bt=0):
    """fp32 (B,C,T,H,W) -> (ceil(B/sn), C, ceil((T-bt)/st), Ho, Wo): batch/frame subsampling composed
    with nearest resize (src = floor(dst*in/out)); either part can be the identity."""
    require_cuda(x)
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 5
    B, C, T, H, W = x.shape
    bt, bt_dev = _bt_args(bt, T, st)
    Bo = (B + sn - 1) // sn
    To = (T - bt + st - 1) // st if T > bt else 0
    y = torch.empty((Bo, C, To, Ho, Wo), device=x.device, dtype=F32)
    check(lib().t2v_pyramid_level(ptr(x), ptr(y), _i32(B, C, T, H, W), Ho, Wo, sn, st, bt, ptr(bt_dev), stream()),
          "t2v_pyramid_level")
    return y


# ------------------------------------------------------------------------------------- LSTM cell / Adam
def lstm_cell_fwd(gates, c_prev, want_h32=False):
    """gates fp32 (..., 4H) [i|f|g|o], c_prev fp32 (..., H) or None -> (c fp32, h bf16, h32|None)."""
    require_cuda(gates, c_prev)
    assert gates.dtype == F32 and gates.is_contiguous()
    Hd = gates.shape[-1] // 4
    shp = tuple(gates.shape[:-1]) + (Hd,)
    c = torch.empty(shp, device=gates.device, dtype=F32)
    h = torch.empty(shp, device=gates.device, dtype=STORE)
    h32 = torch.empty(shp, device=gates.device, dtype=F32) if want_h32 else None
    check(_lib.typed("t2v_lstm_cell_fwd", h)(ptr(gates), ptr(c_prev), ptr(c), ptr(h), ptr(h32), c.numel() // Hd, Hd, stream()),
          "t2v_lstm_cell_fwd")
    return c, h, h32


def lstm_cell_bwd(gates, c_prev, c, dh, dc_next):
    """-> (dgates bf16 (...,4H), dc_prev fp32 (...,H)); dh / dc_next fp32 or None."""
    require_cuda(gates, c)
    Hd = c.shape[-1]
    dgates = torch.empty(gates.shape, device=gates.device, dtype=STORE)
    dc_prev = torch.empty_like(c)
    check(_lib.typed("t2v_lstm_cell_bwd", dgates)(ptr(gates), ptr(c_prev), ptr(c), ptr(dh), ptr(dc_next), ptr(dgates), ptr(dc_prev),
                                  c.numel() // Hd, Hd, stream()), "t2v_lstm_cell_bwd")
    return dgates, dc_prev


def adam_step(params, grads, ms, vs, lr, beta1, beta2, eps, step, grad_scale=1.0, dyn=None):
    """In-place multi-tensor Adam on fp32 tensors that share memory layout pairwise."""
    n = len(params)
    if n == 0:
        return
    require_cuda(*params)
    arr = ctypes.c_void_p * n
    sizes = (ctypes.c_int64 * n)(*[p.numel() for p in params])
    for p, g, m, v in zip(params, grads, ms, vs):
        assert p.dtype == F32 and g.dtype == F32 and p.stride() == g.stride() == m.stride() == v.stride(), \
            (p.shape, p.stride(), g.stride())
    check(lib().t2v_adam_step(n, arr(*[p.data_ptr() for p in params]), arr(*[g.data_ptr() for g in grads]),
                              arr(*[m.data_ptr() for m in ms]), arr(*[v.data_ptr() for v in vs]), sizes, lr, beta1,
                              beta2, eps, step, grad_scale, ptr(dyn), stream()), "t2v_adam_step")


def multi_copy(srcs, dsts):
    """dst[i].memory <- src[i].memory for lists of equally laid-out fp32 tensors (gradient buckets).  Either side may
    be PINNED host memory (read / written by the SMs over UVA): small per-step host values and the loss read-back
    travel this way, because a cudaMemcpyAsync on the compute stream queues behind the prefetcher's H2D pieces on
    the copy engine."""
    n = len(srcs)
    if n == 0:
        return
    for t in list(srcs) + list(dsts):
        if not (t.is_cuda or t.is_pinned()):
            raise _lib.T2VError("multi_copy needs CUDA or pinned host tensors (got %s)" % t.device)
    arr = ctypes.c_void_p * n
    sizes = (ctypes.c_int64 * n)(*[s.numel() for s in srcs])
    for s, d in zip(srcs, dsts):
        assert s.dtype == F32 and d.dtype == F32 and s.numel() == d.numel()
    check(lib().t2v_multi_copy(n, arr(*[s.data_ptr() for s in srcs]), arr(*[d.data_ptr() for d in dsts]), sizes,
                               stream()), "t2v_multi_copy")


# ------------------------------------------------------------------------------------- non-local block primitives
def maxpool122_fwd(x):
    """fp32 (M, H, W, c) -> (pooled fp32 (M, H/2, W/2, c), idx uint8): max-pool (1,2,2) with recorded arg-max"""
    require_cuda(x)
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 4
    M, H, W, c = x.shape
    y = torch.empty((M, H // 2, W // 2, c), device=x.device, dtype=F32)
    idx = torch.empty((M, H // 2, W // 2, c), device=x.device, dtype=torch.uint8)
    check(lib().t2v_maxpool122_fwd(ptr(x), ptr(y), ptr(idx), M, H, W, c, stream()), "t2v_maxpool122_fwd")
    return y, idx


def pool122_gather(x, idx):
    require_cuda(x, idx)
    assert x.dtype == F32 and x.is_contiguous() and idx.dtype == torch.uint8 and idx.is_contiguous()
    M, H, W, c = x.shape
    y = torch.empty(tuple(idx.shape), device=x.device, dtype=F32)
    check(lib().t2v_pool122_gather(ptr(x), ptr(idx), ptr(y), M, H, W, c, stream()), "t2v_pool122_gather")
    return y


def pool122_scatter(dy, idx):
    require_cuda(dy, idx)
    assert dy.dtype == F32 and dy.is_contiguous() and idx.dtype == torch.uint8 and tuple(idx.shape) == tuple(dy.shape)
    M, Hp, Wp, c = dy.shape
    dx = torch.empty((M, 2 * Hp, 2 * Wp, c), device=dy.device, dtype=F32)
    check(lib().t2v_pool122_scatter(ptr(dy), ptr(idx), ptr(dx), M, 2 * Hp, 2 * Wp, c, stream()), "t2v_pool122_scatter")
    return dx


def bmm(a, b, ta=False, tb=False):
    """fp32 batched C = op(A) op(B): a (n, M, K) [ta: (n, K, M)], b (n, K, N) [tb: (n, N, K)] -> (n, M, N)"""
    require_cuda(a, b)
    assert a.dtype == F32 and b.dtype == F32 and a.is_contiguous() and b.is_contiguous() and a.dim() == 3
    n = a.shape[0]
    M, K = (a.shape[2], a.shape[1]) if ta else (a.shape[1], a.shape[2])
    N = b.shape[1] if tb else b.shape[2]
    assert b.shape[0] == n and (b.shape[2] if tb else b.shape[1]) == K, (a.shape, b.shape, ta, tb)
    c = torch.empty((n, M, N), device=a.device, dtype=F32)
    for i0 in range(0, n, 65535):
        i1 = min(n, i0 + 65535)
        check(lib().t2v_bmm_f32(ptr(a[i0:i1]), ptr(b[i0:i1]), ptr(c[i0:i1]), i1 - i0, M, N, K, int(ta), int(tb),
                                stream()), "t2v_bmm_f32")
    return c


def softmax_fwd(s):
    require_cuda(s)
    assert s.dtype == F32 and s.is_contiguous()
    out = torch.empty_like(s)
    check(lib().t2v_softmax_fwd(ptr(s), ptr(out), s.numel() // s.shape[-1], s.shape[-1], stream()), "t2v_softmax_fwd")
    return out


def softmax_bwd(beta, dbeta):
    require_cuda(beta, dbeta)
    assert beta.dtype == F32 and dbeta.dtype == F32 and beta.is_contiguous() and dbeta.is_contiguous()
    out = torch.empty_like(beta)
    check(lib().t2v_softmax_bwd(ptr(beta), ptr(dbeta), ptr(out), beta.numel() // beta.shape[-1], beta.shape[-1],
                                stream()), "t2v_softmax_bwd")
    return out


def softmax_bwd_bwd(beta, dbeta, u):
    """derivative of softmax_bwd(beta, dbeta) against the cotangent u -> (g_beta, g_dbeta)"""
    require_cuda(beta, dbeta, u)
    assert all(t.dtype == F32 and t.is_contiguous() for t in (beta, dbeta, u))
    gb, gd = torch.empty_like(beta), torch.empty_like(beta)
    check(lib().t2v_softmax_bwd_bwd(ptr(beta), ptr(dbeta), ptr(u), ptr(gb), ptr(gd), beta.numel() // beta.shape[-1],
                                    beta.shape[-1], stream()), "t2v_softmax_bwd_bwd")
    return gb, gd


# ------------------------------------------------------------------------------------- heads / losses / penalty
def head_fwd(feat, cond, w, bias):
    """[feat | cond] (B, F [+E]) fp32 . w (F [+E],) + bias -> (B,)"""
    require_cuda(feat, cond, w, bias)
    B, F_ = feat.shape
    E = 0 if cond is None else cond.shape[1]
    assert feat.dtype == F32 and feat.is_contiguous() and w.dtype == F32 and w.is_contiguous() and w.numel() == F_ + E
    assert cond is None or (cond.dtype == F32 and cond.is_contiguous() and cond.shape[0] == B)
    out = torch.empty((B,), device=feat.device, dtype=F32)
    check(lib().t2v_head_fwd(ptr(feat), ptr(cond), ptr(w), ptr(bias), ptr(out), B, F_, E, stream()), "t2v_head_fwd")
    return out


def head_bwd_data(dpred, w, F_, E):
    """-> (dfeat (B,F), dcond (B,E) or None) = dpred (x) w"""
    require_cuda(dpred, w)
    assert dpred.dtype == F32 and dpred.is_contiguous() and w.dtype == F32 and w.is_contiguous()
    B = dpred.numel()
    dfeat = torch.empty((B, F_), device=dpred.device, dtype=F32)
    dcond = torch.empty((B, E), device=dpred.device, dtype=F32) if E else None
    check(lib().t2v_head_bwd_data(ptr(dpred), ptr(w), ptr(dfeat), ptr(dcond), B, F_, E, stream()), "t2v_head_bwd_data")
    return dfeat, dcond


def head_bwd_weight(dpred, feat, cond, want_bias=True):
    """-> (dw (F [+E],), db (1,) or None) = sum_b dpred[b] [feat | cond][b]"""
    require_cuda(dpred, feat, cond)
    B, F_ = feat.shape
    E = 0 if cond is None else cond.shape[1]
    assert dpred.dtype == F32 and dpred.is_contiguous() and dpred.numel() == B and feat.dtype == F32
    assert feat.is_contiguous() and (cond is None or (cond.dtype == F32 and cond.is_contiguous()))
    dw = torch.empty((F_ + E,), device=feat.device, dtype=F32)
    db = torch.empty((1,), device=feat.device, dtype=F32) if want_bias else None
    check(lib().t2v_head_bwd_weight(ptr(dpred), ptr(feat), ptr(cond), ptr(dw), ptr(db), B, F_, E, 0, stream()),
          "t2v_head_bwd_weight")
    return dw, db


def _loss_arrays(a_list, b_list, weights):
    n = len(a_list)
    arr = ctypes.c_void_p * n
    for a, b in zip(a_list, b_list):
        assert a.dtype == F32 and b.dtype == F32 and a.is_contiguous() and b.is_contiguous() and a.numel() == b.numel()
    ns = (ctypes.c_int32 * n)(*[a.numel() for a in a_list])
    ws = (ctypes.c_float * n)(*[float(w) for w in weights])
    return n, arr, ns, ws


def rel_loss_fwd(a_list, b_list, weights, mode):
    """0-d fp32 = sum_e weights[e] * mean_j f(b_e[j] - a_e[j]); mode 0 softplus (RSGAN), 1 identity (WGAN)"""
    require_cuda(*a_list, *b_list)
    n, arr, ns, ws = _loss_arrays(a_list, b_list, weights)
    out = torch.empty((), device=a_list[0].device, dtype=F32)
    check(lib().t2v_rel_loss_fwd(n, arr(*[t.data_ptr() for t in a_list]), arr(*[t.data_ptr() for t in b_list]), ns, ws,
                                 int(mode), ptr(out), stream()), "t2v_rel_loss_fwd")
    return out


def rel_loss_bwd(a_list, b_list, da_list, db_list, weights, mode, gout):
    """da_e / db_e (None to skip; pre-zeroed; entries may share buffers) += d(loss)/d(a_e), d(b_e) * gout"""
    require_cuda(*a_list, *b_list, gout)
    n, arr, ns, ws = _loss_arrays(a_list, b_list, weights)
    assert gout.dtype == F32 and gout.numel() == 1
    pa = arr(*[None if t is None else t.data_ptr() for t in da_list])
    pb = arr(*[None if t is None else t.data_ptr() for t in db_list])
    check(lib().t2v_rel_loss_bwd(n, arr(*[t.data_ptr() for t in a_list]), arr(*[t.data_ptr() for t in b_list]), pa, pb,
                                 ns, ws, int(mode), ptr(gout), stream()), "t2v_rel_loss_bwd")


def lerp_rows(real, fake, alpha):
    """x_hat[b] = alpha[b] * real[b] + (1 - alpha[b]) * fake[b]; real / fake fp32 (B, ...), alpha fp32 (B,)"""
    require_cuda(real, fake, alpha)
    assert real.dtype == F32 and fake.dtype == F32 and alpha.dtype == F32 and real.shape == fake.shape
    assert real.is_contiguous() and fake.is_contiguous() and alpha.is_contiguous() and alpha.numel() == real.shape[0]
    out = torch.empty_like(real)
    B = real.shape[0]
    check(lib().t2v_lerp_rows(ptr(real), ptr(fake), ptr(alpha), ptr(out), B, real.numel() // max(B, 1), stream()),
          "t2v_lerp_rows")
    return out


def gp_norm_fwd(g):
    """g fp32 (B, ...) -> (0-d mean_b (||g_b|| - 1)^2, norms fp32 (B,)), reduced in a fixed order.  One block per
    8192 elements of a row (at most 1024 per row): enough blocks to fill the GPU at B = 1."""
    require_cuda(g)
    assert g.dtype == F32 and g.is_contiguous()
    B = g.shape[0]
    S = g.numel() // max(B, 1)
    splits = max(1, min(1024, -(-S // 8192)))
    partials = torch.empty(B * splits, device=g.device, dtype=F32)
    norms = torch.empty(B, device=g.device, dtype=F32)
    out = torch.empty((), device=g.device, dtype=F32)
    check(lib().t2v_gp_norm_fwd(ptr(g), ptr(partials), ptr(norms), ptr(out), B, S, splits, stream()),
          "t2v_gp_norm_fwd")
    return out, norms


def gp_norm_bwd(g, norms, gout):
    """d/dg of gp_norm_fwd's penalty times gout (0-d fp32 on the device)"""
    require_cuda(g, norms, gout)
    assert g.dtype == F32 and g.is_contiguous() and norms.dtype == F32 and gout.dtype == F32 and gout.numel() == 1
    B = g.shape[0]
    dg = torch.empty_like(g)
    check(lib().t2v_gp_norm_bwd(ptr(g), ptr(norms), ptr(gout), ptr(dg), B, g.numel() // max(B, 1), stream()),
          "t2v_gp_norm_bwd")
    return dg


# ------------------------------------------------------------------------------------- caption LSTM
def lstm_pack_whh(whh):
    """fp32 (ndir, 4H, H) -> (ndir, H, 4H)"""
    require_cuda(whh)
    assert whh.dtype == F32 and whh.is_contiguous() and whh.dim() == 3
    ndir, H4, H = whh.shape
    out = torch.empty((ndir, H, H4), device=whh.device, dtype=F32)
    check(lib().t2v_lstm_pack_whh(ptr(whh), ptr(out), ndir, H, stream()), "t2v_lstm_pack_whh")
    return out


def lstm_seq_fwd(gx, whhT, lengths, h0, c0, save=True):
    """gx fp32 (B, L, ndir*4H); whhT (ndir, H, 4H); lengths int32 (B,) on the device; h0 / c0 fp32 (ndir, B, H) or None
    -> out (B, L, ndir*H) storage, hprev (same) | None, gates fp32 | None, cells fp32 | None, hn, cn (ndir, B, H)"""
    require_cuda(gx, whhT, lengths, h0, c0)
    B, L = gx.shape[0], gx.shape[1]
    ndir, H = whhT.shape[0], whhT.shape[1]
    assert gx.dtype == F32 and gx.is_contiguous() and gx.shape[2] == ndir * 4 * H and lengths.dtype == torch.int32
    dev = gx.device
    out = torch.empty((B, L, ndir * H), device=dev, dtype=STORE)
    hprev = torch.empty_like(out) if save else None
    gates = torch.empty((B, L, ndir * 4 * H), device=dev, dtype=F32) if save else None
    cells = torch.empty((B, L, ndir * H), device=dev, dtype=F32) if save else None
    hn = torch.empty((ndir, B, H), device=dev, dtype=F32)
    cn = torch.empty((ndir, B, H), device=dev, dtype=F32)
    check(_lib.typed("t2v_lstm_seq_fwd", out)(ptr(gx), ptr(whhT), ptr(lengths), ptr(h0), ptr(c0), ptr(out), ptr(hprev),
                                              ptr(gates), ptr(cells), ptr(hn), ptr(cn), B, L, H, ndir, stream()),
          "t2v_lstm_seq_fwd")
    return out, hprev, gates, cells, hn, cn


def lstm_seq_bwd(whh, lengths, c0, gates, cells, dout, dhn, dcn):
    """-> dgates (B, L, ndir*4H) storage, dh0, dc0 fp32 (ndir, B, H)"""
    require_cuda(whh, lengths, gates, cells, dout, dhn, dcn)
    ndir, H = whh.shape[0], whh.shape[2]
    B, L = gates.shape[0], gates.shape[1]
    dev = gates.device
    assert dout is None or (dout.is_contiguous() and dout.dtype == STORE)
    dgates = torch.empty((B, L, ndir * 4 * H), device=dev, dtype=STORE)
    dh0 = torch.empty((ndir, B, H), device=dev, dtype=F32)
    dc0 = torch.empty((ndir, B, H), device=dev, dtype=F32)
    check(_lib.typed("t2v_lstm_seq_bwd", dgates)(ptr(whh), ptr(lengths), ptr(c0), ptr(gates), ptr(cells), ptr(dout),
                                                 ptr(dhn), ptr(dcn), ptr(dgates), ptr(dh0), ptr(dc0), B, L, H, ndir,
                                                 stream()), "t2v_lstm_seq_bwd")
    return dgates, dh0, dc0


def embedding_fwd(tokens, weight):
    """int64 (B, L), fp32 (V, E) -> storage (B, L, E)"""
    require_cuda(tokens, weight)
    assert tokens.dtype == torch.int64 and tokens.is_contiguous() and weight.dtype == F32 and weight.is_contiguous()
    E = weight.shape[1]
    out = torch.empty(tuple(tokens.shape) + (E,), device=weight.device, dtype=STORE)
    check(_lib.typed("t2v_embedding_fwd", out)(ptr(tokens), ptr(weight), ptr(out), tokens.numel(), E, stream()),
          "t2v_embedding_fwd")
    return out


def embedding_bwd(tokens, dout, V):
    require_cuda(tokens, dout)
    _act(dout)
    E = dout.shape[-1]
    dw = torch.empty((V, E), device=dout.device, dtype=F32)
    check(_lib.typed("t2v_embedding_bwd", dout)(ptr(tokens), ptr(dout), ptr(dw), tokens.numel(), E, V, stream()),
          "t2v_embedding_bwd")
    return dw


# ------------------------------------------------------------------------------------- on-device input pipeline (8 f1)
def u8_normalize(src, out=None):
    """uint8 frames -> fp32 (x / 255 - 0.5) / 0.5: transforms.ToTensor() + Normalize(0.5, 0.5), data/__init__.py:362-364"""
    require_cuda(src)
    assert src.dtype == torch.uint8 and src.is_contiguous()
    if out is None:
        out = torch.empty(src.shape, device=src.device, dtype=F32)
    assert out.dtype == F32 and out.is_contiguous() and out.numel() == src.numel()
    check(lib().t2v_u8_normalize(ptr(src), ptr(out), src.numel(), stream()), "t2v_u8_normalize")
    return out


def moving_digits(bank, digit, pos, T, H, W, out_f32=False, layout=0):
    """bank uint8 (n, oh, ow), digit int32 (B,), pos int32 (B, T, 2) = (x, y) -> clips (B,T,3,H,W) [layout 0] or
    (B,3,T,H,W) [layout 1], uint8 as stored or fp32 normalised (data/synthetic/generate.py:18-47)"""
    require_cuda(bank, digit, pos)
    B = digit.numel()
    assert bank.dtype == torch.uint8 and bank.is_contiguous() and bank.dim() == 3
    assert digit.dtype == torch.int32 and pos.dtype == torch.int32 and tuple(pos.shape) == (B, T, 2) and pos.is_contiguous()
    shape = (B, T, 3, H, W) if layout == 0 else (B, 3, T, H, W)
    out = torch.empty(shape, device=bank.device, dtype=F32 if out_f32 else torch.uint8)
    check(lib().t2v_moving_digits(ptr(bank), ptr(digit), ptr(pos), ptr(out), B, T, H, W, bank.shape[1], bank.shape[2],
                                  1 if out_f32 else 0, layout, stream()), "t2v_moving_digits")
    return out


def grammar_tokens(cls, move, table):
    """cls, move int32 (B,), table int64 (23,) -> tokens int64 (B, 8) of "digit {cls} is {a} and {b}." """
    require_cuda(cls, move, table)
    B = cls.numel()
    assert cls.dtype == torch.int32 and move.dtype == torch.int32 and table.dtype == torch.int64 and table.numel() == 23
    tokens = torch.empty((B, 8), device=cls.device, dtype=torch.int64)
    check(lib().t2v_grammar_tokens(ptr(cls), ptr(move), ptr(table), ptr(tokens), B, stream()), "t2v_grammar_tokens")
    return tokens
