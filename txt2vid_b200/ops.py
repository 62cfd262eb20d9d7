"""Differentiable ops of the TGANv2 training step on top of the sm_100a kernels.

Every Function's backward is written in terms of other Functions of this file, so the graph is
closed under differentiation where the reference needs it: the gradient penalty
(txt2vid/gan/losses.py:135-209) differentiates d(D)/d(x_hat) a second time, which here means
conv_fprop <-> conv_dgrad <-> conv_wgrad, ReLU masks, avg-pool/broadcast adjoint pairs.

Activations are "CL" tensors: contiguous (N, D, H, W, C) bf16 (2-D maps: D = 1).  Parameters stay
fp32 `nn.Parameter`s with the reference's logical shapes; conv weights are re-homed once into
channels-last memory ([Cout][taps][Cin]) so that packing is a cast and the weight gradient the
kernels write is the parameter gradient's memory.
"""
import weakref

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import kernels as K   # tests replace this module attribute with tests/cpu_kernels.py

BF16 = torch.bfloat16
F32 = torch.float32

_EPOCH = [0]


def bump_weight_epoch():
    """Called after an optimiser writes parameters through raw pointers (no autograd version bump)."""
    _EPOCH[0] += 1


def round16(c):
    return (c + 15) // 16 * 16


# ------------------------------------------------------------------------------------- precision mode
# "bf16": the product (bf16 activation storage, bf16 tensor-core operands, fp32 accumulation / statistics / master
#         weights) -- BASELINE north_star's 2e-2 bar;
# "fp32": fp32 activation storage on the same kernels instantiated for float, every convolution as exact fp32 FMAs on
#         the CUDA-core kernels of gconv.cu (fp32 accumulation flushed once per tap) -- the 1e-3 bar.  The bf16-only
#         fusions (direct RGB stem, stride-(2,1,1) stem conv, fused skip conv, fused generator attention) fall back to
#         their unfused formulations on the generic kernels.
PRECISION = ["bf16"]


def set_precision(mode):
    assert mode in ("bf16", "fp32"), mode
    K.set_store_dtype(F32 if mode == "fp32" else BF16)
    PRECISION[0] = mode
    PACKS.clear()


def fp32_mode():
    return PRECISION[0] == "fp32"


# ------------------------------------------------------------------------------------- weight handling
def kernel_of(weight):
    """(kd,kh,kw) of a Linear / Conv2d / Conv3d weight."""
    if weight.dim() == 2:
        return (1, 1, 1)
    if weight.dim() == 3:
        return (1, 1, weight.shape[2])
    if weight.dim() == 4:
        return (1, weight.shape[2], weight.shape[3])
    return tuple(weight.shape[2:])


def w3_view(weight):
    """fp32 (Cout, taps, Cin) VIEW of a parameter, re-homing it to channels-last memory if needed."""
    if weight.dim() == 2:
        assert weight.is_contiguous()
        return weight.view(weight.shape[0], 1, weight.shape[1])
    perm = _CL_PERM[weight.dim()]
    if not weight.permute(*perm).is_contiguous():
        with torch.no_grad():
            weight.data = _to_cl_memory(weight.data)
    wp = weight.permute(*perm)
    return wp.reshape(weight.shape[0], -1, weight.shape[1])


_CL_PERM = {3: (0, 2, 1), 4: (0, 2, 3, 1), 5: (0, 2, 3, 4, 1)}
_CL_INV = {3: (0, 2, 1), 4: (0, 3, 1, 2), 5: (0, 4, 1, 2, 3)}


def _to_cl_memory(t):
    return t.permute(*_CL_PERM[t.dim()]).contiguous().permute(*_CL_INV[t.dim()])


def grad_like_weight(dw3, weight):
    """(Cout,taps,Cin) fp32 -> tensor with the parameter's logical shape sharing dw3's memory."""
    if weight.dim() == 2:
        return dw3.view(weight.shape)
    Cout, Cin = weight.shape[0], weight.shape[1]
    if weight.dim() == 3:
        return dw3.view(Cout, weight.shape[2], Cin).permute(0, 2, 1)
    if weight.dim() == 4:
        return dw3.view(Cout, weight.shape[2], weight.shape[3], Cin).permute(0, 3, 1, 2)
    return dw3.view(Cout, weight.shape[2], weight.shape[3], weight.shape[4], Cin).permute(0, 4, 1, 2, 3)


class _PackCache(object):
    """bf16 operand packs per parameter, rebuilt when the parameter changes.  Entries are keyed by the OWNING tensor
    (the parameter itself, or the parameter a differentiable view such as stem_weight_2d was taken from) plus the
    view's geometry, and carry a weak reference to the owner: a view is a new Python object on every call (no dead
    entry per iteration), and a new model whose parameters land on a freed model's addresses never sees its packs."""

    def __init__(self):
        self.store = {}

    def _key(self, w):
        return (w._version, w.data_ptr(), _EPOCH[0])

    @staticmethod
    def _owner(w):
        base = getattr(w, "_base", None)
        return base if base is not None else w

    def _slot_of(self, w):
        return (id(self._owner(w)), tuple(w.shape), tuple(w.stride()))

    def _lookup(self, ident, w):
        ent = self.store.get(ident)
        if ent is None or ent[0] != self._key(w) or ent[2]() is not self._owner(w):
            if len(self.store) > 4096:               # forget the packs of tensors that no longer exist
                for k in [k for k, e in self.store.items() if e[2]() is None]:
                    del self.store[k]
            ent = (self._key(w), {}, weakref.ref(self._owner(w)))
            self.store[ident] = ent
        return ent

    def get(self, w, kind, CoutP, CinP):
        ident = self._slot_of(w)
        ent = self._lookup(ident, w)
        slot = (kind, CoutP, CinP)
        if slot not in ent[1]:
            with torch.no_grad():
                w3 = w3_view(w).detach()       # may re-home the parameter's memory (channels-last)
            if kind == "fprop":
                pack = K.pack_weight(w3, CoutP, CinP)
            elif kind == "gconv":                    # general (strided / transposed) convolution kernels
                if (CoutP, CinP) != (w3.shape[0], w3.shape[2]):
                    wpad = w3.new_zeros((CoutP, w3.shape[1], CinP))
                    wpad[:w3.shape[0], :, :w3.shape[2]] = w3
                    w3 = wpad
                pack = K.gconv_pack(w3)
            else:
                pack = K.pack_dgrad_weight(w3, CoutP, CinP)
            if self._slot_of(w) != ident or ent[0] != self._key(w):     # w3_view re-homed the parameter
                self.store.pop(ident, None)
                ident = self._slot_of(w)
                ent = (self._key(w), {}, weakref.ref(self._owner(w)))
                self.store[ident] = ent
            ent[1][slot] = pack
        return ent[1][slot]

    def clear(self):
        self.store.clear()


PACKS = _PackCache()


# ------------------------------------------------------------------------------------- gradient sinks
# The discriminator's weights are shared by the four pyramid levels and by the loss and penalty graphs, so one
# backward pass produces ~11 partial weight gradients per tensor; summed by autograd that is ~440 fp32 add kernels per
# iteration.  Instead every unpadded conv weight owns one persistent fp32 buffer [Cout][taps][Cin] (= p.grad's memory,
# zeroed by zero_grads) and the weight-gradient kernels accumulate into it directly (fp32 red.add, as they already
# do between their own position splits).  Second-order graphs (create_graph=True) keep the functional path.


def _sinkable(p):
    # only weights that ConvF / ConvSd2F have consumed (marked at their first forward) and that need no channel padding
    return getattr(p, "_t2v_conv", False) and p.dim() >= 2 and p.shape[0] % 16 == 0 and p.shape[1] % 16 == 0


def mark_conv_weights(module):
    """Flag the Conv2d / Conv3d / Linear weights of a product module as consumed by the conv engine (ConvLSTM cells
    excluded: their eight kernels are stacked into one gate GEMM and receive their gradient through torch.cat)."""
    skip = set()
    for name, m in module.named_modules():
        if type(m).__name__ == "ConvLSTMCell":
            skip.update(id(c) for c in m.modules())
    for m in module.modules():
        if id(m) not in skip and isinstance(m, (torch.nn.Conv2d, torch.nn.Conv3d, torch.nn.Linear)):
            m.weight._t2v_conv = True
            if m.bias is not None and isinstance(m, (torch.nn.Conv2d, torch.nn.Conv3d)):
                m.bias._t2v_bias = True
    module._t2v_marked = True


def zero_grads(module):
    """module.zero_grad() (gan/cond_gan.py:91-94,157-161): gradients of sink-owning weights become zeroed persistent
    buffers, all others None (filled by autograd)."""
    if not getattr(module, "_t2v_marked", False):
        mark_conv_weights(module)
    bufs = []
    for p in module.parameters():
        if p.requires_grad and getattr(p, "_t2v_bias", False) and p.dim() == 1 and p.numel() % 16 == 0:
            # conv biases: the column-sum kernel adds into the gradient buffer (t2v_sum_rows_acc)
            if p.grad is None or not getattr(p, "_t2v_bias_sink", False):
                p.grad = torch.empty_like(p)
                p._t2v_bias_sink = True
            bufs.append(p.grad)
            continue
        if not (p.requires_grad and _sinkable(p)):
            p.grad = None
            continue
        w3 = w3_view(p)                                  # re-homes the parameter to channels-last memory if needed
        sink = getattr(p, "_t2v_sink", None)
        if sink is None or sink.shape != w3.shape or sink.device != p.device:
            sink = torch.empty(w3.shape, device=p.device, dtype=F32)
            p._t2v_sink = sink
        bufs.append(sink)
        if p.grad is None or p.grad.data_ptr() != sink.data_ptr():
            p.grad = grad_like_weight(sink, p)
    if bufs:
        torch._foreach_zero_(bufs)


def _wgrad(dy, x, weight, sd2=False):
    """Weight gradient of a convolution: into the parameter's sink when this is a first-order backward pass."""
    sink = getattr(weight, "_t2v_sink", None)
    if (sink is not None and not torch.is_grad_enabled() and weight.grad is not None
            and weight.grad.data_ptr() == sink.data_ptr() and dy.shape[-1] == weight.shape[0]
            and x.shape[-1] == weight.shape[1]):
        if sd2:
            K.conv_wgrad_sd2(dy, x, out=sink, accumulate=True)
        else:
            K.conv_wgrad(dy, x, kernel_of(weight), out=sink, accumulate=True)
        return None
    return (ConvSd2WgradF if sd2 else ConvWgradF).apply(dy, x, weight)


def _bias_grad(dy, bias, Cout):
    """Bias gradient of a convolution (column sums of dy): into the bias' gradient buffer on first-order passes."""
    if (bias is not None and getattr(bias, "_t2v_bias_sink", False) and bias.grad is not None
            and not torch.is_grad_enabled() and dy.shape[-1] == Cout == bias.numel()):
        K.sum_rows(dy, out=bias.grad)
        return None
    return SumRowsF.apply(dy)[:Cout]


def _prof_real(weight, CinP, CoutP):
    """roofline bookkeeping: the next conv launch multiplies CinP x CoutP channel pairs of which weight.shape[:2] are
    real (zero padding of RGB / attention / render channels is not counted as useful work)"""
    if K is not None and getattr(K, "PROFILING", [False])[0]:
        K.prof_real_fraction(weight.shape[0] * weight.shape[1], CinP * CoutP)


def _pad_bias(bias, CoutP):
    if bias is None:
        return None
    b = bias.detach()
    if b.numel() == CoutP:
        return b
    out = torch.zeros((CoutP,), device=b.device, dtype=F32)
    out[:b.numel()] = b
    return out


# ------------------------------------------------------------------------------------- convolution


class ConvF(Function):
    """y = [relu](conv(x, w) + b [+ residual]);  x CL (.., CinP) -> y CL (.., CoutP).

    ReLU-backward fusion (the discriminator's ReLU -> conv chains, layers.py:229-235, resnet3d.py:12-15):
      x_relu      x is the output of a ReLU whose backward THIS op applies: dx = dgrad(dy) * (x > 0), in the
                  data-gradient kernel's epilogue on first-order passes (a separate mask op under create_graph);
      relu_later  the consumer of y applies this op's own ReLU mask (it was built with x_relu): backward does not
                  mask dy again.  Masks are idempotent, so a y with several consumers needs all of them to mask."""

    @staticmethod
    def forward(ctx, x, weight, bias, residual, relu, x_relu=False, relu_later=False):
        k = kernel_of(weight)
        Cout, Cin = weight.shape[0], weight.shape[1]
        CinP, CoutP = x.shape[-1], round16(Cout)
        assert CinP >= Cin and CinP % 16 == 0, (CinP, Cin)
        wp = PACKS.get(weight, "fprop", CoutP, CinP)
        weight._t2v_conv = True
        _prof_real(weight, CinP, CoutP)
        y = K.conv_fprop(x, wp, _pad_bias(bias, CoutP), residual, k, relu)
        ctx.relu = relu and not relu_later
        ctx.x_relu = x_relu
        ctx.has_bias = bias is not None
        ctx.bias_ref = bias
        ctx.has_res = residual is not None
        ctx.save_for_backward(x, weight, y if ctx.relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, y = ctx.saved_tensors
        dy = dy.contiguous()
        if ctx.relu:
            dy = ReluBwdF.apply(dy, y)
        dx = dw = db = dres = None
        if ctx.needs_input_grad[0]:
            if not ctx.x_relu:
                dx = ConvDgradF.apply(dy, weight, x.shape[-1])
            elif torch.is_grad_enabled() or x.shape[-1] % 16 or dy.shape[-1] % 16:
                dx = ReluBwdF.apply(ConvDgradF.apply(dy, weight, x.shape[-1]), x)
            else:
                _prof_real(weight, x.shape[-1], dy.shape[-1])
                dx = K.conv_dgrad(dy, PACKS.get(weight, "dgrad", dy.shape[-1], x.shape[-1]), kernel_of(weight),
                                  relu_ref=x)
        if ctx.needs_input_grad[1]:
            dw = _wgrad(dy, x, weight)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = _bias_grad(dy, ctx.bias_ref, weight.shape[0])
        if ctx.has_res and ctx.needs_input_grad[3]:
            dres = dy
        return dx, dw, db, dres, None, None, None


class ConvSkipF(Function):
    """y = conv(h, w) + b + conv1x1x1(x, ws) + bs: the last convolution of a DownBlock with the block's identity_map
    convolution (models/layers.py:224-243) fused in as extra K of the same implicit GEMM -- the skip tensor is never
    written or re-read, and the two bias gradients (the same column sum of dy) are computed once.  h_relu as in ConvF's
    x_relu.  The backward is composed of the differentiable conv Functions, so second-order graphs work unchanged."""

    @staticmethod
    def forward(ctx, h, x, weight, bias, wskip, bskip, h_relu):
        k = kernel_of(weight)
        Cout = weight.shape[0]
        wp = PACKS.get(weight, "fprop", Cout, h.shape[-1])
        ws = PACKS.get(wskip, "fprop", Cout, x.shape[-1])
        weight._t2v_conv = wskip._t2v_conv = True
        b = None
        if bias is not None or bskip is not None:
            b = (bias.detach() if bias is not None else 0) + (bskip.detach() if bskip is not None else 0)
        ctx.h_relu = h_relu
        ctx.has_b = (bias is not None, bskip is not None)
        ctx.bias_refs = (bias, bskip)
        ctx.save_for_backward(h, x, weight, wskip)
        return K.conv_fprop_skip(h, wp, b, x, ws, k)

    @staticmethod
    def backward(ctx, dy):
        h, x, weight, wskip = ctx.saved_tensors
        dy = dy.contiguous()
        dh = dx = dw = db = dws = dbs = None
        if ctx.needs_input_grad[0]:
            if not ctx.h_relu:
                dh = ConvDgradF.apply(dy, weight, h.shape[-1])
            elif torch.is_grad_enabled():
                dh = ReluBwdF.apply(ConvDgradF.apply(dy, weight, h.shape[-1]), h)
            else:
                dh = K.conv_dgrad(dy, PACKS.get(weight, "dgrad", dy.shape[-1], h.shape[-1]), kernel_of(weight),
                                  relu_ref=h)
        if ctx.needs_input_grad[1]:
            dx = ConvDgradF.apply(dy, wskip, x.shape[-1])
        if ctx.needs_input_grad[2]:
            dw = _wgrad(dy, h, weight)
        if ctx.needs_input_grad[4]:
            dws = _wgrad(dy, x, wskip)
        want = (ctx.has_b[0] and ctx.needs_input_grad[3], ctx.has_b[1] and ctx.needs_input_grad[5])
        if want[0] or want[1]:
            sinks = [b is not None and getattr(b, "_t2v_bias_sink", False) and b.grad is not None
                     for b in ctx.bias_refs]
            if not torch.is_grad_enabled() and all(s_ or not w_ for s_, w_ in zip(sinks, want)):
                for b, w_ in zip(ctx.bias_refs, want):          # the same column sums, added into both buffers
                    if w_:
                        _bias_grad(dy, b, weight.shape[0])
            else:
                s = SumRowsF.apply(dy)[:weight.shape[0]]
                db = s if want[0] else None
                dbs = s if want[1] else None
        return dh, dx, dw, db, dws, dbs, None


def conv_skip(h, x, weight, bias, wskip, bskip, h_relu=False):
    return ConvSkipF.apply(h, x, weight, bias, wskip, bskip, h_relu)


class ConvDgradF(Function):
    """dx = conv_transpose(dy, w)  (the data gradient of ConvF, itself differentiable)."""

    @staticmethod
    def forward(ctx, dy, weight, CinP):
        k = kernel_of(weight)
        wT = PACKS.get(weight, "dgrad", dy.shape[-1], CinP)
        ctx.save_for_backward(dy, weight)
        _prof_real(weight, CinP, dy.shape[-1])
        return K.conv_dgrad(dy, wT, k)

    @staticmethod
    def backward(ctx, ddx):
        dy, weight = ctx.saved_tensors
        ddx = ddx.contiguous()
        g_dy = g_w = None
        if ctx.needs_input_grad[0]:
            g_dy = ConvF.apply(ddx, weight, None, None, False, False, False)
        if ctx.needs_input_grad[1]:
            g_w = _wgrad(dy, ddx, weight)
        return g_dy, g_w, None


class ConvWgradF(Function):
    """dw = sum_pos dy (x) x, returned with the parameter's logical shape (channels-last memory)."""

    @staticmethod
    def forward(ctx, dy, x, weight):
        k = kernel_of(weight)
        _prof_real(weight, x.shape[-1], dy.shape[-1])
        dwp = K.conv_wgrad(dy, x, k)
        dw3 = K.unpack_wgrad(dwp, weight.shape[0], weight.shape[1])
        ctx.save_for_backward(dy, x)
        ctx.k = k
        ctx.wshape = tuple(weight.shape)
        return grad_like_weight(dw3, weight)

    @staticmethod
    @once_differentiable
    def backward(ctx, ddw):
        # d/d(dy) = conv(x, ddw), d/dx = conv_transpose(dy, ddw): only reached by third-order graphs
        dy, x = ctx.saved_tensors
        Cout, Cin = ctx.wshape[0], ctx.wshape[1]
        w3 = w3_view(ddw.detach().clone())
        g_dy = g_x = None
        if ctx.needs_input_grad[0]:
            g_dy = K.conv_fprop(x, K.pack_weight(w3, dy.shape[-1], x.shape[-1]), None, None, ctx.k)
        if ctx.needs_input_grad[1]:
            g_x = K.conv_dgrad(dy, K.pack_dgrad_weight(w3, dy.shape[-1], x.shape[-1]), ctx.k)
        return g_dy, g_x, None


class ConvSd2F(Function):
    """y = conv3d(x, w, stride (2,1,1), padding 1) + b: the even output planes of the stride-1 convolution.
    The discriminator stem (resnet3d.py:15-16) pools its second convolution with AvgPool3d((1,2,2), 2) -- kernel 1,
    stride 2 along d -- so the odd planes are never read; results are identical at half the MACs."""

    @staticmethod
    def forward(ctx, x, weight, bias, x_relu=False):
        wp = PACKS.get(weight, "fprop", weight.shape[0], x.shape[-1])
        weight._t2v_conv = True
        ctx.has_bias = bias is not None
        ctx.bias_ref = bias
        ctx.x_relu = x_relu
        ctx.save_for_backward(x, weight)
        return K.conv_fprop_sd2(x, wp, _pad_bias(bias, weight.shape[0]))

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            if not ctx.x_relu:
                dx = ConvSd2DgradF.apply(dy, weight)
            elif torch.is_grad_enabled():
                dx = ReluBwdF.apply(ConvSd2DgradF.apply(dy, weight), x)
            else:
                dx = K.conv_dgrad_sd2(dy, PACKS.get(weight, "dgrad", dy.shape[-1], weight.shape[1]), relu_ref=x)
        if ctx.needs_input_grad[1]:
            dw = _wgrad(dy, x, weight, sd2=True)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = _bias_grad(dy, ctx.bias_ref, weight.shape[0])
        return dx, dw, db, None


class ConvSd2DgradF(Function):
    @staticmethod
    def forward(ctx, dy, weight):
        wT = PACKS.get(weight, "dgrad", dy.shape[-1], weight.shape[1])
        ctx.save_for_backward(dy, weight)
        return K.conv_dgrad_sd2(dy, wT)

    @staticmethod
    def backward(ctx, ddx):
        dy, weight = ctx.saved_tensors
        ddx = ddx.contiguous()
        g_dy = g_w = None
        if ctx.needs_input_grad[0]:
            g_dy = ConvSd2F.apply(ddx, weight, None, False)
        if ctx.needs_input_grad[1]:
            g_w = _wgrad(dy, ddx, weight, sd2=True)
        return g_dy, g_w


class ConvSd2WgradF(Function):
    @staticmethod
    def forward(ctx, dy, x, weight):
        return grad_like_weight(K.conv_wgrad_sd2(dy, x), weight)

    @staticmethod
    @once_differentiable
    def backward(ctx, ddw):
        raise NotImplementedError("third-order graph through the stride-(2,1,1) weight gradient")


def conv_sd2(x, weight, bias=None, x_relu=False):
    return ConvSd2F.apply(x, weight, bias, x_relu)


class SumRowsF(Function):
    """fp32 (C,) = sum over positions (bias gradient)."""

    @staticmethod
    def forward(ctx, x):
        ctx.shape = tuple(x.shape)
        return K.sum_rows(x)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        N = ctx.shape[0]
        return K.broadcast_spatial(g.view(1, -1).expand(N, -1).contiguous(), ctx.shape)


def conv(x, weight, bias=None, residual=None, relu=False, x_relu=False, relu_later=False):
    """x_relu / relu_later: see ConvF (both must be set consistently by the block that wires producer and consumer)."""
    return ConvF.apply(x, weight, bias, residual, relu, x_relu, relu_later)


# ------------------------------------------------------------------------------------- general conv (TGAN / TCWYT)
def _t3(v):
    """int | 1/2/3-tuple -> (d, h, w) triple padded on the left with `fill` semantics of the caller."""
    return tuple(v)


def conv_args(module):
    """(k, s, p) triples of an nn.Conv{1,2,3}d / nn.ConvTranspose{1,2,3}d container (unit extents on the left)."""
    nd = len(module.kernel_size)
    k = (1,) * (3 - nd) + tuple(module.kernel_size)
    s = (1,) * (3 - nd) + tuple(module.stride)
    p = (0,) * (3 - nd) + tuple(module.padding)
    return k, s, p


class GConvF(Function):
    """Strided / padded convolution on a CL tensor: the k4 s2 p1 and head convolutions of
    models/tcwyt/video_discrim.py:12-46, frame_discrim.py:8-49, motion_discrim.py:8-19.  The backward is composed of
    GConvDgradF / GConvWgradF, so the critics' gradient penalty can differentiate it a second time."""

    @staticmethod
    def forward(ctx, x, weight, bias, k, s, p, out_f32=False):
        Cout, Cin = weight.shape[0], weight.shape[1]
        CinP, CoutP = x.shape[-1], round16(Cout)
        wp = PACKS.get(weight, "gconv", CoutP, CinP)
        y = K.gconv_fprop(x, wp, _pad_bias(bias, CoutP), k, s, p, out_f32, cin_real=Cin)
        ctx.cfg = (k, s, p, bias is not None)
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        k, s, p, has_bias = ctx.cfg
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        if dy.dtype != x.dtype:                      # fp32 output of a critic's last layer in bf16 storage mode
            dy = CastStoreF.apply(dy)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = GConvDgradF.apply(dy, weight, tuple(x.shape[1:4]), x.shape[-1], k, s, p)
        if ctx.needs_input_grad[1]:
            dw = GConvWgradF.apply(dy, x, weight, k, s, p)
        if has_bias and ctx.needs_input_grad[2]:
            db = SumRowsF.apply(dy)[:weight.shape[0]]
        return dx, dw, db, None, None, None, None


class GConvDgradF(Function):
    """dx = gconv_dgrad(dy, w): the data gradient of GConvF, itself differentiable (d/d(dy) = the convolution of the
    upstream gradient, d/dw = the weight gradient of dy against it)."""

    @staticmethod
    def forward(ctx, dy, weight, in_sp, CinP, k, s, p):
        wp = PACKS.get(weight, "gconv", dy.shape[-1], CinP)
        ctx.cfg = (k, s, p)
        ctx.save_for_backward(dy, weight)
        return K.gconv_dgrad(dy, wp, None, in_sp, k, s, p, cin_real=weight.shape[1])

    @staticmethod
    def backward(ctx, ggx):
        k, s, p = ctx.cfg
        dy, weight = ctx.saved_tensors
        ggx = ggx.contiguous()
        g_dy = g_w = None
        if ctx.needs_input_grad[0]:
            g_dy = GConvF.apply(ggx, weight, None, k, s, p, False)
        if ctx.needs_input_grad[1]:
            g_w = GConvWgradF.apply(dy, ggx, weight, k, s, p)
        return g_dy, g_w, None, None, None, None, None


class GConvWgradF(Function):
    """dw = gconv_wgrad(dy, x), returned with the parameter's logical shape."""

    @staticmethod
    def forward(ctx, dy, x, weight, k, s, p):
        Cout, Cin = weight.shape[0], weight.shape[1]
        dw3 = K.unpack_wgrad(K.gconv_wgrad(dy, x, k, s, p, cin_real=Cin), Cout, Cin)
        return grad_like_weight(dw3, weight)

    @staticmethod
    @once_differentiable
    def backward(ctx, ddw):
        raise NotImplementedError("third-order graph through the general convolution's weight gradient")


class GConvTF(Function):
    """Transposed convolution (first-order) = the data-gradient kernel of the convolution that shares its weight
    tensor: weight (Cin_t, Cout_t, k...) is that convolution's (Cout, Cin, k...).  models/tgan/gen.py:21-25,
    tgan/temporal_gen.py:16-20, tcwyt/gen.py:14-30."""

    @staticmethod
    def forward(ctx, x, weight, bias, k, s, p, out_f32=False):
        Cin_t, Cout_t = weight.shape[0], weight.shape[1]
        CinP, CoutP = x.shape[-1], round16(Cout_t)
        wp = PACKS.get(weight, "gconv", CinP, CoutP)                       # [Cin_t p][taps][Cout_t p]
        out_sp = tuple((i - 1) * ss - 2 * pp + kk for i, ss, pp, kk in zip(x.shape[1:4], s, p, k))
        y = K.gconv_dgrad(x, wp, _pad_bias(bias, CoutP), out_sp, k, s, p, out_f32, cin_real=Cout_t)
        ctx.cfg = (k, s, p, bias is not None)
        ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        k, s, p, has_bias = ctx.cfg
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        if dy.dtype != x.dtype:                      # fp32 output handed to a BatchNorm (conv_bn_act) in bf16 mode
            dy = K.cast_bf16(dy)
        Cin_t, Cout_t = weight.shape[0], weight.shape[1]
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            wp = PACKS.get(weight, "gconv", x.shape[-1], dy.shape[-1])
            dx = K.gconv_fprop(dy, wp, None, k, s, p, cin_real=Cout_t)
        if ctx.needs_input_grad[1]:
            dw3 = K.unpack_wgrad(K.gconv_wgrad(x, dy, k, s, p, cin_real=Cout_t), Cin_t, Cout_t)
            dw = grad_like_weight(dw3, weight)
        if has_bias and ctx.needs_input_grad[2]:
            db = K.sum_rows(dy)[:Cout_t]
        return dx, dw, db, None, None, None, None


def gconv(x, module, out_f32=False):
    """nn.Conv{1,2,3}d container applied to a CL tensor (any stride / padding); out_f32: fp32 output (the last layer
    of a critic: its scalar predictions are not rounded to bf16)."""
    k, s, p = conv_args(module)
    return GConvF.apply(x, module.weight, module.bias, k, s, p, out_f32)


def gconv_transpose(x, module, out_f32=False):
    """nn.ConvTranspose{1,2,3}d container applied to a CL tensor (output_padding 0)."""
    k, s, p = conv_args(module)
    return GConvTF.apply(x, module.weight, module.bias, k, s, p, out_f32)


class CastStoreF(Function):
    """fp32 CL -> the storage dtype (bf16 mode: one rounding); backward: the gradient back in fp32.  A cast is
    linear, so each direction's backward is the other one (CastF32F) and second-order graphs pass through."""

    @staticmethod
    def forward(ctx, x):
        return K.cast_bf16(x.contiguous()) if K.STORE == BF16 and x.dtype == F32 else x

    @staticmethod
    def backward(ctx, dy):
        return CastF32F.apply(dy.contiguous()) if dy.dtype == BF16 else dy


class CastF32F(Function):
    """bf16 CL -> fp32 (the backward of CastStoreF); backward: the gradient rounded back to bf16"""

    @staticmethod
    def forward(ctx, x):
        return K.cast_f32(x)

    @staticmethod
    def backward(ctx, g):
        return CastStoreF.apply(g.contiguous())


def conv_bn_act(x, conv_module, bn, act, transpose=False):
    """(transposed) convolution -> BatchNorm (batch statistics) -> activation of the TGAN / TCWYT stacks
    (models/tgan/gen.py:33-43, tgan/temporal_gen.py:26-33, tcwyt/gen.py:13-33, tcwyt/video_discrim.py:11-26,
    tcwyt/frame_discrim.py:8-18).  The convolution's fp32 accumulator goes to the BatchNorm UNROUNDED (statistics,
    normalisation and activation in fp32, typed kernels) and only the activation's output is rounded to bf16 for
    the next convolution: one rounding per layer instead of two, and batch statistics of B = 8 samples that are not
    computed from bf16-rounded values (the critics' means of these families are near-cancelling sums)."""
    f = gconv_transpose if transpose else gconv
    if fp32_mode():
        return bn_act(f(x, conv_module), bn, act)
    return CastStoreF.apply(bn_act(f(x, conv_module, out_f32=True), bn, act))


class LeakyF(Function):
    @staticmethod
    def forward(ctx, x, slope):
        y = K.leaky_relu_fwd(x, slope)
        ctx.slope = slope
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        return LeakyBwdF.apply(dy.contiguous(), y, ctx.slope), None


class LeakyBwdF(Function):
    """dx = dy * (ref > 0 ? 1 : slope); linear in dy, piecewise constant in ref (no gradient w.r.t. ref)."""

    @staticmethod
    def forward(ctx, dy, ref, slope):
        ctx.slope = slope
        ctx.save_for_backward(ref)
        return K.leaky_relu_bwd(dy, ref, slope)

    @staticmethod
    def backward(ctx, ggx):
        (ref,) = ctx.saved_tensors
        return LeakyBwdF.apply(ggx.contiguous(), ref, ctx.slope), None, None


def leaky_relu(x, slope=0.2):
    return LeakyF.apply(x, slope)


class TanhF(Function):
    @staticmethod
    def forward(ctx, x):
        y = K.tanh_fwd(x)
        ctx.save_for_backward(y)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        return K.tanh_bwd(dy.contiguous(), y)


def tanh(x):
    return TanhF.apply(x)


def bn_act(x, bn, act=0):
    """BatchNorm1d/2d/3d (batch statistics in train()) + fused activation on a CL tensor of any rank-5 shape:
    act 0 none, 1 ReLU, 2 LeakyReLU(0.2).  Channel counts that are not a multiple of 16 (BatchNorm1d(356) of
    models/tcwyt/gen.py:37) run on zero/one-padded parameter copies."""
    C, Cp = bn.num_features, x.shape[-1]
    if Cp == C:
        return BnReluUpF.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, act, 1, bn.training, bn.eps,
                               bn.momentum)
    import torch.nn.functional as Fnn
    gamma = Fnn.pad(bn.weight, (0, Cp - C), value=1.0)
    beta = Fnn.pad(bn.bias, (0, Cp - C))
    rm = Fnn.pad(bn.running_mean, (0, Cp - C))
    rv = Fnn.pad(bn.running_var, (0, Cp - C), value=1.0)
    y = BnReluUpF.apply(x, gamma, beta, rm, rv, act, 1, bn.training, bn.eps, bn.momentum)
    if bn.training:
        bn.running_mean.copy_(rm[:C])
        bn.running_var.copy_(rv[:C])
    return y


def linear_cl(x, module):
    """nn.Linear container on a CL tensor (..., CinP) -> (..., CoutP) through the 1x1x1 conv engine."""
    return conv(x, module.weight, module.bias)


def vec_to_cl(v, Cp=None):
    """fp32 (B, C) -> CL bf16 (B,1,1,1,Cp) (zero channel padding)."""
    B, C = v.shape
    return to_cl(v.reshape(B, C, 1, 1, 1), Cp)


# ------------------------------------------------------------------------------------- ReLU
class ReluF(Function):
    @staticmethod
    def forward(ctx, x, later=False):
        y = K.relu_fwd(x)
        ctx.later = later
        if not later:
            ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        if ctx.later:                   # every consumer of y masks its own data gradient (ConvF x_relu)
            return dy, None
        (y,) = ctx.saved_tensors
        return ReluBwdF.apply(dy.contiguous(), y), None


class ReluBwdF(Function):
    """dx = dy * (ref > 0); linear in dy, piecewise constant in ref."""

    @staticmethod
    def forward(ctx, dy, ref):
        ctx.save_for_backward(ref)
        return K.relu_bwd(dy, ref)

    @staticmethod
    def backward(ctx, ddx):
        (ref,) = ctx.saved_tensors
        return ReluBwdF.apply(ddx.contiguous(), ref), None


def relu(x, later=False):
    """later=True: the consumers apply the backward mask (ops.conv(..., x_relu=True))."""
    return ReluF.apply(x, later)


# ------------------------------------------------------------------------------------- avg-pool
class PoolF(Function):
    """y = avg_pool3d(x, kernel, stride, pad, count_include_pad) [+ residual]."""

    @staticmethod
    def forward(ctx, x, residual, kernel, stride, pad):
        ctx.cfg = (tuple(x.shape), tuple(kernel), tuple(stride), tuple(pad))
        ctx.has_res = residual is not None
        return K.avgpool_fwd(x, kernel, stride, pad, residual)

    @staticmethod
    def backward(ctx, dy):
        shape, kernel, stride, pad = ctx.cfg
        dy = dy.contiguous()
        dx = PoolBwdF.apply(dy, shape, kernel, stride, pad) if ctx.needs_input_grad[0] else None
        return dx, (dy if ctx.has_res else None), None, None, None


class PoolBwdF(Function):
    @staticmethod
    def forward(ctx, dy, shape, kernel, stride, pad):
        ctx.cfg = (kernel, stride, pad)
        return K.avgpool_bwd(dy, shape, kernel, stride, pad)

    @staticmethod
    def backward(ctx, ddx):
        kernel, stride, pad = ctx.cfg
        return PoolF.apply(ddx.contiguous(), None, kernel, stride, pad), None, None, None, None


def avg_pool(x, kernel, stride, pad=(0, 0, 0), residual=None):
    return PoolF.apply(x, residual, kernel, stride, pad)


def down_sample_cfg(shape):
    """kernel/stride/pad of the reference's DownSample (models/layers.py:202-217) for a CL shape."""
    k, s, p = [1, 1, 1], [1, 1, 1], [0, 0, 0]
    for i in range(3):
        size = shape[1 + i]
        if size == 1:
            continue
        k[i] = s[i] = 2
        if size % 2:
            p[i] = 1
    return tuple(k), tuple(s), tuple(p)


# ------------------------------------------------------------------------------------- nearest x2
class UpsampleF(Function):
    @staticmethod
    def forward(ctx, x):
        return K.upsample2x_fwd(x)

    @staticmethod
    def backward(ctx, dy):
        return UpsampleBwdF.apply(dy.contiguous())


class UpsampleBwdF(Function):
    @staticmethod
    def forward(ctx, dy):
        return K.upsample2x_bwd(dy)

    @staticmethod
    def backward(ctx, ddx):
        return UpsampleF.apply(ddx.contiguous())


def upsample2x(x):
    return UpsampleF.apply(x)


# ------------------------------------------------------------------------------------- layout boundary
class ToCLF(Function):
    """fp32 (N,C,D,H,W) -> CL bf16 (N,D,H,W,Cp) (zero channel padding)."""

    @staticmethod
    def forward(ctx, x, Cp):
        ctx.C = x.shape[1]
        ctx.Cp = Cp
        return K.nchw_to_cl(x.contiguous(), Cp)

    @staticmethod
    def backward(ctx, dy):
        return FromCLF.apply(dy.contiguous(), ctx.C), None


class RgbToCLF(Function):
    """fp32 (N,3,D,H,W) -> (CL16 bf16, differentiable; CL4 bf16, auxiliary input of the direct stem kernels)."""

    @staticmethod
    def forward(ctx, x):
        y16, y4 = K.rgb_to_cl(x.contiguous(), True)
        ctx.mark_non_differentiable(y4)
        return y16, y4

    @staticmethod
    def backward(ctx, dy16, _):
        return FromCLF.apply(dy16.contiguous(), 3)


def rgb_to_cl(x):
    return RgbToCLF.apply(x)


class FromCLF(Function):
    """CL bf16 (N,D,H,W,Cp) -> fp32 (N,C,D,H,W)."""

    @staticmethod
    def forward(ctx, x, C):
        ctx.Cp = x.shape[-1]
        return K.cl_to_nchw(x, C)

    @staticmethod
    def backward(ctx, dy):
        return ToCLF.apply(dy.contiguous(), ctx.Cp), None


def to_cl(x, Cp=None):
    return ToCLF.apply(x, Cp or round16(x.shape[1]))


def from_cl(x, C):
    return FromCLF.apply(x, C)


# ------------------------------------------------------------------------------------- RGB stem (im2col)
class Im2col3F(Function):
    """fp32 (N,C,D,H,W) clip -> CL bf16 (N,D,H,W,Kp) with the 27 taps of a 3^3 conv unrolled into channels
    (tap-major, then c; zero padded): the first discriminator conv (resnet3d.py:12) becomes a 1x1x1 GEMM."""

    @staticmethod
    def forward(ctx, x, Kp):
        ctx.C = x.shape[1]
        return K.im2col3(x.contiguous(), Kp)

    @staticmethod
    def backward(ctx, dcol):
        return Col2im3F.apply(dcol.contiguous(), ctx.C), None


class Col2im3F(Function):
    @staticmethod
    def forward(ctx, dcol, C):
        ctx.Kp = dcol.shape[-1]
        return K.col2im3(dcol, C)

    @staticmethod
    def backward(ctx, ddx):
        return Im2col3F.apply(ddx.contiguous(), ctx.Kp), None


def _stem_pack(weight):
    """(64, 3, 3,3,3) parameter -> bf16 (64, 128) operand of t2v_stem_fprop: k = tap * 4 + c, zero padded."""
    ent = PACKS.store.get(("stem", id(weight)))
    key = PACKS._key(weight)
    if ent is None or ent[0] != key or ent[2]() is not weight:
        with torch.no_grad():
            wp = K.stem_pack_weight(w3_view(weight).detach())                      # (64, 27, 3) fp32 -> (64, 128)
        ent = (PACKS._key(weight), wp, weakref.ref(weight))
        PACKS.store[("stem", id(weight))] = ent
    return ent[1]


_SKIP_LEAF_INPUT_GRADS = [False]


class skip_leaf_input_grads(object):
    """Inside this context a first-order backward pass does not compute d(loss)/d(input clip) when the clip is a LEAF
    (the gradient penalty's interpolated x_hat, gan/losses.py:140-145): loss.backward() would only deposit it in
    x_hat.grad, which nobody reads -- the discriminator step updates D's parameters (cond_gan.py:157-164).  The
    generator step, whose fake clips are non-leaf, is unaffected."""

    def __enter__(self):
        self.prev = _SKIP_LEAF_INPUT_GRADS[0]
        _SKIP_LEAF_INPUT_GRADS[0] = True

    def __exit__(self, *a):
        _SKIP_LEAF_INPUT_GRADS[0] = self.prev


class StemConvF(Function):
    """h = relu(conv3d(x, w, padding 1) + b), the RGB stem (resnet3d.py:12-13), on t2v_stem_fprop / _wgrad: the
    im2col tile lives in shared memory only.  x is given twice: fp32 (N,3,D,H,W) -- the autograd input -- and its
    bf16 CL16 image xc, which the kernels read.  The ReLU mask of the backward pass is applied by the consumer
    (ConvF / ConvSd2F with x_relu).  The data gradient (gradient penalty, generator step) keeps the im2col
    formulation, which is closed under a second differentiation."""

    @staticmethod
    def forward(ctx, x, xc, weight, bias):
        weight._t2v_conv = True
        ctx.has_bias = bias is not None
        ctx.bias_ref = bias
        ctx.x_leaf = x.is_leaf
        y = K.stem_fprop(xc, _stem_pack(weight), None if bias is None else bias.detach(), True)
        ctx.save_for_backward(xc, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        xc, weight = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0] and not (ctx.x_leaf and _SKIP_LEAF_INPUT_GRADS[0] and not torch.is_grad_enabled()):
            w2d = stem_weight_2d(weight)
            dx = Col2im3F.apply(ConvDgradF.apply(dy, w2d, stem_k(3)), 3)
        if ctx.needs_input_grad[2]:
            dw = StemWgradF.apply(dy, xc, weight)
        if ctx.has_bias and ctx.needs_input_grad[3]:
            db = _bias_grad(dy, ctx.bias_ref, weight.shape[0])
        return dx, None, dw, db


class StemWgradF(Function):
    @staticmethod
    def forward(ctx, dy, xc, weight):
        return grad_like_weight(K.stem_wgrad(dy, xc), weight)

    @staticmethod
    @once_differentiable
    def backward(ctx, ddw):
        raise NotImplementedError("third-order graph through the stem weight gradient")


def stem_conv(x, xc, weight, bias):
    return StemConvF.apply(x, xc.detach(), weight, bias)


def stem_k(C):
    """channel count of the im2col'ed clip: 27*C rounded up to a multiple of 32 (BLOCK_K of the engine)."""
    return (27 * C + 31) // 32 * 32


def im2col3(x):
    return Im2col3F.apply(x, stem_k(x.shape[1]))


def stem_weight_2d(weight):
    """(Cout, C, 3,3,3) parameter -> differentiable (Cout, 27*C) VIEW in (tap, c) order (its channels-last
    memory), i.e. the Linear weight that multiplies an im2col3 row."""
    w3 = w3_view(weight)                      # re-homes the parameter to channels-last memory once
    return w3.reshape(w3.shape[0], w3.shape[1] * w3.shape[2])


# ------------------------------------------------------------------------------------- sum-pool head
class SumSpatialF(Function):
    """torch.sum(x, [2,3,4]) (models/resnet3d.py:48): CL bf16 -> fp32 (N, C)."""

    @staticmethod
    def forward(ctx, x):
        ctx.shape = tuple(x.shape)
        return K.sum_spatial(x)

    @staticmethod
    def backward(ctx, g):
        return BroadcastSpatialF.apply(g.contiguous(), ctx.shape)


class BroadcastSpatialF(Function):
    @staticmethod
    def forward(ctx, g, shape):
        return K.broadcast_spatial(g, shape)

    @staticmethod
    def backward(ctx, dy):
        return SumSpatialF.apply(dy.contiguous()), None


def sum_spatial(x):
    return SumSpatialF.apply(x)


# ------------------------------------------------------------------------------------- BatchNorm(+ReLU+Up)
class BnReluUpF(Function):
    """[nearest x2]([relu](BatchNorm2d(x))) with batch statistics in train(); updates the running
    statistics in place (models/layers.py:171-173,175-176,249-250)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, relu, up, training, eps, momentum):
        y, mean_invstd, scale_shift = K.bn_forward(x, gamma.detach(), beta.detach(), running_mean, running_var, relu,
                                                   up, eps, momentum, training)
        ctx.cfg = (relu, up, training)
        ctx.save_for_backward(x, gamma, mean_invstd, scale_shift)
        return y

    @staticmethod
    def backward(ctx, dy):
        relu, up, training = ctx.cfg
        x, gamma, mean_invstd, scale_shift = ctx.saved_tensors
        assert training, "eval-mode BatchNorm backward is not on the training path"
        if torch.is_grad_enabled():          # create_graph: the backward itself is differentiable (BnBwdF)
            dx, dgamma, dbeta = BnBwdF.apply(dy.contiguous(), x, gamma, mean_invstd, scale_shift, relu, up)
        else:
            dx, dgamma, dbeta = K.bn_backward(dy.contiguous(), x, mean_invstd, scale_shift, relu, up)
        return dx, dgamma, dbeta, None, None, None, None, None, None, None


class BnBwdF(Function):
    """(dx, dgamma, dbeta) = the BatchNorm (+ activation) backward of BnReluUpF as a function of (dy, x, gamma).  With
    up == 1 its backward is the double-backward kernel (the critics' gradient penalty); mean_invstd / scale_shift are
    the forward's saved statistics, whose dependence on x and gamma is part of that kernel's formula.  The upsampling
    form (up == 2, generator only) is first-order: differentiating it again raises."""

    @staticmethod
    def forward(ctx, dy, x, gamma, mean_invstd, scale_shift, relu, up):
        dx, dgamma, dbeta = K.bn_backward(dy, x, mean_invstd, scale_shift, relu, up)
        ctx.cfg = (relu, up)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(dy, x, mean_invstd, scale_shift)
        return dx, dgamma, dbeta

    @staticmethod
    @once_differentiable
    def backward(ctx, ggx, ggamma, ggbeta):
        relu, up = ctx.cfg
        if up != 1:
            raise NotImplementedError("second-order graph through the upsampling BatchNorm backward")
        dy, x, mean_invstd, scale_shift = ctx.saved_tensors
        if ggx is None:
            ggx = torch.zeros_like(x)
        cont = lambda t: None if t is None else t.contiguous()
        gx, gdy, dgamma = K.bn_backward_backward(dy, x, mean_invstd, scale_shift, ggx.contiguous(), cont(ggamma),
                                                 cont(ggbeta), relu, 1)
        return gdy, gx, dgamma, None, None, None, None


def bn_relu_up(x, bn, relu=True, up=1):
    """bn: an nn.BatchNorm2d parameter container."""
    return BnReluUpF.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, relu, up, bn.training, bn.eps,
                           bn.momentum)


# ------------------------------------------------------------------------------------- render tail
class RenderF(Function):
    """tanh + (B*T,1,H,W,Cp) bf16 -> fp32 (B,C,T,H,W) (layers.py:252; tganv2_cond/gen.py:116-119)."""

    @staticmethod
    def forward(ctx, pre, B, T, C):
        y = K.render_fwd(pre, B, T, C)
        ctx.Cp = pre.shape[-1]
        ctx.save_for_backward(y)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        return K.render_bwd(dy.contiguous(), y, ctx.Cp), None, None, None


def render_tail(pre, B, T, C=3):
    return RenderF.apply(pre, B, T, C)


# ------------------------------------------------------------------------------------- frame subsampling
class GatherFramesF(Function):
    """Subsample x[::2, :, bt::2] (layers.py:106-111) on a merged-frame CL map (B*T, 1, H, W, C)."""

    @staticmethod
    def forward(ctx, x, B, T, bt):
        ctx.cfg = (B, T, bt)
        return K.gather_frames(x, B, T, bt)

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        B, T, bt = ctx.cfg
        return K.scatter_frames(dy.contiguous(), B, T, bt), None, None, None


def gather_frames(x, B, T, bt):
    return GatherFramesF.apply(x, B, T, bt)


# ------------------------------------------------------------------------------------- ConvLSTM


class ConvLstmF(Function):
    """The whole TGANv2 temporal generator (models/conv_lstm.py:32-38,75-97): `steps` LSTM steps on a
    (B, 1, fh, fw, C) CL plane.  Step 0 sees the input, later steps see zeros (so Wx*(0) = bias);
    peepholes are identically zero in the reference.  Per step: ONE kernel -- the gate GEMM on the tensor cores
    ([i|f|g|o] interleaved along Cout) with the sigmoid / tanh cell update as its epilogue (t2v_conv_lstm_step; the
    fp32 parity mode keeps the unfused GEMM + cell kernel).  Output: (B*steps, 1, fh, fw, C)
    merged-frame map in (b, t) order (tganv2_cond/gen.py:75-76,91-96)."""

    @staticmethod
    def forward(ctx, x, wx, wh, bx, steps):
        # wx, wh: fp32 (4*Hd, taps, Cin|Hd) stacked [i|f|g|o] views/copies; bx fp32 (4*Hd,)
        B, D, fh, fw, Cin = x.shape
        Hd = wh.shape[0] // 4
        taps = wx.shape[1]
        k = (1, 3, 3) if taps == 9 else (1, 1, 1)
        gates, cs, hs = [], [], []
        h = c = None
        if not fp32_mode() and hasattr(K, "conv_lstm_step") and Hd % 32 == 0 and x.shape[-1] % 16 == 0:
            # gate GEMM + sigmoid / tanh cell update in ONE kernel per step (t2v_conv_lstm_step): the gates are
            # interleaved per 32 hidden units along Cout so that an accumulator tile carries [i|f|g|o] of its units;
            # h_t goes to the next step's operand AND to its (b, t) slot of the merged frame map from the epilogue
            il = K.lstm_gate_interleave(Hd, x.device)
            wx_p = K.pack_weight(wx.detach()[il].contiguous())
            wh_p = K.pack_weight(wh.detach()[il].contiguous())
            b_il = bx.detach()[il].contiguous()
            out = torch.empty((B * steps, 1, fh, fw, Hd), device=x.device, dtype=x.dtype)
            for t in range(steps):
                g, c, h = K.conv_lstm_step(x if t == 0 else h, wx_p if t == 0 else wh_p, b_il, c, k, out, t, steps)
                gates.append(g)
                cs.append(c)
                hs.append(h)
        else:
            wx_p = K.pack_weight(wx.detach().contiguous())
            wh_p = K.pack_weight(wh.detach().contiguous())
            for t in range(steps):
                src = x if t == 0 else h
                wp = wx_p if t == 0 else wh_p
                g = K.conv_fprop(src, wp, bx.detach(), None, k, False, True)           # fp32 (B,1,fh,fw,4Hd)
                c, h, _ = K.lstm_cell_fwd(g, c)
                gates.append(g)
                cs.append(c)
                hs.append(h)
            out = torch.stack(hs, dim=1).reshape(B * steps, 1, fh, fw, Hd)              # (b, t) frame order
        ctx.save_for_backward(x, wx, wh, *gates, *cs, *hs)
        ctx.cfg = (steps, k, Hd)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, dout):
        steps, k, Hd = ctx.cfg
        saved = ctx.saved_tensors
        x, wx, wh = saved[0], saved[1], saved[2]
        gates = saved[3:3 + steps]
        cs = saved[3 + steps:3 + 2 * steps]
        hs = saved[3 + 2 * steps:3 + 3 * steps]
        B, D, fh, fw, Cin = x.shape
        dout = dout.reshape(B, steps, 1, fh, fw, Hd)
        whT = K.pack_dgrad_weight(wh.detach().contiguous())
        dh_rec = None                      # bf16 gradient flowing into h_{t} from step t+1
        dc = None
        dgs = [None] * steps
        for t in range(steps - 1, -1, -1):
            dh = dout[:, t].float()
            if dh_rec is not None:
                dh = dh + dh_rec.float()
            dg, dc = K.lstm_cell_bwd(gates[t], cs[t - 1] if t > 0 else None, cs[t], dh.contiguous(), dc)
            dgs[t] = dg
            if t > 0:
                dh_rec = K.conv_dgrad(dg, whT, k)
        # weight gradients: Wh over steps 1.., Wx from step 0, bias over all steps
        dwh = torch.zeros(wh.shape, device=x.device, dtype=F32)
        if steps > 1:
            dg_all = torch.cat(dgs[1:], dim=0)
            h_all = torch.cat(hs[:steps - 1], dim=0)
            dwh = K.conv_wgrad(dg_all, h_all, k)
        dwx = K.conv_wgrad(dgs[0], x, k)
        db = K.sum_rows(torch.cat(dgs, dim=0))
        dx = None
        if ctx.needs_input_grad[0]:
            dx = K.conv_dgrad(dgs[0], K.pack_dgrad_weight(wx.detach().contiguous()), k)
        return dx, dwx, dwh, db, None


# ------------------------------------------------------------------------------------- non-local block
class AttentionCoreF(Function):
    """o = softmax(theta . maxpool(phi)^T) . maxpool(g) per map (t2v_attention_fwd / _bwd), first-order."""

    @staticmethod
    def forward(ctx, theta, phi, g, c8, c2):
        ctx.cfg = (c8, c2)
        ctx.save_for_backward(theta, phi, g)
        return K.attention_fwd(theta, phi, g, c8, c2)

    @staticmethod
    @once_differentiable
    def backward(ctx, do):
        theta, phi, g = ctx.saved_tensors
        c8, c2 = ctx.cfg
        dtheta, dphi, dg = K.attention_bwd(theta, phi, g, do.contiguous(), c8, c2)
        return dtheta, dphi, dg, None, None


# ---- differentiable primitives (every backward is again one of them: the discriminator's block is differentiated
# ---- twice by the gradient penalty, gan/losses.py:169-178)
class ScaleF(Function):
    """y = s * x  (s: 0-d fp32 tensor on the device)"""

    @staticmethod
    def forward(ctx, x, s):
        ctx.save_for_backward(x, s)
        return K.scale(x, s.detach().reshape(1).float())

    @staticmethod
    def backward(ctx, dy):
        x, s = ctx.saved_tensors
        dy = dy.contiguous()
        dx = ScaleF.apply(dy, s) if ctx.needs_input_grad[0] else None
        ds = DotF.apply(dy, x).reshape(s.shape).to(s.dtype) if ctx.needs_input_grad[1] else None
        return dx, ds


class DotF(Function):
    """0-d fp32 = sum a * b"""

    @staticmethod
    def forward(ctx, a, b):
        ctx.save_for_backward(a, b)
        return K.dot(a, b)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.contiguous()
        da = ScaleF.apply(b, g) if ctx.needs_input_grad[0] else None
        db = ScaleF.apply(a, g) if ctx.needs_input_grad[1] else None
        return da, db


class GradNormPenaltyF(Function):
    """0-d fp32 mean_b (||g_b||_2 - 1)^2 of g fp32 (B, ...): the non-zero-centred gradient penalty (gan/losses.py:
    180-186).  Its backward feeds the double backward through the critic; nothing differentiates it again."""

    @staticmethod
    def forward(ctx, g):
        out, norms = K.gp_norm_fwd(g)
        ctx.save_for_backward(g, norms)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        g, norms = ctx.saved_tensors
        return K.gp_norm_bwd(g, norms, gout.contiguous().reshape(()).float())


class ScaleAddF(Function):
    """y = s * o + x: the non-local block's output gamma * o + x (models/layers.py:36,68); s None: y = o + x"""

    @staticmethod
    def forward(ctx, o, x, s):
        ctx.save_for_backward(o, s)
        return K.scale_add(o, x, None if s is None else s.detach().reshape(1).float())

    @staticmethod
    def backward(ctx, dy):
        o, s = ctx.saved_tensors
        dy = dy.contiguous()
        do = None
        if ctx.needs_input_grad[0]:
            do = dy if s is None else ScaleF.apply(dy, s)
        dx = dy if ctx.needs_input_grad[1] else None
        ds = None
        if s is not None and ctx.needs_input_grad[2]:
            ds = DotF.apply(dy, o).reshape(s.shape).to(s.dtype)
        return do, dx, ds


def scale_add(o, x, s=None):
    return ScaleAddF.apply(o, x, s)


class SliceF32F(Function):
    """CL (..., Cp) -> fp32 (..., c)"""

    @staticmethod
    def forward(ctx, x, c):
        ctx.cfg = (x.shape[-1], x.dtype)
        return K.cl_slice_f32(x, c)

    @staticmethod
    def backward(ctx, dy):
        return PadCLF.apply(dy.contiguous(), ctx.cfg[0], ctx.cfg[1]), None


class PadCLF(Function):
    """fp32 (..., c) -> CL storage (..., Cp), zero padded"""

    @staticmethod
    def forward(ctx, x, Cp, dtype):
        ctx.c = x.shape[-1]
        return K.f32_pad_cl(x, Cp, dtype)

    @staticmethod
    def backward(ctx, dy):
        return SliceF32F.apply(dy.contiguous(), ctx.c), None, None


class MaxPool122F(Function):
    """max-pool (1,2,2) on fp32 (M, H, W, c) (F.max_pool2d / max_pool3d of layers.py:26-27,56-57)"""

    @staticmethod
    def forward(ctx, x):
        y, idx = K.maxpool122_fwd(x)
        ctx.save_for_backward(idx)
        return y

    @staticmethod
    def backward(ctx, dy):
        (idx,) = ctx.saved_tensors
        return PoolScatterF.apply(dy.contiguous(), idx)


class PoolScatterF(Function):
    @staticmethod
    def forward(ctx, dy, idx):
        ctx.save_for_backward(idx)
        return K.pool122_scatter(dy, idx)

    @staticmethod
    def backward(ctx, ddx):
        (idx,) = ctx.saved_tensors
        return PoolGatherF.apply(ddx.contiguous(), idx), None


class PoolGatherF(Function):
    @staticmethod
    def forward(ctx, x, idx):
        ctx.save_for_backward(idx)
        return K.pool122_gather(x, idx)

    @staticmethod
    def backward(ctx, dy):
        (idx,) = ctx.saved_tensors
        return PoolScatterF.apply(dy.contiguous(), idx), None


class BmmF(Function):
    """fp32 batched C = op(A) op(B) (torch.bmm of layers.py:32-33,64-65)"""

    @staticmethod
    def forward(ctx, a, b, ta, tb):
        ctx.save_for_backward(a, b)
        ctx.cfg = (ta, tb)
        return K.bmm(a, b, ta, tb)

    @staticmethod
    def backward(ctx, dc):
        a, b = ctx.saved_tensors
        ta, tb = ctx.cfg
        dc = dc.contiguous()
        da = db = None
        if ctx.needs_input_grad[0]:
            da = BmmF.apply(b, dc, tb, True) if ta else BmmF.apply(dc, b, False, not tb)
        if ctx.needs_input_grad[1]:
            db = BmmF.apply(dc, a, True, ta) if tb else BmmF.apply(a, dc, not ta, False)
        return da, db, None, None


class SoftmaxF(Function):
    @staticmethod
    def forward(ctx, s):
        beta = K.softmax_fwd(s)
        ctx.save_for_backward(beta)
        return beta

    @staticmethod
    def backward(ctx, dbeta):
        (beta,) = ctx.saved_tensors
        return SoftmaxBwdF.apply(beta, dbeta.contiguous())


class SoftmaxBwdF(Function):
    """dS = beta * (dbeta - <beta, dbeta>)"""

    @staticmethod
    def forward(ctx, beta, dbeta):
        ctx.save_for_backward(beta, dbeta)
        return K.softmax_bwd(beta, dbeta)

    @staticmethod
    @once_differentiable
    def backward(ctx, u):
        beta, dbeta = ctx.saved_tensors
        g_beta, g_dbeta = K.softmax_bwd_bwd(beta, dbeta, u.contiguous())
        return g_beta, g_dbeta


def attention_core(theta, phi, g, c8, c2):
    """o = softmax(theta . maxpool(phi)^T) . maxpool(g) per sample over all D*H*W positions, pooling (1,2,2)
    (models/layers.py:25-34, 55-66), from differentiable fp32 primitives.  theta / phi (N,D,H,W,C8p), g (N,D,H,W,C2p)
    CL -> o (N,D,H,W,round16(c2)) CL."""
    N, D, H, W, _ = theta.shape
    th = SliceF32F.apply(theta, c8).reshape(N, D * H * W, c8)
    ph = MaxPool122F.apply(SliceF32F.apply(phi, c8).reshape(N * D, H, W, c8)).reshape(N, -1, c8)
    gp = MaxPool122F.apply(SliceF32F.apply(g, c2).reshape(N * D, H, W, c2)).reshape(N, -1, c2)
    beta = SoftmaxF.apply(BmmF.apply(th, ph, False, True))                  # (N, P, P/4)
    o = BmmF.apply(beta, gp, False, False)                                  # (N, P, c2)
    return PadCLF.apply(o.reshape(N, D, H, W, c2), round16(c2), theta.dtype)


def nonlocal_block(x, w_theta, w_phi, w_g, w_o, gamma, pool=(1, 2, 2), fused=False):
    """SA-GAN / non-local block (models/layers.py:23-36 2-D, :52-68 3-D) on a CL tensor.

    The four 1x1(x1) convs run on the tcgen05 engine (channel counts < 16 are zero-padded).  The attention core is the
    fused kernel pair t2v_attention_fwd / _bwd (_bwd_large) where it applies (the generator's block: first-order
    autograd, bf16 storage, kernels.attention_fused_ok: up to 64 x 64 maps in its c8 = 4 / c2 = 16 configuration) and the
    differentiable primitive composition of attention_core otherwise (the discriminator's block, which the gradient
    penalty differentiates twice; fp32 storage)."""
    N, D, H, W, C = x.shape
    c8, c2 = w_theta.shape[0], w_g.shape[0]
    assert tuple(pool) == (1, 2, 2) and H % 2 == 0 and W % 2 == 0
    theta, phi, g = conv(x, w_theta), conv(x, w_phi), conv(x, w_g)
    if fused and x.dtype == BF16 and K.attention_fused_ok(D, H, W, c8, c2):        # kernels' shared-memory bound
        o = AttentionCoreF.apply(theta, phi, g, c8, c2)
    else:
        o = attention_core(theta, phi, g, c8, c2)
    return ScaleAddF.apply(conv(o, w_o), x, gamma)


# ------------------------------------------------------------------------------------- discriminator heads
class HeadF(Function):
    """pred (B,) = [feat | cond] . w + b: fc_uncond / fc of models/resnet3d.py:50-55 on fp32 (B, F) features."""

    @staticmethod
    def forward(ctx, feat, cond, w, b):
        ctx.save_for_backward(feat, cond, w)
        ctx.has_b = b is not None
        return K.head_fwd(feat.contiguous(), None if cond is None else cond.contiguous(), w.detach().reshape(-1),
                          None if b is None else b.detach())

    @staticmethod
    def backward(ctx, dpred):
        feat, cond, w = ctx.saved_tensors
        dpred = dpred.contiguous()
        dfeat = dcond = dw = db = None
        if ctx.needs_input_grad[0] or (cond is not None and ctx.needs_input_grad[1]):
            dfeat, dcond = HeadBwdDataF.apply(dpred, w, feat.shape[1], 0 if cond is None else cond.shape[1])
        if ctx.needs_input_grad[2] or (ctx.has_b and ctx.needs_input_grad[3]):
            dw, db = HeadBwdWeightF.apply(dpred, feat, cond)
            dw = dw.reshape(w.shape)
        return (dfeat if ctx.needs_input_grad[0] else None, dcond if (cond is not None and ctx.needs_input_grad[1])
                else None, dw if ctx.needs_input_grad[2] else None, db if (ctx.has_b and ctx.needs_input_grad[3])
                else None)


class HeadBwdDataF(Function):
    """(dfeat, dcond | None) = dpred (x) w"""

    @staticmethod
    def forward(ctx, dpred, w, F_, E):
        ctx.save_for_backward(dpred, w)
        return K.head_bwd_data(dpred, w.detach().reshape(-1), F_, E)

    @staticmethod
    def backward(ctx, ddfeat, ddcond):
        dpred, w = ctx.saved_tensors
        ddfeat = ddfeat.contiguous()
        ddc = None if ddcond is None else ddcond.contiguous()
        if ddc is None and w.numel() != ddfeat.shape[1]:        # caption slot present but its gradient unused
            ddc = ddfeat.new_zeros((ddfeat.shape[0], w.numel() - ddfeat.shape[1]))
        g_dpred = g_w = None
        if ctx.needs_input_grad[0]:
            g_dpred = HeadF.apply(ddfeat, ddc, w, None)
        if ctx.needs_input_grad[1]:
            g_w = HeadBwdWeightF.apply(dpred, ddfeat, ddc)[0].reshape(w.shape)
        return g_dpred, g_w, None, None


class HeadBwdWeightF(Function):
    """(dw, db) = (sum_b dpred[b] [feat | cond][b], sum_b dpred[b])"""

    @staticmethod
    def forward(ctx, dpred, feat, cond):
        ctx.save_for_backward(dpred, feat, cond)
        return K.head_bwd_weight(dpred, feat.contiguous(), None if cond is None else cond.contiguous(), True)

    @staticmethod
    def backward(ctx, ddw, ddb):
        dpred, feat, cond = ctx.saved_tensors
        ddw = ddw.contiguous()
        g_dpred = g_feat = g_cond = None
        if ctx.needs_input_grad[0]:
            g_dpred = HeadF.apply(feat, cond, ddw, None if ddb is None else ddb.contiguous())
        if ctx.needs_input_grad[1] or (cond is not None and ctx.needs_input_grad[2]):
            g_feat, g_cond = HeadBwdDataF.apply(dpred, ddw, feat.shape[1], 0 if cond is None else cond.shape[1])
            if cond is None:
                g_cond = None
        return g_dpred, g_feat, g_cond


def head_linear(feat, weight, bias, cond=None):
    """fc_uncond / fc heads (models/resnet3d.py:50-55): Linear(F [+ E], 1) on fp32 (B, F) features [and (B, E)
    captions] -> (B, 1), as one row-dot kernel (no concatenation, no cuBLAS gemv)."""
    return HeadF.apply(feat, cond, weight, bias).reshape(-1, 1)


# ------------------------------------------------------------------------------------- fused loss reduction
class RelLossF(Function):
    """sum_e weight_e * mean_j f(b_e[j] - a_e[j]) over ALL (level, prediction-pair) entries in one kernel
    (gan/cond_gan.py:51-61,108-112 with RSGANLoss / WassersteinGanLoss, gan/losses.py:55-85); mode 0 softplus, 1 id."""

    @staticmethod
    def forward(ctx, mode, weights, *tensors):
        n = len(tensors) // 2
        a_list = [t.detach().reshape(-1).contiguous() for t in tensors[:n]]
        b_list = [t.detach().reshape(-1).contiguous() for t in tensors[n:]]
        ctx.cfg = (mode, tuple(weights), n, [tuple(t.shape) for t in tensors])
        ctx.save_for_backward(*a_list, *b_list)
        ctx.ids = [id(t) for t in tensors]
        return K.rel_loss_fwd(a_list, b_list, weights, mode)

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        mode, weights, n, shapes = ctx.cfg
        saved = ctx.saved_tensors
        a_list, b_list = list(saved[:n]), list(saved[n:])
        # one zeroed buffer for every requested gradient; the kernel accumulates (an input may appear in several entries,
        # but autograd sums the per-argument gradients itself, so every argument gets its own slice)
        need = [ctx.needs_input_grad[2 + i] for i in range(2 * n)]
        sizes = [t.numel() for t in saved]
        buf = torch.zeros(sum(sz for sz, nd in zip(sizes, need) if nd), device=gout.device, dtype=F32)
        grads, off = [], 0
        for sz, nd in zip(sizes, need):
            if nd:
                grads.append(buf[off:off + sz])
                off += sz
            else:
                grads.append(None)
        K.rel_loss_bwd(a_list, b_list, grads[:n], grads[n:], weights, mode, gout.contiguous().float().reshape(1))
        return (None, None) + tuple(None if g is None else g.reshape(shp) for g, shp in zip(grads, shapes))


def rel_loss(pairs, mode):
    """pairs: list of (a, b, weight) -> scalar sum_e weight * mean f(b - a)"""
    a = [p[0] for p in pairs]
    b = [p[1] for p in pairs]
    return RelLossF.apply(mode, [float(p[2]) for p in pairs], *a, *b)


# ------------------------------------------------------------------------------------- caption LSTM
class EmbeddingF(Function):
    """nn.Embedding (models/txt/basic.py:16,51): bit-exact row gather, gradient by atomic row adds"""

    @staticmethod
    def forward(ctx, tokens, weight):
        ctx.save_for_backward(tokens)
        ctx.V = weight.shape[0]
        return K.embedding_fwd(tokens.contiguous(), weight.detach())

    @staticmethod
    @once_differentiable
    def backward(ctx, dout):
        (tokens,) = ctx.saved_tensors
        return None, K.embedding_bwd(tokens.contiguous(), dout.contiguous(), ctx.V)


class LstmLayerF(Function):
    """One (bi)directional LSTM layer over a length-masked batch (nn.LSTM on a PackedSequence,
    models/txt/basic.py:52-56): input projection of all steps and both directions as ONE GEMM on the tcgen05 engine,
    then the persistent recurrence kernel (t2v_lstm_seq_fwd).  x (B, L, In) storage dtype; lengths int32 (B,) device;
    h0 / c0 (ndir, B, H) fp32 or None; params = (w_ih, w_hh, b_ih, b_hh) per direction.
    -> out (B, L, ndir*H) storage, hn, cn (ndir, B, H) fp32."""

    @staticmethod
    def forward(ctx, x, lengths, h0, c0, *params):
        ndir = len(params) // 4
        B, L, In = x.shape
        w_ih = torch.cat([params[4 * d].detach() for d in range(ndir)], dim=0)            # (ndir*4H, In)
        w_hh = torch.stack([params[4 * d + 1].detach() for d in range(ndir)], dim=0).contiguous()   # (ndir, 4H, H)
        bias = torch.cat([(params[4 * d + 2] + params[4 * d + 3]).detach() for d in range(ndir)], dim=0)
        H = w_hh.shape[2]
        x5 = x.reshape(B * L, 1, 1, 1, In)
        gx = K.conv_fprop(x5, K.pack_weight(w_ih.reshape(ndir * 4 * H, 1, In).contiguous()), bias.contiguous(), None,
                          (1, 1, 1), False, True)
        h0c = None if h0 is None else h0.detach().float().contiguous()
        c0c = None if c0 is None else c0.detach().float().contiguous()
        out, hprev, gates, cells, hn, cn = K.lstm_seq_fwd(gx.reshape(B, L, ndir * 4 * H), K.lstm_pack_whh(w_hh), lengths,
                                                          h0c, c0c, True)
        ctx.save_for_backward(x, lengths, c0c, w_ih, w_hh, hprev, gates, cells)
        ctx.cfg = (ndir, H, In, h0 is not None, c0 is not None)
        return out, hn, cn

    @staticmethod
    @once_differentiable
    def backward(ctx, dout, dhn, dcn):
        x, lengths, c0, w_ih, w_hh, hprev, gates, cells = ctx.saved_tensors
        ndir, H, In, has_h0, has_c0 = ctx.cfg
        B, L, _ = x.shape
        dgates, dh0, dc0 = K.lstm_seq_bwd(w_hh, lengths, c0, gates, cells, None if dout is None else dout.contiguous(),
                                          None if dhn is None else dhn.contiguous().float(),
                                          None if dcn is None else dcn.contiguous().float())
        dg5 = dgates.reshape(B * L, 1, 1, 1, ndir * 4 * H)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = K.conv_dgrad(dg5, K.pack_dgrad_weight(w_ih.reshape(ndir * 4 * H, 1, In).contiguous()),
                              (1, 1, 1)).reshape(B, L, In)
        dwih = K.conv_wgrad(dg5, x.reshape(B * L, 1, 1, 1, In), (1, 1, 1)).reshape(ndir * 4 * H, In)
        dwhh = K.conv_wgrad(dg5, hprev.reshape(B * L, 1, 1, 1, ndir * H), (1, 1, 1)).reshape(ndir * 4 * H, ndir * H)
        db = K.sum_rows(dg5)
        grads = []
        for d in range(ndir):
            r = slice(d * 4 * H, (d + 1) * 4 * H)
            grads += [dwih[r], dwhh[r, d * H:(d + 1) * H], db[r], db[r]]
        return (dx, None, dh0 if has_h0 else None, dc0 if has_c0 else None) + tuple(grads)
