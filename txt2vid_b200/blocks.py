"""Building blocks of the TGANv2 networks, B200-native.

Mirrors the public classes of the reference's txt2vid/models/layers.py, conv_lstm.py and resnet3d.py:
same constructor arguments, same sub-module tree (so `state_dict()` keys, `init()` traversal order and
constructor-time RNG consumption are identical), but `forward` runs on the sm_100a kernels through
txt2vid_b200.ops instead of ATen/cuDNN.

The torch.nn.Conv*/BatchNorm*/Linear objects below are PARAMETER CONTAINERS only; their own forward is
never called.  Every block has two entry points:
  forward_cl(x)  channels-last bf16 tensors (N, D, H, W, C) -- used between blocks;
  forward(x)     the reference's signature (fp32, channel-first) -- converts at the boundary.
"""
import torch
import torch.nn as nn
from torch.nn import Parameter as P

from . import ops


def _cl2d(x):
    """fp32 (N,C,H,W) -> CL (N,1,H,W,Cp)."""
    return ops.to_cl(x.unsqueeze(2))


def _ncl2d(y, C):
    return ops.from_cl(y, C).squeeze(2)


class Identity(nn.Module):
    def forward(self, x):
        return x


class ResidualBlock(nn.Module):
    """Container with the reference's attribute names (layers.py:77-96).  Convs inside
    `inner_module` are tagged `is_residual` so that init() applies the sqrt(2) gain (util/torch/init.py:8-14)."""

    def __init__(self, inner_module=None, identity_map=None):
        super().__init__()
        self.inner_module = inner_module
        self.identity_map = identity_map if identity_map is not None else Identity()

        def tag(m):
            m.is_residual = True
        self.inner_module.apply(tag)


class Subsample(nn.Module):
    """x[::sn, :, bt::st] with bt ~ U{0..st-1} from the CPU generator (layers.py:98-111)."""

    def __init__(self, sn=2, st=2):
        super().__init__()
        self.sn = sn
        self.st = st

    def draw(self):
        """python int (eager) or a device int32 tensor (CUDA-graph mode), see hostrng.py"""
        from . import hostrng
        return hostrng.CURRENT.bt(self.st)

    def forward(self, x, bt=None):
        if bt is None:
            bt = self.draw()
        if x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and not x.requires_grad:
            from . import kernels as K
            B, C, T, H, W = x.shape
            return K.pyramid_level(x.contiguous(), H, W, self.sn, self.st, bt), bt
        return x[::self.sn, :, int(bt)::self.st], bt


class Attention(nn.Module):
    """SA-GAN non-local block, 2-D (layers.py:10-36)."""

    def __init__(self, ch, which_conv=nn.Conv2d, name='attention'):
        super().__init__()
        self.ch = ch
        self.which_conv = which_conv
        self.theta = which_conv(ch, ch // 8, kernel_size=1, padding=0, bias=False)
        self.phi = which_conv(ch, ch // 8, kernel_size=1, padding=0, bias=False)
        self.g = which_conv(ch, ch // 2, kernel_size=1, padding=0, bias=False)
        self.o = which_conv(ch // 2, ch, kernel_size=1, padding=0, bias=False)
        self.gamma = P(torch.tensor(0.), requires_grad=True)
        self.pool = (1, 2, 2)
        # The 2-D block lives in the generator (never differentiated twice) and runs on the fused attention-core
        # kernels (t2v_attention_fwd/_bwd, parity-tested): the (P x P/4) attention matrix -- 1 GB fp32 per step at batch
        # 1024 -- never exists.  Measured on B200 (scripts/attn_probe.py, 1024 maps of 32x32): fused bwd 1.49 ms against
        # 3.84 ms for the ATen composite's forward + backward.  The discriminator's 3-D block is on the
        # gradient-penalty path (double backward) and keeps the composite.
        self.fused_core = which_conv is nn.Conv2d

    def forward_cl(self, x):
        return ops.nonlocal_block(x, self.theta.weight, self.phi.weight, self.g.weight, self.o.weight, self.gamma,
                                  self.pool, fused=self.fused_core)

    def forward(self, x, y=None):
        return _ncl2d(self.forward_cl(_cl2d(x)), self.ch)


class Attention3d(Attention):
    """Non-local block, 3-D, max-pool (1,2,2) (layers.py:39-68)."""

    def __init__(self, ch, which_conv=nn.Conv3d, name='attention'):
        super().__init__(ch, which_conv=which_conv, name=name)

    def forward(self, x, y=None):
        return ops.from_cl(self.forward_cl(ops.to_cl(x)), self.ch)


class UpBlock(nn.Module):
    """BN-ReLU-Up2-conv3-BN-ReLU-conv3 + (Up2 [-conv1]) skip [+ attention] (layers.py:152-195).

    B200 schedule: [bn_stats, bn_finalize, bn_apply(+relu+up2)] -> conv3 (tcgen05) -> [bn...] ->
    conv3 with the skip added in the epilogue; the 1x1 skip conv runs at LOW resolution and is
    upsampled afterwards (1x1 conv commutes with nearest upsampling: 4x fewer FLOPs, same values)."""

    def __init__(self, in_channels=128, out_channels=None, which_bn=nn.BatchNorm2d, which_conv=nn.Conv2d,
                 upsample_instead=True, which_unpool=nn.ConvTranspose2d, wide=False, with_non_local=False):
        super().__init__()
        self.in_channels = in_channels
        if out_channels is None:
            out_channels = in_channels
        self.out_channels = out_channels
        mid_ch = self.in_channels if wide else self.out_channels
        assert upsample_instead
        main_path = nn.Sequential(
            which_bn(in_channels), nn.ReLU(inplace=False), nn.Upsample(scale_factor=2),
            which_conv(in_channels, mid_ch, 3, 1, padding=1),
            which_bn(mid_ch), nn.ReLU(inplace=False),
            which_conv(mid_ch, out_channels, 3, 1, padding=1))
        identity_map = nn.Upsample(scale_factor=2)
        if in_channels != out_channels:
            identity_map = nn.Sequential(identity_map, which_conv(in_channels, out_channels, 1))
        self.main = ResidualBlock(inner_module=main_path, identity_map=identity_map)
        self.with_non_local = with_non_local
        if with_non_local:
            self.attn = Attention(out_channels)

    def forward_cl(self, x):
        m = self.main.inner_module
        h = ops.bn_relu_up(x, m[0], relu=True, up=2)
        h = ops.conv(h, m[3].weight, m[3].bias)
        h = ops.bn_relu_up(h, m[4], relu=True, up=1)
        if isinstance(self.main.identity_map, nn.Sequential):
            c1 = self.main.identity_map[1]
            skip = ops.upsample2x(ops.conv(x, c1.weight, c1.bias))
        else:
            skip = ops.upsample2x(x)
        out = ops.conv(h, m[6].weight, m[6].bias, residual=skip)
        if self.with_non_local:
            out = self.attn.forward_cl(out)
        return out

    def forward(self, x):
        return _ncl2d(self.forward_cl(_cl2d(x)), self.out_channels)


class DownSample(nn.Module):
    """avg-pool 2 on every dim of extent > 1, pad 1 when odd (layers.py:197-217)."""

    def forward_cl(self, x, residual=None):
        k, s, p = ops.down_sample_cfg(x.shape)
        return ops.avg_pool(x, k, s, p, residual)

    def forward(self, x):
        return ops.from_cl(self.forward_cl(ops.to_cl(x)), x.shape[1])


class DownBlock(nn.Module):
    """ReLU-conv3^3-ReLU-conv3^3-pool + conv1^3-pool (layers.py:219-243).

    B200 schedule: relu -> conv3^3 with ReLU fused in the epilogue -> conv3^3 with the 1^3 skip conv
    added in the epilogue -> ONE pool (avg-pool is linear: pool(a) + pool(b) = pool(a + b))."""

    def __init__(self, in_channels=3, out_channels=None, which_conv=nn.Conv3d, wide=True):
        super().__init__()
        if out_channels is None:
            out_channels = in_channels
        self.out_channels = out_channels
        mid_ch = out_channels if wide else in_channels
        main_path = nn.Sequential(
            nn.ReLU(inplace=False), which_conv(in_channels, mid_ch, kernel_size=3, padding=1),
            nn.ReLU(inplace=False), which_conv(mid_ch, out_channels, kernel_size=3, padding=1),
            DownSample())
        identity_map = nn.Sequential(which_conv(in_channels, out_channels, 1), DownSample())
        self.main = ResidualBlock(inner_module=main_path, identity_map=identity_map)

    def forward_cl(self, x):
        m = self.main.inner_module
        c1 = self.main.identity_map[0]
        # both ReLU backward masks ride in the data-gradient epilogues of their (single) consumers
        h = ops.conv(ops.relu(x, later=True), m[1].weight, m[1].bias, relu=True, x_relu=True, relu_later=True)
        if not ops.fp32_mode() and x.shape[-1] % 64 == 0 and h.shape[-1] % 64 == 0 \
                and tuple(c1.weight.shape[2:]) == (1, 1, 1):
            # the 1^3 skip convolution is extra K of the second convolution's implicit GEMM
            h = ops.conv_skip(h, x, m[3].weight, m[3].bias, c1.weight, c1.bias, h_relu=True)
        else:
            skip = ops.conv(x, c1.weight, c1.bias)
            h = ops.conv(h, m[3].weight, m[3].bias, residual=skip, x_relu=True)
        k, s, p = ops.down_sample_cfg(h.shape)
        return ops.avg_pool(h, k, s, p)

    def forward(self, x):
        return ops.from_cl(self.forward_cl(ops.to_cl(x)), self.out_channels)


class RenderBlock(nn.Module):
    """BN-ReLU-conv3(C->3)-tanh (layers.py:245-259)."""

    def __init__(self, in_channels=128, out_channels=3, which_bn=nn.BatchNorm2d, which_conv=nn.Conv2d):
        super().__init__()
        self.bn = which_bn(in_channels)
        self.activation = nn.ReLU()
        self.conv = which_conv(in_channels, out_channels, kernel_size=3, padding=1)
        self.final = nn.Tanh()
        self.out_channels = out_channels

    def forward_cl(self, x, B, T):
        """x (B*T,1,H,W,C) -> fp32 (B, 3, T, H, W)."""
        h = ops.bn_relu_up(x, self.bn, relu=True, up=1)
        pre = ops.conv(h, self.conv.weight, self.conv.bias)        # Cout 3 padded to 16 (zero rows)
        return ops.render_tail(pre, B, T, self.out_channels)

    def forward(self, x):
        y = self.forward_cl(_cl2d(x), x.shape[0], 1)               # (N,3,1,H,W)
        return y.squeeze(2)


class ConvLSTMCell(nn.Module):
    """Parameter container of one ConvLSTM cell (conv_lstm.py:6-54); the step loop lives in ConvLSTM."""

    def __init__(self, input_channels, hidden_channels, kernel_size):
        super().__init__()
        assert hidden_channels % 2 == 0
        self.input_channels = input_channels
        self.hidden_channels = hidden_channels
        self.kernel_size = kernel_size
        self.num_features = 4
        self.padding = int((kernel_size - 1) / 2)
        c = lambda cin, bias: nn.Conv2d(cin, hidden_channels, kernel_size, 1, self.padding, bias=bias)
        self.Wxi = c(input_channels, True)
        self.Whi = c(hidden_channels, False)
        self.Wxf = c(input_channels, True)
        self.Whf = c(hidden_channels, False)
        self.Wxc = c(input_channels, True)
        self.Whc = c(hidden_channels, False)
        self.Wxo = c(input_channels, True)
        self.Who = c(hidden_channels, False)
        self.Wci = self.Wcf = self.Wco = None       # zero peepholes in the reference (:46-49)

    def stacked(self, plane_is_1x1):
        """[i|f|g|o]-stacked (4H, taps, C) fp32 operands for the fused gate GEMM.  On a 1x1 plane only
        the centre tap of each 3x3 kernel ever multiplies non-padding (SURVEY appendix C)."""
        def w3(conv):
            w = ops.w3_view(conv.weight)
            return w[:, w.shape[1] // 2:w.shape[1] // 2 + 1, :] if plane_is_1x1 else w
        wx = torch.cat([w3(m) for m in (self.Wxi, self.Wxf, self.Wxc, self.Wxo)], dim=0)
        wh = torch.cat([w3(m) for m in (self.Whi, self.Whf, self.Whc, self.Who)], dim=0)
        bx = torch.cat([m.bias for m in (self.Wxi, self.Wxf, self.Wxc, self.Wxo)], dim=0)
        return wx, wh, bx


class ConvLSTM(nn.Module):
    """conv_lstm.py:57-97 for the single-layer configuration TGANv2 uses."""

    def __init__(self, input_channels, hidden_channels, kernel_size, step=1, effective_step=[1]):
        super().__init__()
        self.input_channels = [input_channels] + hidden_channels
        self.hidden_channels = hidden_channels
        self.kernel_size = kernel_size
        self.num_layers = len(hidden_channels)
        assert self.num_layers == 1 and kernel_size == 3, "TGANv2 uses one 3x3 ConvLSTM layer"
        self.step = step
        self.effective_step = effective_step
        self._all_layers = []
        for i in range(self.num_layers):
            cell = ConvLSTMCell(self.input_channels[i], self.hidden_channels[i], self.kernel_size)
            setattr(self, 'cell{}'.format(i), cell)
            self._all_layers.append(cell)

    def forward_cl(self, x):
        """x (B,1,fh,fw,C) -> merged-frame map (B*step, 1, fh, fw, H) in (b, t) order."""
        one = x.shape[2] == 1 and x.shape[3] == 1
        wx, wh, bx = self.cell0.stacked(one)
        # on a 1x1 plane only the centre tap of the eight 3x3 kernels ever receives a gradient (8/9 of the 75.5 M
        # entries stay exactly zero): the data-parallel exchange reduces that tap alone (parallel.reduce_grads)
        for m in (self.cell0.Wxi, self.cell0.Whi, self.cell0.Wxf, self.cell0.Whf, self.cell0.Wxc, self.cell0.Whc,
                  self.cell0.Wxo, self.cell0.Who):
            m.weight._t2v_live_tap = (1, 1) if one else None
        return ops.ConvLstmF.apply(x, wx, wh, bx, self.step)

    def forward(self, input):
        B = input.shape[0]
        out = self.forward_cl(_cl2d(input))
        frames = _ncl2d(out, self.hidden_channels[0]).view((B, self.step) + tuple(input.shape[1:2]) +
                                                           tuple(input.shape[2:]))
        outputs = [frames[:, t] for t in range(self.step) if t in self.effective_step]
        return outputs, (outputs[-1], None)


class Resnet3D(nn.Module):
    """ResNet-3D discriminator trunk + unconditional / conditional heads (resnet3d.py:6-57)."""

    def __init__(self, num_channels=1, mid_ch=64, which_conv=nn.Conv3d, which_pool=nn.AvgPool3d, cond_dim=0,
                 num_down_blocks=4, wide=False, with_attn=True):
        super().__init__()
        self.activation = nn.ReLU(inplace=False)
        res_path = nn.Sequential(which_conv(num_channels, mid_ch, 3, 1, padding=1), self.activation,
                                 which_conv(mid_ch, mid_ch, 3, 1, padding=1), which_pool((1, 2, 2), 2))
        skip_conn = nn.Sequential(which_pool((1, 2, 2), 2), which_conv(num_channels, mid_ch, 1))
        self.res_block = ResidualBlock(inner_module=res_path, identity_map=skip_conn)
        down = []
        in_ch, out_ch = mid_ch, 128
        for i in range(num_down_blocks):
            down.append(DownBlock(in_channels=in_ch, out_channels=out_ch, which_conv=which_conv, wide=wide))
            if i == 0 and with_attn:
                down.append(Attention3d(out_ch, which_conv=which_conv))
            in_ch = out_ch
            out_ch *= 2
        self.down = nn.ModuleList(down)
        self.fc_uncond = nn.Linear(in_ch, 1)
        if cond_dim > 0:
            self.fc = nn.Linear(in_ch + cond_dim, 1)

    def features(self, x):
        """fp32 (B,C,T,H,W) -> fp32 (B, F) sum-pooled trunk features."""
        m = self.res_block.inner_module
        if not ops.fp32_mode() and x.shape[1] == 3 and m[0].weight.shape[0] == 64:
            # RGB padded to 16 channels (skip path) and to 4 channels (stem gather) in one pass;
            # first conv (K = 27*3 = 81): im2col tile gathered into shared memory, tensor-core GEMM, bias + ReLU
            xc, xc4 = ops.rgb_to_cl(x)
            h = ops.stem_conv(x, xc4, m[0].weight, m[0].bias)
        else:
            xc = ops.to_cl(x)                                         # RGB padded to 16 channels (skip path)
            # im2col once in memory, then a 1x1x1 GEMM on the generic engine
            h = ops.conv(ops.im2col3(x), ops.stem_weight_2d(m[0].weight), m[0].bias, relu=True, relu_later=True)
        c1 = self.res_block.identity_map[1]
        pk, ps = (1, 2, 2), (2, 2, 2)                                 # AvgPool3d((1,2,2), 2): stride 2 in ALL dims
        skip = ops.conv(ops.avg_pool(xc, pk, ps), c1.weight, c1.bias)
        if not ops.fp32_mode() and ops.K.conv_sd2_supported(h.shape, h.shape[-1], m[2].weight.shape[0], tuple(m[2].weight.shape[2:])):
            # the pool keeps only the even d planes of this convolution (kernel 1, stride 2 along d): compute only those
            h = ops.conv_sd2(h, m[2].weight, m[2].bias, x_relu=True)
            h = ops.avg_pool(h, pk, (1, 2, 2), residual=skip)
        else:
            h = ops.conv(h, m[2].weight, m[2].bias, x_relu=True)
            h = ops.avg_pool(h, pk, ps, residual=skip)
        for d in self.down:
            h = d.forward_cl(h)
        return ops.sum_spatial(h)

    def heads(self, feat, cond=None):
        """(uncond, cond, feat) from trunk features (resnet3d.py:50-57)"""
        uncond = ops.head_linear(feat, self.fc_uncond.weight, self.fc_uncond.bias)
        if cond is not None:
            c = ops.head_linear(feat, self.fc.weight, self.fc.bias, cond=cond)     # Linear on cat(feat, cond), no cat
            return uncond, c, feat
        return uncond, None, feat

    def forward(self, x=None, cond=None, xbar=None, computed_features=None):
        uncond = None
        if computed_features is not None:
            feat = computed_features
        else:
            feat = self.features(x)
            computed_features = feat
            uncond = ops.head_linear(feat, self.fc_uncond.weight, self.fc_uncond.bias)
        if cond is not None:
            c = ops.head_linear(feat, self.fc.weight, self.fc.bias, cond=cond)
            return uncond, c, computed_features
        return uncond, None, computed_features
