"""Gradient penalty through the TGAN and TCWYT critics (the WGAN-GP recipe of scripts/run_tgan.sh:17: WGAN loss,
gradient penalty lambda = 10): the BatchNorm double-backward kernel, the second-order closure of the critic ops
(general convolution on every route, BatchNorm + activation, LeakyReLU, the fp32 -> storage cast), and whole
direct-drive steps against the fp64 oracle (tests/families_gp_oracle.py; the penalty there is restated from the
reference source, which cannot run it at HEAD).

Gradient bars follow test_families.py: 1e-2 worst tensor for TGAN, 2e-2 for TCWYT (the fp32 oracle itself is that far
from the fp64 one on the near-cancelling WGAN / relativistic gradients, see that module's docstring).
"""
import json
import math
import os

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import bn_double_backward_spec as BNS
import cpu_kernels
import families_gp_oracle as GP
import test_families as TF
from helpers import ROOT, golden, l2rel

LAMBDA = 10.0
GP_SEED = 4321
F64 = torch.float64


@pytest.fixture()
def emulated_fp32(monkeypatch):
    from txt2vid_b200 import ops
    monkeypatch.setattr(ops, "K", cpu_kernels)
    BNS.install(monkeypatch)
    monkeypatch.setattr(ops, "BF16", torch.float32)
    cpu_kernels.set_store_dtype(torch.float32)
    ops.PACKS.clear()
    yield
    cpu_kernels.set_store_dtype(torch.bfloat16)
    ops.PACKS.clear()


@pytest.fixture()
def fp32_mode():
    from txt2vid_b200 import ops
    ops.set_precision("fp32")
    yield
    ops.set_precision("bf16")


# ------------------------------------------------------------------------------------- product direct drive
def _gp(dis, x, fake, cond=None):
    """the product's penalty on a scalar critic, alpha drawn after seeding the CPU generator with GP_SEED"""
    from txt2vid_b200.gan import _gradient_penalty
    torch.manual_seed(GP_SEED)
    return _gradient_penalty(dis, real_x=x, fake_x=fake, real_cond=cond, fake_cond=cond)


def _alpha(B):
    torch.manual_seed(GP_SEED)
    return GP.draw_gp_alpha(B)


def product_tgan_gp_iteration(gen, dis, x, z, gp_lambda=LAMBDA):
    """families_gp_oracle.tgan_iteration on the product modules"""
    from txt2vid_b200.gan import WassersteinGanLoss
    loss = WassersteinGanLoss()
    fake = gen(z)
    d_fake, d_real = dis(x=fake.detach()), dis(x=x)
    gp = _gp(dis, x, fake.detach())
    lossD = loss.discrim_loss(fake=d_fake, real=d_real) + gp_lambda * gp
    lossD.backward()
    gD = TF._grads(dis)
    dis.zero_grad()
    lossG = loss.gen_loss(fake=dis(x=fake), real=None)
    lossG.backward()
    return {"lossD": float(lossD), "lossG": float(lossG), "fake": fake.detach().float().cpu(), "gD": gD,
            "gG": TF._grads(gen), "d_real": float(d_real), "d_fake": float(d_fake), "gp": float(gp)}


def product_tcwyt_gp_iteration(mods, x, z, cond, gp_lambda=LAMBDA):
    """families_gp_oracle.tcwyt_iteration on the product modules"""
    from txt2vid_b200.gan import RaLSGANLoss
    gen, dv, df, dm, fm = mods
    loss = RaLSGANLoss()

    def d_all(vid):
        m = fm.forward_cl(vid)
        return [dv(x=vid, cond=cond), df(x=vid, cond=cond, xbar=m), dm(x=vid, cond=cond, xbar=m)]
    fake = gen(z, cond=cond)
    real_o, fake_o = d_all(x), d_all(fake.detach())
    terms = [loss.discrim_loss(fake=f, real=r) for f, r in zip(fake_o, real_o)]
    gp = _gp(dv, x, fake.detach(), cond)
    terms[0] = terms[0] + gp_lambda * gp
    lossD = sum(terms) / 3
    lossD.backward()
    gD = {"video": TF._grads(dv), "frame": TF._grads(df), "motion": TF._grads(dm), "map": TF._grads(fm)}
    for m in (dv, df, dm, fm):
        m.zero_grad()
    fake_o2 = d_all(fake)
    lossG = sum(loss.gen_loss(fake=f, real=r.detach()) for f, r in zip(fake_o2, real_o)) / 3
    lossG.backward()
    return {"lossD": float(lossD), "lossG": float(lossG), "fake": fake.detach().float().cpu(), "gD": gD,
            "gG": TF._grads(gen), "gp": float(gp)}


def _compare_gp(orc, got, loss_tol, grad_tol, groups, gp_tol=None, **kw):
    """the penalty itself at gp_tol (default loss_tol) relative; then test_families._compare on the losses WITHOUT
    the penalty term (the WGAN ones on the critic scale |D(real)| + |D(fake)|) and on the gradients; the total lossD
    on the scale of its terms."""
    gp_tol = loss_tol if gp_tol is None else gp_tol
    assert abs(got["gp"] - orc["gp"]) <= gp_tol * abs(orc["gp"]), (got["gp"], orc["gp"])
    strip = lambda o: dict(o, lossD=o["lossD"] - LAMBDA * o["gp"] / o.get("gp_div", 1.0))
    worst = TF._compare(strip(orc), strip(got), loss_tol, grad_tol, groups, **kw)
    scale = LAMBDA * abs(orc["gp"]) + (abs(orc["d_real"]) + abs(orc["d_fake"]) if "d_real" in orc else abs(orc["lossD"]))
    assert abs(got["lossD"] - orc["lossD"]) <= max(loss_tol, kw.get("wgan_tol") or 0) * scale, (got["lossD"], orc["lossD"])
    return worst


def _tgan_setup(B):
    fx = golden("tgan_B8.json")
    gen, dis = TF.build_tgan()
    x, z = TF._synth(B, 16, 64, fx["input_seed"]), torch.tensor(fx["z"])[:B]
    return gen, dis, x, z


def _tgan_oracle(gen, dis, x, z, dtype=F64, track_buffers=False):
    import oracle.families_oracle as O
    return GP.tgan_iteration(O.leaves(gen.state_dict(), dtype), O.leaves(dis.state_dict(), dtype), x.to(dtype),
                             z.to(dtype), LAMBDA, _alpha(x.shape[0]), track_buffers=track_buffers)


def _tcwyt_setup():
    fx = golden("tcwyt_B4.json")
    mods = TF.build_tcwyt()
    x, z, cond = TF._synth(fx["B"], 16, 48, fx["input_seed"]), torch.tensor(fx["z"]), torch.tensor(fx["cond"])
    return mods, x, z, cond


def _tcwyt_oracle(mods, x, z, cond, dtype=F64):
    import oracle.families_oracle as O
    sds = [O.leaves(m.state_dict(), dtype) for m in mods]
    o = GP.tcwyt_iteration(*sds, x.to(dtype), z.to(dtype), cond.to(dtype), LAMBDA, _alpha(x.shape[0]))
    o["gp_div"] = 3.0
    return o


def _tcwyt_groups(orc, got):
    return [(n, orc["gD"][n], got["gD"][n]) for n in ("video", "frame", "motion", "map")] + [("G", orc["gG"], got["gG"])]


# ------------------------------------------------------------------------------------- CPU: the kernel spec
def _bn_reference(x, gamma, beta, act):
    C = x.shape[-1]
    xn = x.reshape(-1, C)
    z = F.batch_norm(xn, None, None, gamma, beta, training=True, eps=1e-5)
    return z if act == 0 else (F.relu(z) if act == 1 else F.leaky_relu(z, 0.2))


@pytest.mark.parametrize("act", [0, 1, 2])
@pytest.mark.parametrize("shape,creal", [((6, 1, 1, 1, 24), 24),        # BatchNorm1d
                                         ((3, 1, 5, 4, 16), 16),        # BatchNorm2d
                                         ((2, 3, 4, 5, 32), 32),        # BatchNorm3d
                                         ((2, 2, 3, 3, 32), 20)])       # padded channels (bn_act's padded copies)
@pytest.mark.parametrize("with_gg", [False, True])
def test_bn_backward_backward_spec_matches_autograd(act, shape, creal, with_gg):
    """the spec of bn_backward_backward (bn_double_backward_spec) in fp64 == torch.autograd.grad twice through F.batch_norm + activation"""
    g = torch.Generator().manual_seed(11 + act)
    C = shape[-1]
    x = torch.randn(shape, generator=g, dtype=F64)
    x[..., creal:] = 0                                        # padding channels carry zeros, gamma 1, beta 0
    gamma = torch.rand(C, generator=g, dtype=F64) + 0.5
    beta = torch.randn(C, generator=g, dtype=F64)
    gamma[creal:], beta[creal:] = 1, 0
    dy, ggx = torch.randn(shape, generator=g, dtype=F64), torch.randn(shape, generator=g, dtype=F64)
    ggamma = torch.randn(C, generator=g, dtype=F64) if with_gg else None
    ggbeta = torch.randn(C, generator=g, dtype=F64) if with_gg else None
    xr, gr, dyr = x.clone().requires_grad_(True), gamma.clone().requires_grad_(True), dy.clone().requires_grad_(True)
    betar = beta.clone().requires_grad_(True)
    y = _bn_reference(xr, gr, betar, act)
    dx, dgam, dbet = torch.autograd.grad(y, (xr, gr, betar), dyr.reshape(y.shape), create_graph=True)
    outs, cots = [dx, dgam, dbet], [ggx.reshape(dx.shape), ggamma, ggbeta]
    keep = [i for i, c in enumerate(cots) if c is not None]
    gx, gdy, ggam = torch.autograd.grad([outs[i] for i in keep], (xr, dyr, gr), [cots[i] for i in keep])
    mean = x.reshape(-1, C).mean(0)
    invstd = torch.rsqrt(x.reshape(-1, C).var(0, unbiased=False) + 1e-5)
    cpu_kernels.set_store_dtype(F64)
    try:
        sx, sdy, sgam = BNS.bn_backward_backward(dy, x, torch.cat((mean, invstd)),
                                                         torch.cat((gamma * invstd, beta - mean * gamma * invstd)),
                                                         ggx, ggamma, ggbeta, act, 1)
    finally:
        cpu_kernels.set_store_dtype(torch.bfloat16)
    assert sx.dtype == F64 and sx.shape == x.shape
    for mine, ref in ((sx, gx), (sdy, gdy), (sgam, ggam)):
        assert float((mine.reshape(-1) - ref.reshape(-1)).norm()) <= 1e-10 * max(float(ref.norm()), 1.0)


def test_bn_backward_backward_rejects_upsampling_and_odd_channels():
    """T2V_ERR_ARG before any CUDA call: up = 2, C % 8 != 0"""
    from txt2vid_b200 import _lib
    lib = _lib.lib()
    ERR_ARG = -1                                      # T2V_ERR_ARG of include/t2v.h
    for sfx in ("", "_f32"):
        fn = getattr(lib, "t2v_bn_bwd_bwd" + sfx)
        assert fn(None, None, None, None, None, None, None, None, None, None, None, 5, 16, 0, 2, None) == ERR_ARG
        assert fn(None, None, None, None, None, None, None, None, None, None, None, 5, 12, 0, 1, None) == ERR_ARG


# ------------------------------------------------------------------------------------- CPU: autograd formulas
def test_tgan_wgan_gp_step_cpu(emulated_fp32):
    """WGAN-GP (lambda = 10) direct-drive TGAN step at B = 4, product ops on the CPU spec (fp32 storage), against the
    fp64 oracle"""
    gen, dis, x, z = _tgan_setup(4)
    orc = _tgan_oracle(gen, dis, x, z)
    got = product_tgan_gp_iteration(gen, dis, x, z)
    _compare_gp(orc, got, 1e-3, 1e-2, [("D", orc["gD"], got["gD"]), ("G", orc["gG"], got["gG"])])


def test_tcwyt_video_gp_step_cpu(emulated_fp32):
    """conditional TCWYT step (video critic with the penalty, frame / motion critics without) at B = 4 on the CPU
    spec against the fp64 oracle"""
    mods, x, z, cond = _tcwyt_setup()
    orc = _tcwyt_oracle(mods, x, z, cond)
    got = product_tcwyt_gp_iteration(mods, x, z, cond)
    got["gp_div"] = 3.0
    _compare_gp(orc, got, 1e-3, 2e-2, _tcwyt_groups(orc, got))


def test_gradient_penalty_of_tuple_critic_unchanged(emulated_fp32):
    """a critic returning (uncond, cond, features) is penalised as before scalar critics were accepted: d(u + c)/dx_hat,
    mean_b (||g_b|| - 1)^2 (and the zero-centred sum)"""
    from txt2vid_b200.gan import _gradient_penalty

    class TupleCritic(nn.Module):
        def __init__(self):
            super().__init__()
            self.w = nn.Parameter(torch.randn(3 * 4 * 5 * 5, generator=torch.Generator().manual_seed(3)))
            self.v = nn.Parameter(torch.randn(8, generator=torch.Generator().manual_seed(4)))

        def forward(self, x=None, cond=None, xbar=None):
            h = torch.tanh(x.reshape(x.shape[0], -1) * self.w)
            u = (h ** 2).sum(1)
            c = None if cond is None else (h.sum(1, keepdim=True) * cond * self.v).sum(1)
            return u, c, h

    g = torch.Generator().manual_seed(5)
    real, fake = torch.randn(3, 3, 4, 5, 5, generator=g), torch.randn(3, 3, 4, 5, 5, generator=g)
    rc, fc = torch.randn(3, 8, generator=g), torch.randn(3, 8, generator=g)
    D = TupleCritic()
    for cond in (False, True):
        for zero_center, combine in ((False, torch.mean), (True, torch.sum)):
            torch.manual_seed(9)
            got = _gradient_penalty(D, real_x=real, fake_x=fake, real_cond=rc if cond else None,
                                    fake_cond=fc if cond else None, zero_center=zero_center, combine=combine)
            torch.manual_seed(9)
            a = torch.rand(3)
            xh = (a.view(-1, 1, 1, 1, 1) * real + (1 - a.view(-1, 1, 1, 1, 1)) * fake).requires_grad_(True)
            ch = (a.view(-1, 1) * rc + (1 - a.view(-1, 1)) * fc).requires_grad_(True) if cond else None
            u, c, _ = D(x=xh, cond=ch)
            outs = [u] + ([c] if cond else [])
            gr = torch.autograd.grad(outs, [xh] + ([ch] if cond else []), [torch.ones_like(o) for o in outs])[0]
            n2 = gr.reshape(3, -1).pow(2).sum(1)
            want = combine(n2) if zero_center else combine((n2.sqrt() - 1) ** 2)
            assert abs(float(got) - float(want)) <= 1e-6 * abs(float(want)), (cond, zero_center, float(got), float(want))


# ------------------------------------------------------------------------------------- GPU: the kernel
_BN_CASES = [(C, P) for C in (16, 64, 128, 368, 512) for P in (300, 20000, 262144)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("C,P", _BN_CASES)
def test_bn_bwd_bwd_kernel_vs_spec(C, P, dtype):
    """t2v_bn_bwd_bwd[_f32] against the spec evaluated in fp64 on the same (storage-rounded) inputs: 1e-5 rel L2 in
    fp32 storage, 1e-2 in bf16 (its outputs are rounded to bf16); activation and the optional ggamma / ggbeta vary
    with the case"""
    from txt2vid_b200 import kernels
    i = _BN_CASES.index((C, P))
    act, with_gg = i % 3, i % 2 == 0
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(100 + i)
    x = (torch.randn(P, 1, 1, 1, C, device=dev, generator=g) * 2 + 0.3).to(dtype)
    dy = torch.randn(P, 1, 1, 1, C, device=dev, generator=g).to(dtype)
    ggx = torch.randn(P, 1, 1, 1, C, device=dev, generator=g).to(dtype)
    gamma = torch.rand(C, device=dev, generator=g) + 0.5
    beta = torch.randn(C, device=dev, generator=g) * 0.5
    ggamma = torch.randn(C, device=dev, generator=g) if with_gg else None
    ggbeta = torch.randn(C, device=dev, generator=g) if with_gg else None
    _, mean_invstd, scale_shift = kernels.bn_forward(x, gamma, beta, torch.zeros(C, device=dev),
                                                     torch.ones(C, device=dev), act, 1)
    gx, gdy, dgamma = kernels.bn_backward_backward(dy, x, mean_invstd, scale_shift, ggx, ggamma, ggbeta, act, 1)
    cpu_kernels.set_store_dtype(F64)
    try:
        d = lambda t: None if t is None else t.double()
        rx, rdy, rgam = BNS.bn_backward_backward(d(dy), d(x), d(mean_invstd), d(scale_shift), d(ggx),
                                                         d(ggamma), d(ggbeta), act, 1)
    finally:
        cpu_kernels.set_store_dtype(torch.bfloat16)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    for name, mine, ref in (("gx", gx, rx), ("gdy", gdy, rdy), ("dgamma", dgamma, rgam)):
        err = float((mine.double() - ref).norm() / ref.norm())
        assert err <= tol, (name, C, P, dtype, act, err)


# ------------------------------------------------------------------------------------- GPU: op-level second order
def _cl(t5, Cp):
    """(N,C,D,H,W) fp64 -> CL (N,D,H,W,Cp) with zero channel padding"""
    out = torch.zeros(t5.shape[0], *t5.shape[2:], Cp, dtype=t5.dtype, device=t5.device)
    out[..., :t5.shape[1]] = t5.permute(0, 2, 3, 4, 1)
    return out


def _second_order(fn, x, v, u, wrt):
    """gradients of <(dy/dx)^T v, u> w.r.t. the tensors in wrt (None where the graph does not reach)"""
    y = fn(x)
    (gx,) = torch.autograd.grad(y, x, v, create_graph=True)
    L = (gx.to(u.dtype) * u).sum()
    return torch.autograd.grad(L, wrt, allow_unused=True)


def _err(mine, ref, C=None):
    if ref is None or float(ref.norm()) == 0:
        return 0.0 if mine is None else float(mine.float().norm())
    m = mine.double().cpu()
    if C is not None:
        m = m[..., :C]
    return float((m.reshape(-1) - ref.reshape(-1)).norm() / ref.norm())


# (label, conv dims, Cin, Cout, kernel, stride, padding, input spatial (D,H,W), out_f32)
_GCONV_ROUTES = [
    ("s2d3d_rgb", 3, 3, 64, 4, 2, 1, (8, 16, 16), False),          # shifted space-to-depth, 3-D, RGB (cin_real 3)
    ("s2d3d", 3, 64, 128, 4, 2, 1, (4, 8, 8), False),
    ("s2d2d", 2, 64, 128, 4, 2, 1, (1, 8, 8), False),              # 2-D (FrameMap)
    ("s2d2d_rgb", 2, 3, 64, 4, 2, 1, (1, 16, 16), False),
    ("same", 3, 512 + 256, 512, 1, 1, 0, (1, 3, 3), False),        # 1x1x1 (TCWYT pred[0])
    ("full", 3, 512, 1, (1, 3, 3), 1, 0, (1, 3, 3), True),         # TCWYT pred[3]: out_f32, the critic's last layer
    ("window", 3, 512, 1, (1, 3, 3), 2, 0, (1, 4, 4), True),       # TGAN pred: one output reading a corner window
    ("cudacore", 3, 32, 48, 3, 2, 1, (5, 6, 6), False),            # no engine route: CUDA-core kernels
]


def _gconv_case(label, nd, cin, cout, k, s, p, sp, out_f32, tc=True):
    from txt2vid_b200 import kernels, ops
    torch.manual_seed(31)
    conv = (nn.Conv3d if nd == 3 else nn.Conv2d)(cin, cout, k, s, p, bias=False)
    conv = conv.cuda()
    N, Cp = 2, ops.round16(cin)
    x5 = torch.randn(N, cin, *sp, dtype=F64)
    st = kernels.STORE
    x = _cl(x5, Cp).to(st).cuda().requires_grad_(True)
    x5 = x.detach()[..., :cin].double().cpu().permute(0, 4, 1, 2, 3)            # the storage-rounded input
    w5 = conv.weight.detach().double().cpu()
    if nd == 2:
        w5 = w5.unsqueeze(2)
    kk, ss, pp = ops.conv_args(conv)
    y_ref = F.conv3d(x5, w5, None, ss, pp)
    v5 = torch.randn(y_ref.shape, dtype=F64)
    v = _cl(v5, ops.round16(cout)).to(torch.float32 if (out_f32 or st == torch.float32) else st).cuda()
    v5 = v.detach()[..., :cout].double().cpu().permute(0, 4, 1, 2, 3)
    u5 = torch.randn(x5.shape, dtype=F64)
    u = _cl(u5, Cp).to(st).cuda()
    u5 = u[..., :cin].double().cpu().permute(0, 4, 1, 2, 3)
    v.requires_grad_(True)
    old = kernels.GCONV_TC
    kernels.GCONV_TC = tc
    try:
        gv, gw = _second_order(lambda t: ops.gconv(t, conv, out_f32=out_f32), x, v, u.float() if u.dtype != st else u,
                               (v, conv.weight))
    finally:
        kernels.GCONV_TC = old
    x5r, v5r, w5r = x5.clone().requires_grad_(True), v5.clone().requires_grad_(True), w5.clone().requires_grad_(True)
    r = _second_order(lambda t: F.conv3d(t, w5r, None, ss, pp), x5r, v5r, u5, (v5r, w5r))
    rv = r[0].permute(0, 2, 3, 4, 1)
    rw = r[1].squeeze(2) if nd == 2 else r[1]
    return _err(gv, rv, cout), _err(gw.detach().cpu(), rw)


def _bar():
    from txt2vid_b200 import ops
    return 1e-4 if ops.fp32_mode() else 2e-2


def _check_gconv(case, tc=True):
    ev, ew = _gconv_case(*case, tc=tc)
    print("%s tc=%s: d/dv %.2e d/dw %.2e" % (case[0], tc, ev, ew))
    assert ev <= _bar() and ew <= _bar(), (case[0], ev, ew)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _GCONV_ROUTES, ids=[c[0] for c in _GCONV_ROUTES])
def test_gconv_second_order_bf16(case):
    _check_gconv(case)


@pytest.mark.gpu
def test_gconv_second_order_bf16_cudacore_fallback():
    """every general convolution on the CUDA-core kernels (kernels.GCONV_TC off)"""
    for case in _GCONV_ROUTES:
        _check_gconv(case, tc=False)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _GCONV_ROUTES, ids=[c[0] for c in _GCONV_ROUTES])
def test_gconv_second_order_fp32(case, fp32_mode):
    _check_gconv(case)


def _bn_case(shape, creal, act, xdtype):
    from txt2vid_b200 import ops
    torch.manual_seed(41 + act)
    C = shape[-1]
    bn = nn.BatchNorm1d(creal).cuda()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.normal_(0, 0.5)
    x64 = torch.randn(shape, dtype=F64) * 1.5 + 0.2
    x64[..., creal:] = 0
    x = x64.to(xdtype).cuda().requires_grad_(True)
    x64 = x.detach().double().cpu()
    v = torch.randn(shape, dtype=F64).to(xdtype).cuda()
    v64 = v.double().cpu()
    v.requires_grad_(True)
    u = torch.randn(shape, dtype=F64).to(xdtype).cuda()
    u64 = u.double().cpu()
    gx, gv, gg = _second_order(lambda t: ops.bn_act(t, bn, act), x, v, u, (x, v, bn.weight))
    xr = x64[..., :creal].reshape(-1, creal).clone().requires_grad_(True)
    vr = v64[..., :creal].reshape(-1, creal).clone().requires_grad_(True)
    gr = bn.weight.detach().double().cpu().requires_grad_(True)
    br = bn.bias.detach().double().cpu()
    rx, rv, rg = _second_order(lambda t: _bn_reference(t, gr, br, act), xr, vr, u64[..., :creal].reshape(-1, creal),
                               (xr, vr, gr))
    to = lambda t: t.reshape(*shape[:-1], creal)
    return _err(gx.detach().cpu(), to(rx), creal), _err(gv.detach().cpu(), to(rv), creal), _err(gg.detach().cpu(), rg)


_BN_OP_CASES = [((8, 1, 1, 1, 256), 256), ((4, 2, 6, 6, 64), 64), ((4, 1, 1, 1, 368), 356), ((4, 2, 3, 3, 32), 20)]


def _check_bn(xdtype):
    for shape, creal in _BN_OP_CASES:
        for act in (0, 1, 2):
            e = _bn_case(shape, creal, act, xdtype)
            print("bn %s act %d %s: d/dx %.2e d/dv %.2e d/dgamma %.2e" % (shape, act, xdtype, *e))
            assert max(e) <= _bar(), (shape, creal, act, xdtype, e)


@pytest.mark.gpu
def test_bn_act_second_order_bf16():
    """BatchNorm + activation in bf16 mode: fp32 input (behind a convolution's fp32 accumulator, conv_bn_act) and
    bf16 input (the caption path's BatchNorm1d)"""
    _check_bn(torch.float32)
    _check_bn(torch.bfloat16)


@pytest.mark.gpu
def test_bn_act_second_order_fp32(fp32_mode):
    _check_bn(torch.float32)


def _pointwise_case(fn, ref_fn, xdtype, vdtype):
    torch.manual_seed(51)
    shape = (4, 2, 5, 5, 32)
    x = torch.randn(shape, dtype=F64).to(xdtype).cuda().requires_grad_(True)
    v = torch.randn(shape, dtype=F64).to(vdtype).cuda()
    u = torch.randn(shape, dtype=F64).to(xdtype).cuda()
    x64, v64, u64 = x.detach().double().cpu(), v.double().cpu(), u.double().cpu()
    v.requires_grad_(True)
    gx, gv = _second_order(fn, x, v, u, (x, v))
    xr, vr = x64.clone().requires_grad_(True), v64.clone().requires_grad_(True)
    rx, rv = _second_order(ref_fn, xr, vr, u64, (xr, vr))
    assert gx is None or float(gx.float().norm()) == 0           # both ops are piecewise linear in x
    return _err(gv.detach().cpu(), rv)


def _check_pointwise():
    from txt2vid_b200 import kernels, ops
    st = kernels.STORE
    e = _pointwise_case(lambda t: ops.leaky_relu(t, 0.2), lambda t: F.leaky_relu(t, 0.2), st, st)
    print("leaky_relu: d/dv %.2e" % e)
    assert e <= _bar(), e
    e = _pointwise_case(ops.CastStoreF.apply, lambda t: t, torch.float32, st)
    print("cast to storage: d/dv %.2e" % e)
    assert e <= _bar(), e


@pytest.mark.gpu
def test_leaky_and_cast_second_order_bf16():
    _check_pointwise()


@pytest.mark.gpu
def test_leaky_and_cast_second_order_fp32(fp32_mode):
    _check_pointwise()


# ------------------------------------------------------------------------------------- GPU: whole steps
def _floor_gp(family):
    """measured bf16 floor of the WGAN-GP step (scripts/bf16_floor_families.py --gp ->
    profiles/r03_bf16_floor_families_gp.json)"""
    with open(os.path.join(ROOT, "profiles", "r03_bf16_floor_families_gp.json")) as f:
        for line in f:
            if line.strip() and json.loads(line)["family"] == family:
                return json.loads(line)
    raise KeyError(family)


def _buffers(module):
    return {k: v.detach().float().cpu() for k, v in module.state_dict().items() if "running_" in k}


@pytest.mark.gpu
def test_tgan_wgan_gp_step_gpu_fp32_mode(fp32_mode):
    """B = 8, lambda = 10 on the B200 in fp32 storage against the fp64 oracle: 1e-3 on the losses and the penalty,
    1e-2 worst gradient tensor, and the BatchNorm running statistics after the step"""
    gen, dis, x, z = _tgan_setup(8)
    orc = _tgan_oracle(gen, dis, x, z, track_buffers=True)
    got = product_tgan_gp_iteration(gen.cuda(), dis.cuda(), x.cuda(), z.cuda())
    for k in ("lossG", "d_real", "d_fake", "gp"):
        assert abs(got[k] - orc[k]) <= 1e-3 * abs(orc[k]), (k, got[k], orc[k])
    worst = _compare_gp(orc, got, 1e-3, 1e-2, [("D", orc["gD"], got["gD"]), ("G", orc["gG"], got["gG"])], wgan_tol=1e-3)
    for name, mod, ref in (("D", dis, orc["buffers_D"]), ("G", gen, orc["buffers_G"])):
        mine = _buffers(mod)
        assert set(mine) == set(ref), name
        for k in ref:
            assert l2rel(mine[k], ref[k].float()) <= 1e-3, (name, k, l2rel(mine[k], ref[k].float()))
    print("tgan gp fp32 mode: lossD %.6f (oracle %.6f) gp %.6f (oracle %.6f) worst grad L2 %s"
          % (got["lossD"], orc["lossD"], got["gp"], orc["gp"], worst))


@pytest.mark.gpu
def test_tgan_wgan_gp_step_gpu_bf16():
    """B = 8, lambda = 10 in bf16 storage: 1.5x the measured bf16 floor of the same step"""
    fl = _floor_gp("tgan_B8_gp")
    gen, dis, x, z = _tgan_setup(8)
    orc = _tgan_oracle(gen, dis, x, z, dtype=torch.float32)
    got = product_tgan_gp_iteration(gen.cuda(), dis.cuda(), x.cuda(), z.cuda())
    wgan_tol = 1.5 * max(fl["lossD_over_critic_scale"], fl["lossG_over_critic_scale"])
    worst = _compare_gp(orc, got, 2e-2, {"D": 1.5 * fl["gradD_worst"], "G": 1.5 * fl["gradG_worst"]},
                        [("D", orc["gD"], got["gD"]), ("G", orc["gG"], got["gG"])], gp_tol=max(2e-2, 1.5 * fl["gp_rel"]),
                        wgan_tol=wgan_tol, fake_tol=max(2e-2, 1.5 * fl["fake"]))
    print("tgan gp bf16: gp %.5f (oracle %.5f) lossD %.5f (oracle %.5f) worst grad L2 %s"
          % (got["gp"], orc["gp"], got["lossD"], orc["lossD"], worst))


@pytest.mark.gpu
def test_tcwyt_video_gp_step_gpu_fp32_mode(fp32_mode):
    mods, x, z, cond = _tcwyt_setup()
    orc = _tcwyt_oracle(mods, x, z, cond)
    got = product_tcwyt_gp_iteration([m.cuda() for m in mods], x.cuda(), z.cuda(), cond.cuda())
    got["gp_div"] = 3.0
    worst = _compare_gp(orc, got, 1e-3, 2e-2, _tcwyt_groups(orc, got))
    print("tcwyt gp fp32 mode: lossD %.6f (oracle %.6f) gp %.6f (oracle %.6f) worst grad L2 %s"
          % (got["lossD"], orc["lossD"], got["gp"], orc["gp"], worst))


@pytest.mark.gpu
def test_tgan_wgan_gp_five_critic_steps_then_generator_bf16():
    """the recipe's schedule (5 critic steps per generator step) with FusedAdam in bf16: finite losses, and every
    critic parameter moves"""
    from txt2vid_b200.gan import WassersteinGanLoss
    from txt2vid_b200.optim import FusedAdam
    gen, dis, x, z = _tgan_setup(8)
    gen, dis, x, z = gen.cuda(), dis.cuda(), x.cuda(), z.cuda()
    optD = FusedAdam(dis.parameters(), lr=1e-4, betas=(0.0, 0.9))
    optG = FusedAdam(gen.parameters(), lr=1e-4, betas=(0.0, 0.9))
    loss = WassersteinGanLoss()
    before = {k: p.detach().clone() for k, p in dis.named_parameters()}
    for _ in range(5):
        dis.zero_grad()
        with torch.no_grad():
            fake = gen(z)
        lossD = loss.discrim_loss(fake=dis(x=fake), real=dis(x=x)) + LAMBDA * _gp(dis, x, fake)
        lossD.backward()
        optD.step()
        assert math.isfinite(float(lossD))
    gen.zero_grad()
    lossG = loss.gen_loss(fake=dis(x=gen(z)), real=None)
    lossG.backward()
    optG.step()
    assert math.isfinite(float(lossG))
    for k, p in dis.named_parameters():
        assert not torch.equal(p.detach(), before[k]), k
