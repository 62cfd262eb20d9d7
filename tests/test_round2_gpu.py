"""GPU (round 2): the kernels that replaced the last library calls, checked against the ORACLE's functions
(oracle/txt2vid_oracle.py: the restatement of the reference pinned to the live reference), and the fp32 storage mode
of the whole engine at BASELINE north_star's fp32 bar (1e-3).

  * fp32 storage twins of the HBM-bound kernels vs their executable spec, and the fp32 convolution engine (exact fp32
    FMAs on the CUDA cores) vs F.conv3d in fp64;
  * non-local block (Attention3d with gamma != 0) forward, backward AND double backward vs oracle attention3d;
  * caption encoder (Embedding + 4-layer length-masked Bi-LSTM) forward / backward vs oracle seq2seq_encode;
  * discriminator heads + fused relativistic loss vs the oracle's per-level composition;
  * ConvLSTM vs oracle conv_lstm;
  * Adam kernel vs the oracle's Adam over three steps.
Every test runs in both precision modes with its own bar."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import cpu_kernels as C
from helpers import l2rel

pytestmark = pytest.mark.gpu
BF, F32 = torch.bfloat16, torch.float32
TOL = {"fp32": 1e-3, "bf16": 2e-2}


@pytest.fixture(params=["fp32", "bf16"])
def precision(request):
    from txt2vid_b200 import ops
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ops.set_precision(request.param)
    C.set_store_dtype(F32 if request.param == "fp32" else BF)
    yield request.param
    ops.set_precision("bf16")
    C.set_store_dtype(BF)


def K():
    from txt2vid_b200 import kernels
    return kernels


def rel(a, b):
    return l2rel(a.float(), b.float())


# ------------------------------------------------------------------------------------- fp32 storage twins
def test_fp32_storage_kernels_match_spec(precision):
    """the typed HBM-bound kernels in both storage types against tests/cpu_kernels.py on the same tensors"""
    dt = F32 if precision == "fp32" else BF
    tol = 2e-6 if precision == "fp32" else 1e-2
    g = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g).to(dt)
    x, dy = r(3, 2, 6, 8, 32), r(3, 2, 6, 8, 32)
    assert torch.equal(K().relu_fwd(x), C.relu_fwd(x)) and torch.equal(K().relu_bwd(dy, x), C.relu_bwd(dy, x))
    assert rel(K().leaky_relu_fwd(x, 0.2), C.leaky_relu_fwd(x, 0.2)) < tol
    assert rel(K().tanh_fwd(x), C.tanh_fwd(x)) < tol
    k, s, p = (2, 2, 2), (2, 2, 2), (0, 0, 0)
    y = K().avgpool_fwd(x, k, s, p)
    assert y.dtype == dt and rel(y, C.avgpool_fwd(x, k, s, p)) < tol
    assert rel(K().avgpool_bwd(y, x.shape, k, s, p), C.avgpool_bwd(y, x.shape, k, s, p)) < tol
    x2 = r(5, 1, 4, 6, 64)
    assert torch.equal(K().upsample2x_fwd(x2), C.upsample2x_fwd(x2))
    dy2 = r(5, 1, 8, 12, 64)
    assert rel(K().upsample2x_bwd(dy2), C.upsample2x_bwd(dy2)) < tol
    xf = torch.randn(2, 3, 4, 8, 8, device="cuda", generator=g)
    cl = K().nchw_to_cl(xf, 16)
    assert cl.dtype == dt and rel(K().cl_to_nchw(cl, 3), xf) < (1e-7 if precision == "fp32" else 5e-3)
    assert rel(K().sum_rows(x), C.sum_rows(x)) < 1e-4 and rel(K().sum_spatial(x), C.sum_spatial(x)) < 1e-4
    gamma, beta = torch.rand(64, device="cuda") + 0.5, torch.randn(64, device="cuda")
    for up, act in ((1, 1), (2, 1), (1, 0)):
        rm, rv = torch.zeros(64, device="cuda"), torch.ones(64, device="cuda")
        rm2, rv2 = rm.clone(), rv.clone()
        yk, mi, ss = K().bn_forward(x2, gamma, beta, rm, rv, act, up)
        yc, mic, ssc = C.bn_forward(x2, gamma, beta, rm2, rv2, act, up)
        assert rel(yk, yc) < max(tol, 2e-5) and rel(rm, rm2) < 1e-5 and rel(rv, rv2) < 1e-4
        dyy = r(*yk.shape)
        dk, dc_ = K().bn_backward(dyy, x2, mi, ss, act, up), C.bn_backward(dyy, x2, mic, ssc, act, up)
        for a, b in zip(dk, dc_):
            assert rel(a, b) < max(tol, 1e-4), (up, act, rel(a, b))
    sc = torch.tensor([0.37], device="cuda")
    assert rel(K().scale(x, sc), C.scale(x, sc)) < tol and rel(K().scale_add(x, dy, sc), C.scale_add(x, dy, sc)) < tol
    assert abs(float(K().dot(x, dy)) - float(C.dot(x, dy))) < 1e-3 * float(x.float().norm() * dy.float().norm())
    sl = K().cl_slice_f32(x, 20)
    assert torch.equal(sl, x[..., :20].float())
    assert torch.equal(K().f32_pad_cl(sl, 32, dt)[..., :20].float(), sl.to(dt).float())


@pytest.mark.parametrize("Cc", [48, 368])
def test_fp32_batchnorm_statistics_are_bit_reproducible(Cc):
    """fp32 storage: BatchNorm statistics are reduced in a fixed order for every channel count, so two runs on the same
    input agree bit for bit (C = 48: C/8 does not divide 256; C = 368: a narrower second 256-channel slab)"""
    x = torch.randn(20000, 1, 1, 1, Cc, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)) + 0.5
    gamma, beta = torch.rand(Cc, device="cuda") + 0.5, torch.randn(Cc, device="cuda")
    runs = []
    for _ in range(2):
        rm, rv = torch.zeros(Cc, device="cuda"), torch.ones(Cc, device="cuda")
        y, mi, ss = K().bn_forward(x, gamma, beta, rm, rv, 1, 1)
        runs.append((y, mi, ss, rm, rv))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("epilogue", ["residual", "relu"])
@pytest.mark.parametrize("geom", [((4, 1, 8, 8), 64, 64, (1, 3, 3)), ((2, 4, 4, 4), 128, 64, (3, 3, 3)),
                                  ((16, 1, 1, 1), 256, 512, (1, 1, 1)), ((2, 2, 8, 8), 16, 32, (3, 3, 3)),
                                  ((3, 1, 4, 4), 1024, 256, (1, 3, 3))])
def test_conv_engine_fp32_mode(geom, epilogue):
    """The convolution engine of the fp32 storage mode against F.conv3d in fp64 (TF32 off): fp32 operands, exact fp32
    FMAs on the CUDA cores, a few 1e-7 -- what the 1e-3 gradient bar needs -- fprop (epilogue bias + residual, or
    bias + ReLU) / dgrad / wgrad."""
    from txt2vid_b200 import ops
    (N, D, H, W), Cin, Cout, k = geom
    tol = 3e-6
    ops.set_precision("fp32")
    torch.backends.cudnn.allow_tf32 = False
    try:
        g = torch.Generator(device="cuda").manual_seed(1)
        x = torch.randn(N, D, H, W, Cin, device="cuda", generator=g)
        w = torch.randn(Cout, k[0] * k[1] * k[2], Cin, device="cuda", generator=g) * 0.1
        bias = torch.randn(Cout, device="cuda", generator=g)
        res = torch.randn(N, D, H, W, Cout, device="cuda", generator=g)
        w5 = w.view(Cout, k[0], k[1], k[2], Cin).permute(0, 4, 1, 2, 3).contiguous()
        pad = tuple(kk // 2 for kk in k)
        # fp64 reference (cuDNN's own fp32 kernels sit ~1e-6 from it on the K = 9216 case)
        ref = F.conv3d(x.permute(0, 4, 1, 2, 3).double(), w5.double(), bias.double(), padding=pad).permute(0, 2, 3, 4, 1)
        if epilogue == "residual":
            ref = ref + res
            y = K().conv_fprop(x, K().pack_weight(w), bias, res, k)
        else:
            ref = ref.clamp_min(0)
            y = K().conv_fprop(x, K().pack_weight(w), bias, None, k, relu=True)
        assert y.dtype == F32 and rel(y, ref) < tol, rel(y, ref)
        dy = torch.randn(N, D, H, W, Cout, device="cuda", generator=g)
        xr = x.permute(0, 4, 1, 2, 3).detach().double().requires_grad_(True)
        wr = w5.detach().double().requires_grad_(True)
        F.conv3d(xr, wr, None, padding=pad).backward(dy.permute(0, 4, 1, 2, 3).double())
        dx = K().conv_dgrad(dy, K().pack_dgrad_weight(w), k)
        assert rel(dx, xr.grad.permute(0, 2, 3, 4, 1)) < tol
        dw = K().conv_wgrad(dy, x, k)
        assert rel(dw, wr.grad.permute(0, 2, 3, 4, 1).reshape(Cout, -1, Cin)) < tol
        # fused ReLU mask of the data gradient with an fp32 reference
        dxm = K().conv_dgrad(dy, K().pack_dgrad_weight(w), k, relu_ref=x)
        assert rel(dxm, xr.grad.permute(0, 2, 3, 4, 1) * (x > 0)) < tol
    finally:
        ops.set_precision("bf16")


# ------------------------------------------------------------------------------------- non-local block
@pytest.mark.parametrize("shape", [(3, 2, 8, 8), (2, 1, 16, 16), (4, 4, 2, 2)])
def test_attention3d_vs_oracle_with_double_backward(precision, shape):
    """blocks.Attention3d (gamma = 0.7) vs oracle attention3d (models/layers.py:52-68): output, first-order gradients
    and the gradients of a gradient-penalty-like second-order loss."""
    import oracle.txt2vid_oracle as O
    from txt2vid_b200.blocks import Attention3d
    N, D, H, W = shape
    ch = 128
    torch.manual_seed(3)
    blk = Attention3d(ch)
    with torch.no_grad():
        for p_ in blk.parameters():
            if p_.dim() > 1:
                p_.normal_(0, 0.08)
        blk.gamma.fill_(0.7)
    x = torch.randn(N, ch, D, H, W)
    r = torch.randn(N, ch, D, H, W)
    sd = {"a." + k: v.detach().clone().requires_grad_(True) for k, v in blk.state_dict().items()}

    def second_order(fn, params, xin):
        xin = xin.detach().requires_grad_(True)
        y = fn(xin)
        gx, = torch.autograd.grad((y * r.to(y.device)).sum(), xin, create_graph=True)
        loss = (gx ** 2).sum() + y.square().mean()
        grads = torch.autograd.grad(loss, params)
        return y.detach(), gx.detach(), grads

    names = [k for k in sd]
    y_o, gx_o, g_o = second_order(lambda t: O.attention3d(t, sd, "a"), [sd[k] for k in names], x)
    blk = blk.cuda()
    pm = dict(blk.named_parameters())
    y_p, gx_p, g_p = second_order(lambda t: blk(t), [pm[k[2:]] for k in names], x.cuda())
    tol = TOL[precision]
    bars = {"y": tol, "gx": 1.5 * tol}
    bars.update({n: 3 * tol for n in names})
    if precision == "bf16":
        # what bf16 itself costs on this second-order quantity: the ORACLE under torch.autocast(bfloat16) (library
        # kernels, fp32 accumulation) against the same oracle in fp32; the bar is 1.5x that floor where the floor
        # exceeds the nominal bar (VERDICT r1 item 2b)
        sd_c = {k: v.detach().cuda().requires_grad_(True) for k, v in sd.items()}

        def autocast_fn(t):
            with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
                return O.attention3d(t, sd_c, "a").float()
        y_a, gx_a, g_a = second_order(autocast_fn, [sd_c[k] for k in names], x.cuda())
        floor = {"y": rel(y_a.cpu(), y_o), "gx": rel(gx_a.cpu(), gx_o)}
        floor.update({n: rel(a.cpu(), b) for n, a, b in zip(names, g_a, g_o)})
        print("autocast floor:", {k: "%.3g" % v for k, v in floor.items()})
        bars = {k: max(v, 1.5 * floor[k]) for k, v in bars.items()}
    errs = {"y": rel(y_p.cpu(), y_o), "gx": rel(gx_p.cpu(), gx_o)}
    errs.update({n: rel(a.cpu(), b) for n, a, b in zip(names, g_p, g_o)})
    print("product:", {k: "%.3g" % v for k, v in errs.items()})
    for k, e in errs.items():
        assert e < bars[k], (k, e, bars[k])


def test_generator_attention_vs_oracle(precision):
    """blocks.Attention (2-D, gamma = 0.7: the fused core kernels in bf16, the primitives in fp32) vs oracle attention2d"""
    import oracle.txt2vid_oracle as O
    from txt2vid_b200.blocks import Attention
    torch.manual_seed(4)
    blk = Attention(32)
    with torch.no_grad():
        for p_ in blk.parameters():
            if p_.dim() > 1:
                p_.normal_(0, 0.2)
        blk.gamma.fill_(0.7)
    x = torch.randn(6, 32, 32, 32)
    sd = {"a." + k: v.detach().clone().requires_grad_(True) for k, v in blk.state_dict().items()}
    xo = x.clone().requires_grad_(True)
    yo = O.attention2d(xo, sd, "a")
    # cotangent correlated with the output: d(gamma) = sum r * attn(x) is then a well-conditioned sum (with a purely
    # random cotangent it is a cancelling sum of 2e5 terms whose value is rounding noise in any 16-bit storage)
    r = yo.detach() + 0.3 * torch.randn(6, 32, 32, 32)
    go = torch.autograd.grad((yo * r).sum(), [xo] + list(sd.values()))
    blk = blk.cuda()
    xp = x.cuda().requires_grad_(True)
    yp = blk(xp)
    gp = torch.autograd.grad((yp * r.cuda()).sum(), [xp] + [dict(blk.named_parameters())[k[2:]] for k in sd])
    tol = TOL[precision]
    assert rel(yp.cpu(), yo) < tol
    errs = {n: rel(a.cpu(), b) for n, a, b in zip(["x"] + list(sd), gp, go)}
    print("generator attention:", {k: "%.3g" % v for k, v in errs.items()})
    for n, e in errs.items():
        assert e < 2 * tol, (n, e)


# ------------------------------------------------------------------------------------- caption encoder
@pytest.mark.parametrize("B,V", [(8, 50), (37, 400)])
def test_caption_encoder_vs_oracle(precision, B, V):
    """text.Seq2Seq.encode (t2v_embedding_fwd + engine GEMMs + t2v_lstm_seq_fwd / _bwd) vs oracle seq2seq_encode
    (models/txt/basic.py:49-70): padded outputs, h_n, and every parameter gradient of a loss on (out, hn)."""
    import oracle.txt2vid_oracle as O
    from helpers import synth_batch
    from txt2vid_b200.text import Seq2Seq
    torch.manual_seed(5)
    m = Seq2Seq(vocab_size=V)
    _, tokens, lengths = synth_batch(B, V, T=1, S=1, seed=9)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    out_o, hn_o = O.seq2seq_encode(sd, tokens, lengths)
    r1, r2 = torch.randn_like(out_o), torch.randn_like(hn_o)
    names = [k for k in sd if k.startswith("encoder.lstm") or k.startswith("encoder.embed")]
    g_o = torch.autograd.grad((out_o * r1).sum() + (hn_o * r2).sum(), [sd[k] for k in names])
    m = m.cuda()
    out_p, hidden, hn_p = m.encode(tokens.cuda(), lengths)
    assert tuple(out_p.shape) == tuple(out_o.shape) and tuple(hidden[0].shape) == (8, B, 128)
    pm = dict(m.named_parameters())
    g_p = torch.autograd.grad((out_p * r1.cuda()).sum() + (hn_p * r2.cuda()).sum(), [pm[k] for k in names])
    tol = TOL[precision]
    assert rel(out_p.cpu(), out_o) < tol and rel(hn_p.cpu(), hn_o) < tol, (rel(out_p.cpu(), out_o), rel(hn_p.cpu(), hn_o))
    # padded positions are exactly zero, as pad_packed_sequence
    for b, L in enumerate(lengths):
        assert float(out_p[b, L:].abs().max() if L < out_p.shape[1] else 0.0) == 0.0
    for n, a, b in zip(names, g_p, g_o):
        assert rel(a.cpu(), b) < 3 * tol, (n, rel(a.cpu(), b))


def test_embedding_gather_is_bit_exact():
    from txt2vid_b200 import ops
    w = torch.randn(300, 256, device="cuda")
    t = torch.randint(0, 300, (7, 13), device="cuda")
    ops.set_precision("fp32")
    try:
        assert torch.equal(K().embedding_fwd(t, w), w[t])
    finally:
        ops.set_precision("bf16")
    assert torch.equal(K().embedding_fwd(t, w), w[t].to(BF))


# ------------------------------------------------------------------------------------- heads + fused loss + penalty ops
def test_heads_and_fused_loss_vs_oracle_composition(precision):
    """HeadF (row-dot kernels) + RelLossF (one reduction kernel over all levels and pairs) vs the oracle's
    F.linear / per-level RSGAN composition (gan/cond_gan.py:51-61), values and gradients; then the generator form."""
    import oracle.txt2vid_oracle as O
    from txt2vid_b200 import ops
    g = torch.Generator().manual_seed(6)
    levels = [8, 4, 2, 1]
    Fd, E = 1024, 256
    wu, bu = torch.randn(1, Fd, generator=g) * 0.03, torch.randn(1, generator=g)
    wc, bc = torch.randn(1, Fd + E, generator=g) * 0.03, torch.randn(1, generator=g)
    feats = {k: [torch.randn(b, Fd, generator=g) for b in levels] for k in ("real", "fake")}
    conds = {k: [torch.randn(b, E, generator=g) for b in levels] for k in ("real", "perm")}

    def run(dev, lin, rsgan_pairs):
        P = [t.to(dev).requires_grad_(True) for t in (wu, bu, wc, bc)]
        fr = [t.to(dev).requires_grad_(True) for t in feats["real"]]
        ff = [t.to(dev).requires_grad_(True) for t in feats["fake"]]
        cr, cp = [t.to(dev) for t in conds["real"]], [t.to(dev) for t in conds["perm"]]
        ur = [lin(f, None, P[0], P[1]) for f in fr]
        uf = [lin(f, None, P[0], P[1]) for f in ff]
        c_rr = [lin(f, c, P[2], P[3]) for f, c in zip(fr, cr)]
        c_fr = [lin(f, c, P[2], P[3]) for f, c in zip(ff, cr)]
        c_rp = [lin(f, c, P[2], P[3]) for f, c in zip(fr, cp)]
        loss = rsgan_pairs(ur, uf, c_rr, c_fr, c_rp)
        grads = torch.autograd.grad(loss, P + fr + ff)
        return float(loss), [t.cpu() for t in grads]

    def lin_o(f, c, w, b):
        return F.linear(f if c is None else torch.cat((f, c), 1), w, b)

    def loss_o(ur, uf, c_rr, c_fr, c_rp):
        lu = torch.stack([O.RSGAN.discrim_loss(f, r) for f, r in zip(uf, ur)]).mean()
        l1 = torch.stack([O.RSGAN.discrim_loss(f, r) for f, r in zip(c_fr, c_rr)]).mean()
        l2 = torch.stack([O.RSGAN.discrim_loss(f, r) for f, r in zip(c_rp, c_rr)]).mean()
        return (lu + (l1 + l2) / 2) / 2

    def lin_p(f, c, w, b):
        return ops.head_linear(f, w, b, cond=c)

    def loss_p(ur, uf, c_rr, c_fr, c_rp):
        n = float(len(ur))
        pairs = [(r, f, 0.5 / n) for f, r in zip(uf, ur)] + [(r, f, 0.25 / n) for f, r in zip(c_fr, c_rr)] + \
                [(r, f, 0.25 / n) for f, r in zip(c_rp, c_rr)]
        return ops.rel_loss(pairs, 0)

    lo, go = run("cpu", lin_o, loss_o)
    lp, gp = run("cuda", lin_p, loss_p)
    assert abs(lp - lo) < 1e-5 * abs(lo), (lp, lo)
    for a, b in zip(gp, go):
        assert rel(a, b) < 1e-4, rel(a, b)


def test_head_double_backward_matches_autograd(precision):
    """the heads under the gradient penalty: d/dw of || d(pred)/d(feat) ||^2 through HeadF's differentiable backward"""
    from txt2vid_b200 import ops
    g = torch.Generator().manual_seed(8)
    f0, c0 = torch.randn(6, 1024, generator=g), torch.randn(6, 256, generator=g)
    w0, b0 = torch.randn(1, 1280, generator=g) * 0.05, torch.randn(1, generator=g)

    def run(dev, lin):
        f, c, w, b = (t.to(dev).requires_grad_(True) for t in (f0, c0, w0, b0))
        pred = lin(f, c, w, b)
        gf, gc = torch.autograd.grad(pred, [f, c], torch.ones_like(pred), create_graph=True)
        loss = (gf ** 2).sum() + (gc ** 2).sum() * 0.5 + (pred ** 2).sum()
        return [t.cpu() for t in torch.autograd.grad(loss, [w, b, f, c])]

    go = run("cpu", lambda f, c, w, b: F.linear(torch.cat((f, c), 1), w, b))
    gp = run("cuda", lambda f, c, w, b: ops.head_linear(f, w, b, cond=c))
    for a, b_ in zip(gp, go):
        assert rel(a, b_) < 1e-4, rel(a, b_)


def test_gradient_penalty_arithmetic_kernels():
    """lerp_rows == alpha*real + (1-alpha)*fake bit for bit (same IEEE operations, gan/losses.py:140-145); sum ||g||^2"""
    g = torch.Generator(device="cuda").manual_seed(2)
    real, fake = torch.randn(5, 3, 4, 8, 8, device="cuda", generator=g), torch.randn(5, 3, 4, 8, 8, device="cuda", generator=g)
    a = torch.rand(5, device="cuda", generator=g)
    av = a.view(5, 1, 1, 1, 1)
    assert torch.allclose(K().lerp_rows(real, fake, a), av * real + (1 - av) * fake, rtol=0, atol=1e-6)
    assert abs(float(K().dot(real, real)) - float(real.double().pow(2).sum())) < 1e-3


# ------------------------------------------------------------------------------------- ConvLSTM
@pytest.mark.parametrize("plane", [1, 2])
def test_conv_lstm_vs_oracle(precision, plane):
    """blocks.ConvLSTM (gate GEMM on the engine + cell kernels) vs oracle conv_lstm (models/conv_lstm.py:32-38,75-97):
    all 16 hidden states and the parameter / input gradients."""
    import oracle.txt2vid_oracle as O
    from txt2vid_b200.blocks import ConvLSTM
    torch.manual_seed(10)
    steps, ch, B = 16, 64, 6
    m = ConvLSTM(input_channels=ch, hidden_channels=[ch], kernel_size=3, step=steps, effective_step=range(steps))
    with torch.no_grad():
        for p_ in m.parameters():
            p_.normal_(0, 0.05)
    x = torch.randn(B, ch, plane, plane)
    sd = {"c." + k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    xo = x.clone().requires_grad_(True)
    hs_o = O.conv_lstm(xo, sd, "c.cell0", steps)                  # list of (B, ch, h, w)
    r = torch.randn(steps, B, ch, plane, plane)
    names = list(sd)
    g_o = torch.autograd.grad(sum((h * r[t]).sum() for t, h in enumerate(hs_o)), [xo] + [sd[k] for k in names])
    m = m.cuda()
    xp = x.cuda().requires_grad_(True)
    outs, _ = m(xp)
    pm = dict(m.named_parameters())
    g_p = torch.autograd.grad(sum((h * r[t].cuda()).sum() for t, h in enumerate(outs)), [xp] + [pm[k[2:]] for k in names])
    tol = TOL[precision]
    for t in range(steps):
        assert rel(outs[t].cpu(), hs_o[t]) < tol, (t, rel(outs[t].cpu(), hs_o[t]))
    for n, a, b in zip(["x"] + names, g_p, g_o):
        if float(b.norm()) > 1e-8:
            assert rel(a.cpu(), b) < 3 * tol, (n, rel(a.cpu(), b))


# ------------------------------------------------------------------------------------- Adam
def test_adam_kernel_vs_oracle_adam():
    """t2v_adam_step (multi-tensor) against the oracle's torch.optim.Adam restatement (train/gan.py:93-94) over three
    steps on tensors of odd sizes"""
    import oracle.txt2vid_oracle as O
    from txt2vid_b200.optim import FusedAdam
    g = torch.Generator().manual_seed(12)
    shapes = [(7,), (33, 5), (128, 3, 3, 3), (1,)]
    w0 = [torch.randn(*s, generator=g) for s in shapes]
    grads = [[torch.randn(*s, generator=g) * (10.0 ** (i - 1)) for s in shapes] for i in range(3)]
    sd = {str(i): w.clone() for i, w in enumerate(w0)}
    oa = O.Adam(list(sd), 2e-4, (0.5, 0.999))
    params = [torch.nn.Parameter(w.clone().cuda()) for w in w0]
    opt = FusedAdam([{"params": params}], lr=2e-4, betas=(0.5, 0.999))
    for step in range(3):
        oa.step(sd, {str(i): gr for i, gr in enumerate(grads[step])})
        for p_, gr in zip(params, grads[step]):
            p_.grad = gr.cuda()
        opt.step()
    for i, p_ in enumerate(params):
        assert torch.allclose(p_.detach().cpu(), sd[str(i)], rtol=1e-6, atol=1e-7), i


@pytest.mark.parametrize("B,plane,Cin,Hd", [(8, 1, 1024, 1024), (5, 2, 64, 128), (300, 1, 256, 64)])
def test_fused_lstm_step_equals_gemm_plus_cell_kernel(B, plane, Cin, Hd):
    """t2v_conv_lstm_step (cell update in the gate GEMM's epilogue, gate-interleaved columns) against the unfused
    pair t2v_conv_fprop (fp32 gates) + t2v_lstm_cell_fwd on the same operands: gates bit for bit (same MMA order), c and
    h to fp32 / bf16 rounding, and h written into its (b, t) slot of the merged map."""
    g = torch.Generator(device="cuda").manual_seed(2)
    k = (1, 3, 3) if plane > 1 else (1, 1, 1)
    taps = k[1] * k[2]
    x = torch.randn(B, 1, plane, plane, Cin, device="cuda", generator=g).to(BF)
    w = (torch.randn(4 * Hd, taps, Cin, device="cuda", generator=g) / (taps * Cin) ** 0.5)
    bias = torch.randn(4 * Hd, device="cuda", generator=g)
    c_prev = torch.randn(B, 1, plane, plane, Hd, device="cuda", generator=g)
    steps, t = 3, 1
    gates_ref = K().conv_fprop(x, K().pack_weight(w), bias, None, k, False, True)
    c_ref, h_ref, _ = K().lstm_cell_fwd(gates_ref, c_prev)
    il = K().lstm_gate_interleave(Hd, "cuda")
    merged = torch.zeros(B * steps, 1, plane, plane, Hd, device="cuda", dtype=BF)
    gates, c, h = K().conv_lstm_step(x, K().pack_weight(w[il].contiguous()), bias[il].contiguous(), c_prev, k, merged, t, steps)
    # same MMA order -> identical gates; the cell formulas may contract their FMAs differently in the two kernels
    assert torch.equal(gates, gates_ref)
    assert float((c - c_ref).abs().max()) <= 1e-6 * float(c_ref.abs().max())
    assert float((h.float() - h_ref.float()).abs().max()) <= 2.0 ** -8 * float(h_ref.float().abs().max())
    m = merged.view(B, steps, 1, plane, plane, Hd)
    assert torch.equal(m[:, t], h) and float(m[:, 0].abs().max()) == 0 and float(m[:, 2].abs().max()) == 0
    # first step: no previous cell state
    gates0, c0, h0 = K().conv_lstm_step(x, K().pack_weight(w[il].contiguous()), bias[il].contiguous(), None, k, merged, 0, steps)
    c_ref0, h_ref0, _ = K().lstm_cell_fwd(gates_ref, None)
    assert float((c0 - c_ref0).abs().max()) <= 1e-6 * float(c_ref0.abs().max())
    assert float((h0.float() - h_ref0.float()).abs().max()) <= 2.0 ** -8 * float(h_ref0.float().abs().max())


# ------------------------------------------------------------------------------------- caption pre-training (8 f4)
def _golden_caption():
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "caption_pretrain.json")) as f:
        return json.load(f)


def _probe_index(numel):
    n = min(64, numel)
    return [(i * 2654435761) % numel for i in range(n)]


def run_caption_pretrain_against_golden(device, loss_tol, grad_tol, probe_tol):
    """train_txt.pretrain_step (train/txt.py:166-181) on the fixture recorded from the LIVE reference by
    oracle/make_golden_caption_pretrain.py: same initial weights (checksums), then per mode the loss, the decoded
    symbols, every parameter's gradient norm and a 64-entry probe of every gradient tensor."""
    from txt2vid_b200.text import Seq2Seq
    from txt2vid_b200.train_txt import pretrain_step
    fx = _golden_caption()
    torch.manual_seed(fx["seed"])
    m = Seq2Seq(vocab_size=fx["V"])
    for n, p in m.state_dict().items():
        s, a = fx["weights"][n]
        assert abs(float(p.double().sum()) - s) <= 1e-9 * max(1.0, a) and abs(float(p.double().abs().sum()) - a) <= 1e-9 * a, n
    m = m.to(device)
    sent = torch.tensor(fx["sent"], dtype=torch.long, device=device)
    rep = {}
    for mode, tf in (("teacher_force", True), ("greedy", False)):
        want = fx["modes"][mode]
        loss, sym = pretrain_step(m, sent, fx["lengths"], None, teacher_force=tf)
        rep[mode] = {"loss": abs(float(loss) - want["loss"]) / abs(want["loss"])}
        assert rep[mode]["loss"] < loss_tol, (mode, float(loss), want["loss"])
        if tf:                           # greedy decoding feeds its own arg-max back: symbols are only pinned when forced
            agree = float((sym.cpu() == torch.tensor(want["symbols"])).float().mean())
            assert agree >= (1.0 if loss_tol <= 1e-3 else 0.9), agree
        worst = 0.0
        if not tf and loss_tol > 1e-3:
            continue                     # bf16 greedy decoding: one flipped arg-max changes the decoder's INPUTS
        for n, p in m.named_parameters():
            g = p.grad.detach().float().reshape(-1).cpu()
            w = want["grads"][n]
            e_norm = abs(float(g.double().norm()) - w["norm"]) / (w["norm"] + 1e-12)
            probe = torch.tensor(w["probe"])
            e_probe = float((g[_probe_index(g.numel())] - probe).norm() / (probe.norm() + 1e-12))
            worst = max(worst, e_norm)
            assert e_norm < grad_tol, (mode, n, e_norm)
            assert e_probe < probe_tol or float(probe.norm()) < 1e-6 * w["norm"], (mode, n, e_probe)
            rep[mode]["worst_grad_norm"] = worst
    return rep


def test_caption_pretraining_step_vs_reference_golden(precision):
    """SURVEY 8(f4) on the B200: embedding gather, engine GEMMs, t2v_lstm_seq_fwd / _bwd (encoder: 4-layer Bi-LSTM;
    decoder: the same LSTM stepped token by token from the encoder's final state), vocabulary projection, cross
    entropy -- loss within the north-star bar (fp32 1e-3 / bf16 2e-2), gradients within 3x / probes 5x of it."""
    tol = TOL[precision]
    n0 = K().lib().t2v_launch_count()
    rep = run_caption_pretrain_against_golden("cuda", tol, 3 * tol, 5 * tol)
    assert K().lib().t2v_launch_count() - n0 > 100
    print("caption pre-training deviations:", precision, rep)
