"""GPU: every non-conv kernel of the C ABI against its executable specification (tests/cpu_kernels.py,
run on the same CUDA tensors with torch ops).  Index / layout kernels must be bit-exact."""
import pytest
import torch

import cpu_kernels as C

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def K():
    from txt2vid_b200 import kernels
    return kernels


def rnd(*shape, dtype=BF, scale=1.0):
    return (torch.randn(*shape, device="cuda") * scale).to(dtype)


def close(a, b, tol=1e-2):
    a, b = a.float(), b.float()
    err = float((a - b).abs().max() / (b.abs().max() + 1e-12))
    assert err < tol, err


def test_relu():
    x, dy = rnd(3, 2, 5, 7, 16), rnd(3, 2, 5, 7, 16)
    assert torch.equal(K().relu_fwd(x), C.relu_fwd(x))
    assert torch.equal(K().relu_bwd(dy, x), C.relu_bwd(dy, x))


@pytest.mark.parametrize("shape,k,s,p", [((2, 4, 8, 8, 32), (2, 2, 2), (2, 2, 2), (0, 0, 0)),
                                         ((3, 1, 4, 4, 64), (1, 2, 2), (1, 2, 2), (0, 0, 0)),
                                         ((2, 8, 8, 8, 16), (1, 2, 2), (2, 2, 2), (0, 0, 0)),
                                         ((2, 3, 5, 7, 16), (2, 2, 2), (2, 2, 2), (1, 1, 1)),
                                         ((4, 2, 1, 1, 128), (2, 1, 1), (2, 1, 1), (0, 0, 0))])
def test_avgpool(shape, k, s, p):
    x = rnd(*shape)
    y = K().avgpool_fwd(x, k, s, p)
    close(y, C.avgpool_fwd(x, k, s, p), 5e-3)
    res = rnd(*y.shape)
    close(K().avgpool_fwd(x, k, s, p, res), C.avgpool_fwd(x, k, s, p, res), 5e-3)
    dy = rnd(*y.shape)
    close(K().avgpool_bwd(dy, shape, k, s, p), C.avgpool_bwd(dy, shape, k, s, p), 5e-3)


def test_upsample():
    x = rnd(5, 1, 4, 6, 32)
    assert torch.equal(K().upsample2x_fwd(x), C.upsample2x_fwd(x))
    dy = rnd(5, 1, 8, 12, 32)
    close(K().upsample2x_bwd(dy), C.upsample2x_bwd(dy), 5e-3)


@pytest.mark.parametrize("shape", [(3, 3, 4, 5, 6), (2, 1, 2, 8, 8), (1, 3, 16, 8, 8), (2, 3, 1, 3, 2)])
def test_im2col3_and_adjoint(shape):
    """RGB-stem im2col (index kernel: bit-exact) and its adjoint, incl. <x, A^T y> == <A x, y>."""
    x = torch.randn(*shape, device="cuda")
    Kp = (27 * shape[1] + 31) // 32 * 32
    col = K().im2col3(x, Kp)
    assert torch.equal(col, C.im2col3(x, Kp))
    dcol = rnd(shape[0], shape[2], shape[3], shape[4], Kp)
    dx = K().col2im3(dcol, shape[1])
    close(dx, C.col2im3(dcol, shape[1]), 1e-5)
    xb = x.to(BF).float()
    lhs = float((K().im2col3(xb, Kp).float() * dcol.float()).sum())
    rhs = float((xb * dx).sum())
    assert abs(lhs - rhs) <= 1e-3 * max(1.0, abs(lhs)), (lhs, rhs)


@pytest.mark.parametrize("shape,c8,c2", [((5, 1, 32, 32), 4, 16), ((3, 1, 8, 12), 4, 16), ((2, 2, 4, 6), 8, 16),
                                         ((4, 1, 16, 16), 2, 8),
                                         # maps beyond one CTA of the backward kernel (t2v_attention_bwd_large): the 64 x 64
                                         # map of BASELINE configs[4], and a key count that is not a multiple of 64
                                         ((3, 1, 64, 64), 4, 16), ((2, 1, 48, 40), 4, 16), ((2, 2, 24, 28), 4, 16)])
def test_attention_core(shape, c8, c2):
    """fused non-local core (max-pool + QK^T + softmax + beta.g) and its gradient vs the composite torch formulation"""
    N, D, H, W = shape
    def padded(c, scale):
        t = torch.zeros(N, D, H, W, 16, device="cuda")
        t[..., :c] = torch.randn(N, D, H, W, c, device="cuda") * scale
        return t.to(BF)
    theta, phi, g = padded(c8, 1.0), padded(c8, 1.0), padded(c2, 1.0)
    o = K().attention_fwd(theta, phi, g, c8, c2)
    close(o, C.attention_fwd(theta, phi, g, c8, c2), 1e-2)
    assert float(o[..., c2:].abs().max()) == 0.0 if c2 < 16 else True
    do = padded(c2, 1.0)
    got = K().attention_bwd(theta, phi, g, do, c8, c2)
    ref = C.attention_bwd(theta, phi, g, do, c8, c2)
    for a, b in zip(got, ref):
        close(a, b, 2e-2)


def test_layout_roundtrip():
    x = torch.randn(3, 3, 4, 5, 6, device="cuda")
    y = K().nchw_to_cl(x, 16)
    assert torch.equal(y, C.nchw_to_cl(x, 16))
    assert torch.equal(K().cl_to_nchw(y, 3), C.cl_to_nchw(y, 3))


@pytest.mark.parametrize("Cc", [16, 64, 96, 256, 1024, 40, 24, 48, 368, 1000])
def test_sum_rows_paths(Cc):
    """vectorised column reduction: C/8 a power of two (every thread reads rows), C/8 not dividing 256 (idle threads
    past the last row slot), 256-channel slabs with a narrower last slab"""
    x = rnd(37, 1, 3, 5, Cc)
    close(K().sum_rows(x), C.sum_rows(x), 1e-3)
    x = rnd(5000, 1, 1, 1, Cc)
    close(K().sum_rows(x), C.sum_rows(x), 2e-3)


def test_reductions():
    x = rnd(7, 2, 3, 5, 96)
    close(K().sum_rows(x), C.sum_rows(x), 1e-3)
    close(K().sum_spatial(x), C.sum_spatial(x), 1e-3)
    g = torch.randn(7, 96, device="cuda")
    assert torch.equal(K().broadcast_spatial(g, x.shape), C.broadcast_spatial(g, x.shape))
    x = rnd(70000, 1, 1, 2, 16)                      # more samples than a grid.y / grid.z dimension holds
    close(K().sum_spatial(x), C.sum_spatial(x), 1e-3)


@pytest.mark.parametrize("dt", [BF, torch.float32])
@pytest.mark.parametrize("S", [1, 16, 300])
@pytest.mark.parametrize("Cc", [96, 368, 1024])
def test_sum_spatial_paths(Cc, S, dt):
    """per-sample spatial sum (one block row per sample) in both storage types"""
    x = rnd(5, 1, 1, S, Cc, dtype=dt)
    close(K().sum_spatial(x), C.sum_spatial(x), 1e-4)


def test_activations():
    x, dy = rnd(3, 2, 5, 7, 32), rnd(3, 2, 5, 7, 32)
    assert torch.equal(K().leaky_relu_fwd(x, 0.2), C.leaky_relu_fwd(x, 0.2))
    assert torch.equal(K().leaky_relu_bwd(dy, x, 0.2), C.leaky_relu_bwd(dy, x, 0.2))
    y = K().tanh_fwd(x)
    close(y, C.tanh_fwd(x), 1e-2)
    close(K().tanh_bwd(dy, y), C.tanh_bwd(dy, y), 1e-2)


GCONV_CASES = [
    # x shape (N,D,H,W,Cin), Cout, k, s, p
    ((2, 16, 16, 16, 16), 64, (4, 4, 4), (2, 2, 2), (1, 1, 1)),      # Conv3d k4 s2 p1 (tcwyt/video_discrim.py:12)
    ((3, 1, 12, 12, 64), 128, (1, 4, 4), (1, 2, 2), (0, 1, 1)),      # Conv2d k4 s2 p1 (frame_discrim.py:12)
    ((4, 1, 4, 4, 512), 16, (1, 3, 3), (1, 2, 2), (0, 0, 0)),        # head (1,3,3) s2 p0 (video_discrim.py:46)
    ((4, 2, 3, 3, 80), 16, (1, 3, 3), (1, 1, 1), (0, 0, 0)),         # head (1,3,3) s1 p0 (video_discrim.py:41)
    ((5, 1, 2, 2, 48), 16, (1, 2, 2), (1, 2, 2), (0, 0, 0)),         # Conv2d k2 s2 (frame_discrim.py:49)
    ((3, 1, 1, 7, 32), 48, (1, 1, 3), (1, 1, 1), (0, 0, 1)),         # 1-D
]


@pytest.mark.parametrize("case", GCONV_CASES)
def test_gconv(case):
    """general strided convolution: fprop, data gradient (= transposed convolution) and weight gradient"""
    xs, Cout, k, s, p = case
    x = rnd(*xs)
    taps = k[0] * k[1] * k[2]
    w = (torch.randn(Cout, taps, xs[-1], device="cuda") / (taps * xs[-1]) ** 0.5).to(BF)
    bias = torch.randn(Cout, device="cuda")
    y = K().gconv_fprop(x, w, bias, k, s, p)
    y2 = C.gconv_fprop(x, w, bias, k, s, p)
    assert y.shape == y2.shape
    close(y, y2, 1e-2)
    dy = rnd(*y.shape)
    bias_i = torch.randn(xs[-1], device="cuda")
    dx = K().gconv_dgrad(dy, w, bias_i, xs[1:4], k, s, p)
    close(dx, C.gconv_dgrad(dy, w, bias_i, xs[1:4], k, s, p), 1e-2)
    close(K().gconv_wgrad(dy, x, k, s, p), C.gconv_wgrad(dy, x, k, s, p), 2e-3)


@pytest.mark.parametrize("Cc,shape", [(64, (6, 1, 8, 8)), (512, (4, 2, 3, 3)), (1024, (16, 1, 2, 2)), (48, (5, 1, 4, 4)),
                                      (368, (50, 1, 2, 3))])
@pytest.mark.parametrize("act", [0, 1, 2])
def test_batchnorm_any_shape(Cc, shape, act):
    """BatchNorm1d/2d/3d statistics over all leading dims + fused activation codes (0 none, 1 ReLU, 2 LeakyReLU)"""
    x = rnd(*shape, Cc, scale=1.5) + 0.25
    gamma, beta = torch.rand(Cc, device="cuda") + 0.5, torch.randn(Cc, device="cuda") * 0.3
    rm1, rv1 = torch.zeros(Cc, device="cuda"), torch.ones(Cc, device="cuda")
    rm2, rv2 = rm1.clone(), rv1.clone()
    y, mi, ss = K().bn_forward(x, gamma, beta, rm1, rv1, act, 1)
    y2, mi2, ss2 = C.bn_forward(x, gamma, beta, rm2, rv2, act, 1)
    assert y.shape == x.shape
    close(mi, mi2, 1e-4), close(ss, ss2, 1e-4), close(rm1, rm2, 1e-4), close(rv1, rv2, 1e-4)
    close(y, y2, 1e-2)
    dy = rnd(*shape, Cc)
    dx, dg, db = K().bn_backward(dy, x, mi2, ss2, act, 1)
    dx2, dg2, db2 = C.bn_backward(dy, x, mi2, ss2, act, 1)
    close(dx, dx2, 1e-2), close(dg, dg2, 2e-3), close(db, db2, 2e-3)


@pytest.mark.parametrize("up", [1, 2])
@pytest.mark.parametrize("relu", [True, False])
def test_batchnorm(up, relu):
    N, H, W, Cc = 6, 8, 8, 64
    x = rnd(N, 1, H, W, Cc, scale=1.5) + 0.25
    gamma, beta = torch.rand(Cc, device="cuda") + 0.5, torch.randn(Cc, device="cuda") * 0.3
    rm1, rv1 = torch.zeros(Cc, device="cuda"), torch.ones(Cc, device="cuda")
    rm2, rv2 = rm1.clone(), rv1.clone()
    y, mi, ss = K().bn_forward(x, gamma, beta, rm1, rv1, relu, up)
    y2, mi2, ss2 = C.bn_forward(x, gamma, beta, rm2, rv2, relu, up)
    close(mi, mi2, 1e-4), close(ss, ss2, 1e-4), close(rm1, rm2, 1e-4), close(rv1, rv2, 1e-4)
    close(y, y2, 1e-2)
    dy = rnd(N, 1, H * up, W * up, Cc)
    dx, dg, db = K().bn_backward(dy, x, mi2, ss2, relu, up)
    dx2, dg2, db2 = C.bn_backward(dy, x, mi2, ss2, relu, up)
    close(dx, dx2, 1e-2), close(dg, dg2, 1e-3), close(db, db2, 1e-3)
    # eval mode
    ye, _, _ = K().bn_forward(x, gamma, beta, rm2, rv2, relu, up, training=False)
    ye2, _, _ = C.bn_forward(x, gamma, beta, rm2, rv2, relu, up, training=False)
    close(ye, ye2, 1e-2)


def test_render():
    B, T, H, W = 3, 4, 8, 8
    pre = rnd(B * T, 1, H, W, 16)
    y = K().render_fwd(pre, B, T, 3)
    close(y, C.render_fwd(pre, B, T, 3), 1e-5)
    dy = torch.randn_like(y)
    close(K().render_bwd(dy, y, 16), C.render_bwd(dy, y, 16), 1e-2)


@pytest.mark.parametrize("B,T,bt", [(8, 16, 0), (8, 16, 1), (5, 7, 1), (1, 1, 1), (2, 2, 0)])
def test_gather_scatter_frames_bit_exact(B, T, bt):
    x = rnd(B * T, 1, 4, 4, 32)
    y = K().gather_frames(x, B, T, bt)
    assert torch.equal(y, C.gather_frames(x, B, T, bt))
    assert torch.equal(K().scatter_frames(y, B, T, bt), C.scatter_frames(y, B, T, bt))


def test_pyramid_bit_exact_vs_reference_semantics():
    """x[::2, :, bt::2] and F.interpolate(nearest) must be reproduced bit for bit (SURVEY 8a rows A2/A3)."""
    import torch.nn.functional as F
    x = torch.randn(8, 3, 16, 64, 64, device="cuda")
    for fs in (8, 16, 32):
        assert torch.equal(K().pyramid_level(x, fs, fs), F.interpolate(x, size=(16, fs, fs)))
    for bt in (0, 1):
        assert torch.equal(K().pyramid_level(x, 64, 64, 2, 2, bt), x[::2, :, bt::2].contiguous())
    x = torch.randn(5, 2, 7, 20, 10, device="cuda")
    assert torch.equal(K().pyramid_level(x, 7, 16), F.interpolate(x, size=(7, 7, 16)))
    assert torch.equal(K().pyramid_level(x, 20, 10, 2, 2, 1), x[::2, :, 1::2].contiguous())


def test_lstm_cell():
    P, Hd = 37, 128
    gates = torch.randn(P, 4 * Hd, device="cuda")
    cp = torch.randn(P, Hd, device="cuda")
    c, h, h32 = K().lstm_cell_fwd(gates, cp, True)
    c2, h2, h322 = C.lstm_cell_fwd(gates, cp, True)
    close(c, c2, 1e-5), close(h, h2, 1e-2), close(h32, h322, 1e-5)
    dh, dc = torch.randn(P, Hd, device="cuda"), torch.randn(P, Hd, device="cuda")
    dg, dcp = K().lstm_cell_bwd(gates, cp, c2, dh, dc)
    dg2, dcp2 = C.lstm_cell_bwd(gates, cp, c2, dh, dc)
    close(dg, dg2, 1e-2), close(dcp, dcp2, 1e-5)
    c0, h0, _ = K().lstm_cell_fwd(gates, None)
    c02, h02, _ = C.lstm_cell_fwd(gates, None)
    close(c0, c02, 1e-5)


def test_adam():
    shapes = [(1024, 27, 64), (64,), (3, 5), (1000, 256)] * 20          # > one AdamChunk
    ps = [torch.randn(s, device="cuda") for s in shapes]
    gs = [torch.randn(s, device="cuda") * 0.1 for s in shapes]
    ms = [torch.zeros_like(p) for p in ps]
    vs = [torch.zeros_like(p) for p in ps]
    ps2, ms2, vs2 = [p.clone() for p in ps], [m.clone() for m in ms], [v.clone() for v in vs]
    for step in (1, 2, 3):
        K().adam_step(ps, gs, ms, vs, 2e-4, 0.5, 0.999, 1e-8, step)
        C.adam_step(ps2, gs, ms2, vs2, 2e-4, 0.5, 0.999, 1e-8, step)
    for a, b in zip(ps, ps2):
        assert float((a - b).abs().max()) < 2e-6


def test_weight_packs():
    w = torch.randn(3, 27, 3, device="cuda")
    assert torch.equal(K().pack_weight(w, 16, 16), C.pack_weight(w, 16, 16))
    assert torch.equal(K().pack_dgrad_weight(w, 16, 16), C.pack_dgrad_weight(w, 16, 16))
    w = torch.randn(128, 9, 64, device="cuda")
    assert torch.equal(K().pack_weight(w), C.pack_weight(w))
    assert torch.equal(K().pack_dgrad_weight(w), C.pack_dgrad_weight(w))
    dwp = torch.randn(16, 27, 16, device="cuda")
    assert torch.equal(K().unpack_wgrad(dwp, 3, 3), C.unpack_wgrad(dwp, 3, 3))


def test_no_cpu_fallback():
    from txt2vid_b200._lib import T2VError
    with pytest.raises(T2VError):
        K().relu_fwd(torch.zeros(8, dtype=BF))


def test_data_prefetcher_ring_delivers_every_batch_intact():
    """data.data_prefetcher (data/__init__.py:131-156): chunked side-stream copies into a ring of four staging slots,
    slot reuse guarded by events two hand-outs back.  Each batch must arrive intact and in order even when the
    consumer's work (a long kernel per batch) lags behind the host."""
    from txt2vid_b200.data import data_prefetcher
    old = data_prefetcher.CHUNK_BYTES
    data_prefetcher.CHUNK_BYTES = 1 << 16                   # force many pieces per copy
    try:
        n = 14
        host = [(torch.full((64, 4, 3, 16, 16), float(i)).pin_memory(), torch.full((64, 7), i, dtype=torch.long), [7] * 64)
                for i in range(n)]
        pf = data_prefetcher(iter(host), device="cuda")
        big = torch.randn(4096, 4096, device="cuda")
        sums, toks = [], []
        x, y = pf.next()
        while x is not None:
            for _ in range(3):                               # consumer work that keeps the device behind the host
                big = torch.tanh(big @ big * 1e-4)
            sums.append(x.sum() / x.numel())                 # consumed on the compute stream, after the lag
            toks.append(torch.stack((y[0].min(), y[0].max())))
            assert y[1] == [7] * 64
            x, y = pf.next()
        torch.cuda.synchronize()
        assert len(sums) == n
        assert [float(s) for s in sums] == [float(i) for i in range(n)]
        assert [t.tolist() for t in toks] == [[i, i] for i in range(n)]
    finally:
        data_prefetcher.CHUNK_BYTES = old


def test_data_prefetcher_uint8_frames_normalised_like_the_reference_transforms():
    """uint8 frames through data_prefetcher == transforms.ToTensor() + Normalize(0.5, 0.5) on the CPU, bit for bit."""
    from txt2vid_b200.data import data_prefetcher
    g = torch.Generator().manual_seed(3)
    frames = torch.randint(0, 256, (6, 4, 3, 16, 16), generator=g, dtype=torch.uint8)
    ref = frames.float().div(255).sub(0.5).div(0.5)
    pf = data_prefetcher(iter([(frames.pin_memory(), torch.zeros(6, 5, dtype=torch.long), [5] * 6)]), device="cuda")
    x, y = pf.next()
    torch.cuda.synchronize()
    assert x.dtype == torch.float32 and torch.equal(x.cpu(), ref)
