"""GPU parity of the convolution engine (tcgen05 implicit GEMM + SIMT) through the C ABI.

Checker: torch conv3d in fp32 (TF32 off) on the same bf16-rounded operands.  Every case runs and is
logged to gpurun_out/conv_engine.log so that one GPU call shows all failures at once.
"""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

LOG = []


def _log(msg):
    LOG.append(msg)
    print(msg, flush=True)


def _ref_conv(x, w, k, bias=None):
    # x (N,D,H,W,Cin) bf16, w (Cout,taps,Cin) bf16 -> fp32 (N,D,H,W,Cout)
    Cout, taps, Cin = w.shape
    w5 = w.float().view(Cout, k[0], k[1], k[2], Cin).permute(0, 4, 1, 2, 3).contiguous()
    y = F.conv3d(x.float().permute(0, 4, 1, 2, 3), w5, bias, padding=(k[0] // 2, k[1] // 2, k[2] // 2))
    return y.permute(0, 2, 3, 4, 1).contiguous()


def _rel(a, b):
    return float((a.float() - b.float()).abs().max() / (b.float().abs().max() + 1e-12))


FPROP_CASES = [
    # N, D, H, W, Cin, Cout, k
    (4, 1, 8, 8, 64, 64, (1, 3, 3)),
    (2, 4, 8, 8, 64, 128, (3, 3, 3)),
    (64, 1, 2, 2, 128, 256, (1, 3, 3)),
    (16, 1, 1, 1, 1024, 512, (1, 1, 1)),
    (16, 1, 1, 1, 1024, 512, (3, 3, 3)),
    (8, 1, 16, 16, 32, 32, (1, 3, 3)),
    (8, 1, 16, 16, 16, 48, (1, 3, 3)),
    (2, 2, 8, 8, 16, 64, (3, 3, 3)),
    (3, 3, 6, 10, 64, 64, (3, 3, 3)),
    (8, 8, 16, 16, 64, 64, (3, 3, 3)),
    (2, 1, 64, 64, 32, 16, (1, 3, 3)),
    (4, 2, 4, 4, 256, 512, (3, 3, 3)),
    (5, 1, 1, 1, 1280, 16, (1, 1, 1)),
]


def _mk(N, D, H, W, Cin, Cout, k, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((N, D, H, W, Cin), device="cuda", generator=g).to(torch.bfloat16)
    taps = k[0] * k[1] * k[2]
    w = (torch.randn((Cout, taps, Cin), device="cuda", generator=g) / (taps * Cin) ** 0.5).to(torch.bfloat16)
    return x, w


@pytest.fixture(scope="module", autouse=True)
def _setup():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/conv_engine.log", "a") as f:
        f.write("\n".join(LOG) + "\n")


# halo-resident fprop (Cin = Cout = 64): lines along h (H >= 16), lines along d (D >= 16, small H), 2-D maps,
# ragged extents / partial tiles / dummy tiles
HALO_FPROP_CASES = [
    (3, 2, 16, 16, 64, 64, (3, 3, 3)),
    (2, 5, 40, 24, 64, 64, (3, 3, 3)),
    (5, 16, 8, 8, 64, 64, (3, 3, 3)),
    (3, 19, 6, 12, 64, 64, (3, 3, 3)),
    (7, 1, 16, 16, 64, 64, (1, 3, 3)),
    (5, 1, 36, 20, 64, 64, (1, 3, 3)),
    (80, 16, 8, 8, 64, 64, (3, 3, 3)),
]


@pytest.mark.parametrize("algo", [1, 2, 3], ids=["tc", "simt", "tcgeneric"])
@pytest.mark.parametrize("case", FPROP_CASES + HALO_FPROP_CASES)
def test_fprop(case, algo):
    from txt2vid_b200 import kernels as K
    N, D, H, W, Cin, Cout, k = case
    x, w = _mk(*case)
    y = K.conv_fprop(x, w, k=k, algo=algo)
    torch.cuda.synchronize()
    ref = _ref_conv(x, w, k)
    e = _rel(y, ref)
    _log("fprop algo=%d case=%s rel=%.3e" % (algo, case, e))
    assert e < 1.5e-2


@pytest.mark.parametrize("algo", [1, 2], ids=["tc", "simt"])
def test_fprop_epilogue(algo):
    from txt2vid_b200 import kernels as K
    for case in [(2, 4, 8, 8, 64, 128, (3, 3, 3)), (3, 4, 16, 16, 64, 64, (3, 3, 3))]:
        Cout = case[5]
        x, w = _mk(*case, seed=1)
        bias = torch.randn(Cout, device="cuda")
        res = torch.randn(case[:4] + (Cout,), device="cuda").to(torch.bfloat16)
        y = K.conv_fprop(x, w, bias=bias, residual=res, k=case[6], relu=True, out_f32=True, algo=algo)
        ref = torch.relu(_ref_conv(x, w, case[6], bias) + res.float())
        e = _rel(y, ref)
        _log("fprop epilogue algo=%d case=%s rel=%.3e" % (algo, case, e))
        assert y.dtype == torch.float32 and e < 2e-3
        yb = K.conv_fprop(x, w, bias=bias, residual=res, k=case[6], relu=True, algo=algo)
        assert yb.dtype == torch.bfloat16 and _rel(yb, ref) < 1.5e-2


@pytest.mark.parametrize("algo", [1, 2], ids=["tc", "simt"])
@pytest.mark.parametrize("case", FPROP_CASES[:4] + FPROP_CASES[8:10] + HALO_FPROP_CASES[:2] + HALO_FPROP_CASES[4:5])
def test_dgrad(case, algo):
    from txt2vid_b200 import kernels as K
    N, D, H, W, Cin, Cout, k = case
    x, w = _mk(*case, seed=2)
    dy = torch.randn((N, D, H, W, Cout), device="cuda").to(torch.bfloat16)
    wT = K.pack_dgrad_weight(w.float())
    dx = K.conv_dgrad(dy, wT, k=k, algo=algo)
    xr = x.float().requires_grad_(True)
    yr = _ref_conv(xr, w, k)
    (gr,) = torch.autograd.grad(yr, xr, dy.float())
    e = _rel(dx, gr)
    _log("dgrad algo=%d case=%s rel=%.3e" % (algo, case, e))
    assert e < 1.5e-2


WGRAD_CASES = [
    (4, 1, 8, 8, 64, 64, (1, 3, 3)),
    (2, 4, 8, 8, 64, 128, (3, 3, 3)),
    (64, 1, 2, 2, 128, 256, (1, 3, 3)),
    (16, 1, 1, 1, 1024, 512, (3, 3, 3)),
    (3, 3, 6, 10, 64, 64, (3, 3, 3)),
    (8, 8, 16, 16, 64, 64, (3, 3, 3)),
    (32, 1, 1, 1, 512, 1024, (1, 1, 1)),
]


# shapes that take the halo-resident 64-channel kernels (halo_sm100.cu): ragged extents, partial tiles,
# both tap-class splits (Cout 64 -> 2 classes, Cout 128 -> 4), 2-D maps, more tiles than CTAs
HALO_CASES = [
    (2, 2, 64, 64, 64, 64, (3, 3, 3)),
    (3, 5, 12, 20, 64, 64, (3, 3, 3)),
    (40, 16, 8, 8, 64, 64, (3, 3, 3)),
    (5, 8, 16, 16, 64, 128, (3, 3, 3)),
    (6, 1, 16, 16, 64, 64, (1, 3, 3)),
    (3, 1, 36, 24, 64, 128, (1, 3, 3)),
]


@pytest.mark.parametrize("algo", [1, 2, 3], ids=["tc", "simt", "tcgeneric"])
@pytest.mark.parametrize("case", WGRAD_CASES + HALO_CASES + [(8, 1, 16, 16, 32, 48, (1, 3, 3)), (4, 2, 4, 4, 3, 5, (3, 3, 3))])
def test_wgrad(case, algo):
    from txt2vid_b200 import kernels as K
    N, D, H, W, Cin, Cout, k = case
    if algo in (1, 3) and (Cin % 64 or Cout % 64):
        pytest.skip("tcgen05 wgrad needs 64-multiples")
    x, w = _mk(*case, seed=3)
    dy = torch.randn((N, D, H, W, Cout), device="cuda").to(torch.bfloat16)
    dw = K.conv_wgrad(dy, x, k=k, algo=algo)
    wr = w.float().requires_grad_(True)
    yr = _ref_conv(x, wr, k)
    (gr,) = torch.autograd.grad(yr, wr, dy.float())
    e = _rel(dw, gr)
    _log("wgrad algo=%d case=%s rel=%.3e" % (algo, case, e))
    assert e < 2e-3
    dw2 = K.conv_wgrad(dy, x, k=k, out=dw.clone(), accumulate=True, algo=algo)
    e2 = _rel(dw2, 2 * gr)
    assert e2 < 2e-3


# stride-(2,1,1) stem convolution (even output planes only): levels 1-3 of the pyramid (D = 8, 4, 2), ragged H / W,
# more tiles than CTAs, odd sample counts for the sample-paired D = 2 case
SD2_CASES = [(3, 8, 16, 16), (2, 4, 32, 32), (5, 2, 64, 64), (3, 2, 16, 16), (2, 6, 40, 24), (1, 2, 20, 12),
             (70, 4, 32, 32)]


def _ref_sd2(x, w, bias=None):
    w5 = w.float().view(64, 3, 3, 3, 64).permute(0, 4, 1, 2, 3).contiguous()
    y = F.conv3d(x.float().permute(0, 4, 1, 2, 3), w5, bias, stride=(2, 1, 1), padding=1)
    return y.permute(0, 2, 3, 4, 1).contiguous()


@pytest.mark.parametrize("shape", SD2_CASES)
def test_sd2_conv(shape):
    """fprop / dgrad / wgrad of Conv3d(64,64,3,stride=(2,1,1),padding=1) against torch fp32 autograd."""
    from txt2vid_b200 import kernels as K
    N, D, H, W = shape
    assert K.conv_sd2_supported((N, D, H, W), 64, 64)
    x, w = _mk(N, D, H, W, 64, 64, (3, 3, 3), seed=7)
    bias = torch.randn(64, device="cuda")
    y = K.conv_fprop_sd2(x, w, bias)
    assert tuple(y.shape) == (N, D // 2, H, W, 64)
    ref = _ref_sd2(x, w, bias)
    e = _rel(y, ref)
    # identical to the even planes of the stride-1 kernel
    full = K.conv_fprop(x, w, bias=bias, k=(3, 3, 3))
    e_same = _rel(y, full[:, ::2])
    dy = torch.randn((N, D // 2, H, W, 64), device="cuda").to(torch.bfloat16)
    xr, wr = x.float().requires_grad_(True), w.float().requires_grad_(True)
    gx, gw = torch.autograd.grad(_ref_sd2(xr, wr), (xr, wr), dy.float())
    dx = K.conv_dgrad_sd2(dy, K.pack_dgrad_weight(w.float()))
    dw = K.conv_wgrad_sd2(dy, x)
    e_dx, e_dw = _rel(dx, gx), _rel(dw, gw)
    _log("sd2 %s fprop %.3e (vs stride-1 kernel %.3e) dgrad %.3e wgrad %.3e" % (shape, e, e_same, e_dx, e_dw))
    assert e < 1.5e-2 and e_same < 1e-6 and e_dx < 1.5e-2 and e_dw < 2e-3


@pytest.mark.parametrize("case", [(2, 4, 8, 8, 64, 128, (3, 3, 3)), (3, 4, 16, 16, 64, 64, (3, 3, 3)),
                                  (4, 1, 4, 4, 256, 256, (3, 3, 3)), (2, 4, 32, 32, 64, 64, (3, 3, 3))])
def test_dgrad_relu_mask_epilogue(case):
    """dx = dgrad(dy) * (ref > 0) in the epilogue (T2V_EPI_RELU_MASK) == the unfused composite, bit for bit."""
    from txt2vid_b200 import kernels as K
    N, D, H, W, Cin, Cout, k = case
    x, w = _mk(*case, seed=11)
    ref = torch.relu(x)
    dy = torch.randn((N, D, H, W, Cout), device="cuda").to(torch.bfloat16)
    wT = K.pack_dgrad_weight(w.float())
    fused = K.conv_dgrad(dy, wT, k=k, relu_ref=ref)
    comp = K.relu_bwd(K.conv_dgrad(dy, wT, k=k), ref)
    assert torch.equal(fused, comp)
    assert float((fused != 0).float().mean()) > 0.2
    if K.conv_sd2_supported((N, D, H, W), Cin, Cout, k):
        dyh = dy[:, ::2].contiguous()
        assert torch.equal(K.conv_dgrad_sd2(dyh, wT, relu_ref=ref), K.relu_bwd(K.conv_dgrad_sd2(dyh, wT), ref))


@pytest.mark.parametrize("shape", [(2, 4, 8, 8), (3, 2, 16, 16), (1, 2, 64, 64), (5, 3, 6, 10), (1, 1, 5, 7),
                                   (37, 16, 8, 8), (150, 16, 8, 8), (40, 2, 64, 64)])
def test_stem_direct(shape):
    """t2v_stem_fprop / t2v_stem_wgrad (im2col tile in shared memory) against torch conv3d fp32 on the bf16 operands."""
    from txt2vid_b200 import kernels as K
    N, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand((N, 3, D, H, W), device="cuda", generator=g) * 2 - 1
    xc16, xc = K.rgb_to_cl(x)
    assert torch.equal(xc16, K.nchw_to_cl(x, 16)) and torch.equal(xc, K.nchw_to_cl(x, 4))
    w3 = torch.randn((64, 27, 3), device="cuda", generator=g) / 9.0
    bias = torch.randn(64, device="cuda", generator=g)
    wp = torch.zeros((64, 32, 4), device="cuda")
    wp[:, :27, :3] = w3
    wp = wp.reshape(64, 128).to(torch.bfloat16).contiguous()
    y = K.stem_fprop(xc, wp, bias, relu=True)
    assert torch.equal(y, K.stem_fprop(xc16, wp, bias, relu=True))
    for _ in range(3):                      # persistent CTAs, double-buffered tiles: run-to-run bit-identical
        assert torch.equal(y, K.stem_fprop(xc, wp, bias, relu=True))
    w5 = wp.float()[:, :108].reshape(64, 27, 4)[..., :3].reshape(64, 3, 3, 3, 3).permute(0, 4, 1, 2, 3).contiguous()
    xin = xc.float()[..., :3].permute(0, 4, 1, 2, 3).contiguous()
    ref = torch.relu(F.conv3d(xin, w5, bias, padding=1)).permute(0, 2, 3, 4, 1)
    e = _rel(y, ref)
    dy = torch.randn((N, D, H, W, 64), device="cuda", generator=g).to(torch.bfloat16)
    dw = K.stem_wgrad(dy, xc)
    gref = torch.nn.grad.conv3d_weight(xin, (64, 3, 3, 3, 3), dy.float().permute(0, 4, 1, 2, 3), padding=1)
    gref = gref.permute(0, 2, 3, 4, 1).reshape(64, 27, 3)
    e_w = _rel(dw, gref)
    dw2 = K.stem_wgrad(dy, xc, out=dw.clone(), accumulate=True)
    _log("stem direct %s fprop %.3e wgrad %.3e" % (shape, e, e_w))
    assert e < 1.5e-2 and e_w < 2e-3 and _rel(dw2, 2 * gref) < 2e-3


@pytest.mark.parametrize("case", [(4, 4, 8, 8, 64, 128, 64), (3, 2, 4, 4, 128, 256, 128), (2, 1, 4, 4, 256, 512, 256),
                                  (5, 1, 2, 2, 512, 1024, 512), (2, 2, 6, 10, 64, 128, 64)])
def test_fprop_fused_skip(case):
    """y = conv3^3(h, w) + conv1^3(x, ws) + b in one implicit GEMM (t2v_conv_fprop_skip) vs the two-launch form."""
    from txt2vid_b200 import kernels as K
    N, D, H, W, Cin, Cout, Cin2 = case
    h, w = _mk(N, D, H, W, Cin, Cout, (3, 3, 3), seed=13)
    x, ws = _mk(N, D, H, W, Cin2, Cout, (1, 1, 1), seed=14)
    bias = torch.randn(Cout, device="cuda")
    y = K.conv_fprop_skip(h, w, bias, x, ws, k=(3, 3, 3))
    ref = _ref_conv(h, w, (3, 3, 3), bias) + _ref_conv(x, ws, (1, 1, 1))
    e = _rel(y, ref)
    two = K.conv_fprop(h, w, bias=bias, residual=K.conv_fprop(x, ws, k=(1, 1, 1)), k=(3, 3, 3))
    _log("fused skip case=%s rel=%.3e (two-launch form %.3e)" % (case, e, _rel(two, ref)))
    assert e < 1.5e-2


def test_sd2_unsupported_shapes():
    from txt2vid_b200 import kernels as K
    assert not K.conv_sd2_supported((4, 16, 8, 8), 64, 64)      # level 0: 8x8 planes stay on the stride-1 kernel
    assert not K.conv_sd2_supported((4, 3, 16, 16), 64, 64)     # odd D
    assert not K.conv_sd2_supported((4, 4, 16, 16), 64, 128)


@pytest.mark.parametrize("case", [(6, 1, 32, 32, 32, 32, (1, 3, 3)), (3, 1, 64, 64, 32, 16, (1, 3, 3)),
                                  (5, 1, 16, 16, 32, 32, (1, 3, 3)), (4, 1, 32, 32, 64, 32, (1, 3, 3)),
                                  (4, 1, 16, 16, 64, 16, (1, 3, 3)), (2, 4, 8, 8, 64, 32, (3, 3, 3)),
                                  (3, 1, 20, 24, 32, 32, (1, 3, 3)), (300, 1, 16, 16, 32, 32, (1, 3, 3))])
def test_wgrad_small_channels_auto(case):
    """algo = auto on the generator's small-channel layers: Cin = 32 runs on position pairs (64-channel views on the
    halo-resident kernel + t2v_wgrad_fold_pairs), Cin = 64 with Cout < 64 on the halo kernel with N = Cout."""
    from txt2vid_b200 import kernels as K
    N, D, H, W, Cin, Cout, k = case
    x, w = _mk(*case, seed=9)
    dy = torch.randn((N, D, H, W, Cout), device="cuda").to(torch.bfloat16)
    dw = K.conv_wgrad(dy, x, k=k)
    wr = w.float().requires_grad_(True)
    (gr,) = torch.autograd.grad(_ref_conv(x, wr, k), wr, dy.float())
    e = _rel(dw, gr)
    dw2 = K.conv_wgrad(dy, x, k=k, out=dw.clone(), accumulate=True)
    _log("wgrad small-channel auto case=%s rel=%.3e" % (case, e))
    assert e < 2e-3 and _rel(dw2, 2 * gr) < 2e-3
    assert _rel(dw, K.conv_wgrad(dy, x, k=k, algo=2)) < 2e-3          # CUDA-core cross-check


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_gconv_same_matches_cuda_core_conv(dtype, monkeypatch):
    """A stride-1 "same" layer through t2v_gconv_fprop (bf16, engine routes off) or t2v_gconv_fprop_f32 and through the
    CUDA-core route of t2v_conv_fprop (algo = 2, or the fp32 parity mode) is one kernel with one summation order
    (16-channel chunks, one flush per tap): bit-identical outputs."""
    from txt2vid_b200 import kernels as K
    monkeypatch.setattr(K, "GCONV_TC", False)
    N, D, H, W, Cin, Cout, k = 3, 3, 6, 10, 64, 80, (3, 3, 3)
    g = torch.Generator(device="cuda").manual_seed(6)
    x = torch.randn((N, D, H, W, Cin), device="cuda", generator=g).to(dtype)
    w = (torch.randn((Cout, 27, Cin), device="cuda", generator=g) / (27 * Cin) ** 0.5).to(dtype)
    bias = torch.randn(Cout, device="cuda", generator=g)
    for out_f32 in (True, False) if dtype == torch.bfloat16 else (True,):
        y = K.gconv_fprop(x, w, bias, k, (1, 1, 1), (1, 1, 1), out_f32=out_f32)
        ref = K.conv_fprop(x, w, bias=bias, k=k, out_f32=out_f32, algo=2)
        assert y.dtype == ref.dtype and torch.equal(y, ref)


def test_simt_odd_channels():
    from txt2vid_b200 import kernels as K
    case = (4, 2, 4, 4, 3, 5, (3, 3, 3))
    x, w = _mk(*case, seed=4)
    y = K.conv_fprop(x, w, k=case[6], algo=0)
    e = _rel(y, _ref_conv(x, w, case[6]))
    _log("simt odd rel=%.3e" % e)
    assert e < 1.5e-2


def test_perf_probe():
    """Not a parity test: first timing of the engine on representative TGANv2 shapes."""
    from txt2vid_b200 import kernels as K
    shapes = [
        ("D stem conv2 3^3 64->64 L0 B=256", (256, 16, 8, 8, 64, 64, (3, 3, 3))),
        ("D stem conv2 3^3 64->64 L1 B=256", (128, 8, 16, 16, 64, 64, (3, 3, 3))),
        ("D stem conv2 3^3 64->64 L2 B=256", (64, 4, 32, 32, 64, 64, (3, 3, 3))),
        ("D stem conv2 3^3 64->64 L3 B=256", (32, 2, 64, 64, 64, 64, (3, 3, 3))),
        ("D down0 conv2 64->128 B=256", (256, 8, 4, 4, 64, 128, (3, 3, 3))),
        ("G up0 conv1 1024->512 @2x2", (4096, 1, 2, 2, 1024, 512, (1, 3, 3))),
        ("G up2 conv1 256->128 @8x8", (4096, 1, 8, 8, 256, 128, (1, 3, 3))),
        ("clstm gate gemm 1024->4096", (256, 1, 1, 1, 1024, 4096, (1, 1, 1))),
    ]
    for name, case in shapes:
        N, D, H, W, Cin, Cout, k = case
        x, w = _mk(*case, seed=5)
        dy = torch.randn((N, D, H, W, Cout), device="cuda").to(torch.bfloat16)
        for what, fn in (("fprop", lambda: K.conv_fprop(x, w, k=k, algo=1)),
                         ("fprop-generic", lambda: K.conv_fprop(x, w, k=k, algo=3)),
                         ("wgrad", lambda: K.conv_wgrad(dy, x, k=k, algo=1)),
                         ("wgrad-generic", lambda: K.conv_wgrad(dy, x, k=k, algo=3))):
            for _ in range(3):
                fn()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(10):
                fn()
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / 10
            live = [kk if ext > 1 else 1 for kk, ext in zip(k, (D, H, W))]
            fl = 2.0 * N * D * H * W * Cin * Cout * live[0] * live[1] * live[2]
            _log("perf %-36s %s %.3f ms  %.1f TFLOP/s (live taps)" % (name, what, ms, fl / ms / 1e9))
