"""Times the conv engine (fprop + wgrad, CUDA events, 20 launches after 3 warm-ups) on the TGANv2 shapes that
carry the step at batch 1024 / GPU.  Usage: python scripts/perf_shapes.py [tag]  (the tag labels the output)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from txt2vid_b200 import kernels as K

SHAPES = [
    ("G0 128->128 @8x8", (16384, 1, 8, 8, 128, 128, (1, 3, 3))),
    ("G0 256->256 @4x4", (16384, 1, 4, 4, 256, 256, (1, 3, 3))),
    ("G0 512->512 @2x2", (16384, 1, 2, 2, 512, 512, (1, 3, 3))),
    ("G0 1024->512 @2x2", (16384, 1, 2, 2, 1024, 512, (1, 3, 3))),
    ("G0 256->128 @8x8", (16384, 1, 8, 8, 256, 128, (1, 3, 3))),
    ("D 64->64 (512,4,8,8)", (512, 4, 8, 8, 64, 64, (3, 3, 3))),
    ("D 64->64 (1024,8,4,4)", (1024, 8, 4, 4, 64, 64, (3, 3, 3))),
    ("D 128->64 (512,4,8,8)", (512, 4, 8, 8, 128, 64, (3, 3, 3))),
    ("D 64->128 (1024,8,4,4)", (1024, 8, 4, 4, 64, 128, (3, 3, 3))),
    ("D 128->128 (512,2,4,4)", (512, 2, 4, 4, 128, 128, (3, 3, 3))),
    ("D 128->256 (1024,4,2,2)", (1024, 4, 2, 2, 128, 256, (3, 3, 3))),
    ("D 256->256 (256,1,4,4)", (256, 1, 4, 4, 256, 256, (3, 3, 3))),
    ("D 512->512 (256,1,2,2)", (256, 1, 2, 2, 512, 512, (3, 3, 3))),
    ("D 512->1024 (128,1,4,4)", (128, 1, 4, 4, 512, 1024, (3, 3, 3))),
    ("G 32->32 @64x64", (256, 1, 64, 64, 32, 32, (1, 3, 3))),
    ("G 64->32 @32x32", (1024, 1, 32, 32, 64, 32, (1, 3, 3))),
    ("G 128->64 @16x16", (4096, 1, 16, 16, 128, 64, (1, 3, 3))),
    ("G render 128->16 @8x8", (16384, 1, 8, 8, 128, 16, (1, 3, 3))),
    ("stem1 96->64 1x1 L0", (1024, 16, 8, 8, 96, 64, (1, 1, 1))),
    ("LSTM 1024->4096", (1024, 1, 1, 1, 1024, 4096, (1, 1, 1))),
]


def mk(N, D, H, W, Cin, Cout, k, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((N, D, H, W, Cin), device="cuda", generator=g).to(torch.bfloat16)
    taps = k[0] * k[1] * k[2]
    w = (torch.randn((Cout, taps, Cin), device="cuda", generator=g) / (taps * Cin) ** 0.5).to(torch.bfloat16)
    dy = torch.randn((N, D, H, W, Cout), device="cuda", generator=g).to(torch.bfloat16)
    return x, w, dy


def t(fn, n=20):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


tag = sys.argv[1] if len(sys.argv) > 1 else ""
tot_f = tot_w = 0.0
for name, case in SHAPES:
    N, D, H, W, Cin, Cout, k = case
    x, w, dy = mk(*case)
    live = [kk if ext > 1 else 1 for kk, ext in zip(k, (D, H, W))]
    fl = 2.0 * N * D * H * W * Cin * Cout * live[0] * live[1] * live[2]
    tf = t(lambda: K.conv_fprop(x, w, k=k))
    tw = t(lambda: K.conv_wgrad(dy, x, k=k))
    tot_f += tf; tot_w += tw
    print("%-6s %-26s fprop %.3f ms %6.0f TF/s | wgrad %.3f ms %6.0f TF/s" % (tag, name, tf, fl / tf / 1e9, tw, fl / tw / 1e9), flush=True)
    del x, w, dy
print("%-6s TOTAL fprop %.3f ms wgrad %.3f ms" % (tag, tot_f, tot_w))

# stride-(2,1,1) stem convolution vs the stride-1 kernels on the same input (levels 1-3 at batch 1024)
for shp in [(512, 8, 16, 16), (256, 4, 32, 32), (128, 2, 64, 64)]:
    x, w, _ = mk(*shp, 64, 64, (3, 3, 3))
    dyf = torch.randn(shp + (64,), device="cuda").to(torch.bfloat16)
    dyh = dyf[:, ::2].contiguous()
    wT = K.pack_dgrad_weight(w.float())
    fl = 2.0 * x.numel() * 64 * 27
    r = [t(lambda: K.conv_fprop(x, w, k=(3, 3, 3))), t(lambda: K.conv_fprop_sd2(x, w)),
         t(lambda: K.conv_dgrad(dyf, wT, k=(3, 3, 3))), t(lambda: K.conv_dgrad_sd2(dyh, wT)),
         t(lambda: K.conv_wgrad(dyf, x, k=(3, 3, 3))), t(lambda: K.conv_wgrad_sd2(dyh, x))]
    print("%-6s sd2 %s fprop %.3f -> %.3f ms (%.0f TF/s useful) | dgrad %.3f -> %.3f ms | wgrad %.3f -> %.3f ms"
          % (tag, shp, r[0], r[1], fl / 2 / r[1] / 1e9, r[2], r[3], r[4], r[5]), flush=True)

# RGB stem conv: direct kernels vs im2col + 1x1 GEMM (levels 0-3 at batch 1024)
for shp in [(1024, 16, 8, 8), (512, 8, 16, 16), (256, 4, 32, 32), (128, 2, 64, 64)]:
    N, D, H, W = shp
    x = torch.rand((N, 3, D, H, W), device="cuda") * 2 - 1
    xc16, xc = K.rgb_to_cl(x)
    w3 = torch.randn((64, 27, 3), device="cuda") / 9
    wp = K.stem_pack_weight(w3)
    w96 = torch.zeros((64, 1, 96), device="cuda"); w96[:, 0, :81] = w3.reshape(64, 81); w96 = w96.to(torch.bfloat16)
    dy = torch.randn((N, D, H, W, 64), device="cuda").to(torch.bfloat16)
    col = K.im2col3(x, 96)
    r = [t(lambda: K.stem_fprop(xc, wp)), t(lambda: K.im2col3(x, 96)), t(lambda: K.conv_fprop(col, w96, k=(1, 1, 1), relu=True)),
         t(lambda: K.stem_wgrad(dy, xc)), t(lambda: K.conv_wgrad(dy, col, k=(1, 1, 1))),
         t(lambda: K.rgb_to_cl(x)), t(lambda: K.nchw_to_cl(x, 16))]
    print("%-6s stem %s fprop direct %.3f ms | im2col %.3f + GEMM %.3f ms || wgrad direct %.3f ms | GEMM %.3f ms || rgb_to_cl %.3f vs nchw_to_cl16 %.3f ms"
          % (tag, shp, r[0], r[1], r[2], r[3], r[4], r[5], r[6]), flush=True)
