"""GPU: one full TGANv2 training iteration (B=8, 64x64x16) on the sm_100a kernels against the CPU oracle
on the same weights, inputs and host-RNG stream.  bf16 mode: losses inside BASELINE north_star's 2e-2 bar, bit-exact
real pyramid, generated clips and gradients within 1.5x the MEASURED bf16 floor of this network (the oracle itself
under torch.autocast(bfloat16) vs fp32 on a B200: profiles/r02_bf16_floor_*.json, helpers.bf16_bars).  fp32 mode:
everything within 1e-3."""
import pytest
import torch

from helpers import bf16_bars, golden
from test_product_vs_oracle_cpu import compare, run_product_iteration

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,conditional", [("tganv2_cond_B8.json", True), ("tganv2_uncond_B8.json", False)])
def test_full_iteration_on_b200(name, conditional):
    from txt2vid_b200 import _lib, ops
    ops.PACKS.clear()
    n0 = _lib.lib().t2v_launch_count()
    orc, got = run_product_iteration(conditional, golden(name), "cuda")
    launches = _lib.lib().t2v_launch_count() - n0
    print("kernel launches in one iteration:", launches)
    assert launches > 500
    loss_tol, g_l2, g_cos, fake_tol, d_l2, d_cos = bf16_bars("cond_g0" if conditional else "uncond_g0")
    rep = compare(orc, got, loss_tol, g_l2, g_cos, fake_tol)
    assert rep["gradD"]["l2"] < d_l2 and rep["gradD"]["cos"] > d_cos, rep
    import json, os
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/iteration_parity_%s.json" % name.split(".")[0], "w") as f:
        json.dump({"launches": int(launches), "report": rep}, f)


def _record(tag, payload):
    import json, os
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/iteration_parity_%s.json" % tag, "w") as f:
        json.dump(payload, f)


@pytest.mark.parametrize("name,conditional,perturb", [("tganv2_cond_B8.json", True, False),
                                                      ("tganv2_cond_B8.json", True, True),
                                                      ("tganv2_uncond_B8.json", False, False)])
def test_full_iteration_fp32_mode_on_b200(name, conditional, perturb):
    """BASELINE north_star, fp32 bar: one full iteration through the REAL kernels in the fp32 storage mode (same
    typed kernels instantiated for float, convolutions as exact fp32 FMAs on the CUDA cores) within 1e-3 relative of the
    oracle on both losses, the generated clips and the gradients of G and D -- with the non-local blocks switched on
    (gamma = 0.5) and non-trivial BatchNorm affine parameters in the `perturb` case."""
    from test_product_vs_oracle_cpu import adam_update_stats
    from txt2vid_b200 import _lib, ops
    ops.PACKS.clear()
    n0 = _lib.lib().t2v_launch_count()
    orc, got = run_product_iteration(conditional, golden(name), "cuda", perturb=perturb, precision="fp32")
    launches = _lib.lib().t2v_launch_count() - n0
    assert launches > 500
    rep = compare(orc, got, 1e-3, 1e-3, 0.999999, 1e-3)
    assert rep["gradD"]["worst"][1] < 4e-3 and rep["gradG"]["worst"][1] < 4e-3, rep
    rep["adamD"], rep["adamG"] = adam_update_stats(orc, got, "D"), adam_update_stats(orc, got, "G")
    # first Adam step = -lr * g / (|g| + eps): elements whose gradient is at rounding level may flip sign
    assert rep["adamD"] < 2e-2 and rep["adamG"] < 2e-2, rep
    _record("%s_fp32%s" % (name.split(".")[0], "_attn_on" if perturb else ""),
            {"precision": "fp32", "perturb": perturb, "launches": int(launches), "report": rep})


def test_full_iteration_bf16_attention_on_b200():
    """bf16 mode with the non-local blocks ON (gamma = 0.5) and non-trivial BatchNorm affine parameters (SURVEY 7.3)"""
    from txt2vid_b200 import ops
    ops.PACKS.clear()
    orc, got = run_product_iteration(True, golden("tganv2_cond_B8.json"), "cuda", perturb=True, precision="bf16")
    loss_tol, g_l2, g_cos, fake_tol, d_l2, d_cos = bf16_bars("cond_g0.5")
    rep = compare(orc, got, loss_tol, g_l2, g_cos, fake_tol)
    assert rep["gradD"]["l2"] < d_l2 and rep["gradD"]["cos"] > d_cos, rep
    _record("tganv2_cond_B8_bf16_attn_on", {"precision": "bf16", "perturb": True, "report": rep})


def test_config5_128x128x32_iteration_on_b200():
    """BASELINE configs[4]: TGANv2 conditional at 128x128x32 (ConvLSTM plane 2x2, frame sizes 16/32/64/128), one full
    iteration at B = 8 against the oracle on the same weights / inputs / host-RNG stream.  Same bars as the 64x64x16
    test; exercises the kernels on the larger planes (all four pyramid levels take the stride-(2,1,1) stem conv)."""
    from txt2vid_b200 import ops
    ops.PACKS.clear()
    fx = golden("tganv2_cond_128x128x32_B8.json")         # recorded from the LIVE reference at this size (make_golden.py)
    orc, got = run_product_iteration(True, fx, "cuda", size=128, frames=32, frame_sizes=(16, 32, 64, 128))
    loss_tol, g_l2, g_cos, fake_tol, d_l2, d_cos = bf16_bars("cond_g0")      # same network, larger planes
    rep = compare(orc, got, loss_tol, g_l2, g_cos, fake_tol)
    # the reference's own recorded losses (the oracle reproduces them to 6e-8 / 0 on the CPU: test_oracle_golden.py)
    assert abs(orc["lossD"] - fx["lossD"]) < 2e-5 and abs(orc["lossG"] - fx["lossG"]) < 2e-5
    assert abs(got["lossD"] - fx["lossD"]) <= loss_tol * abs(fx["lossD"]), (got["lossD"], fx["lossD"])
    assert abs(got["lossG"] - fx["lossG"]) <= loss_tol * abs(fx["lossG"]), (got["lossG"], fx["lossG"])
    assert rep["gradD"]["l2"] < d_l2 and rep["gradD"]["cos"] > d_cos, rep
    import json, os
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/iteration_parity_tganv2_cond_128x128x32_B8.json", "w") as f:
        json.dump({"report": rep}, f)


def test_eval_mode_generation_matches_oracle():
    """SURVEY 8(f2): eval-mode sampling (gan/trainer.py:44-90, models/tganv2_cond/gen.py:101,114-115): no subsampling,
    ONE full-resolution output, BatchNorm on its running statistics.  Running statistics are first moved off their
    initial values by one training-mode forward (both sides update them with the same momentum formula)."""
    import oracle.txt2vid_oracle as O
    from helpers import build_product_models, state_to_cpu
    from txt2vid_b200 import ops
    ops.PACKS.clear()
    B = 8
    txt, gen, dis = build_product_models(True, V=100, seed=11)
    sd = O.as_leaves(state_to_cpu(gen))
    g = torch.Generator().manual_seed(3)
    z, cond = torch.randn(B, 256, generator=g), torch.randn(B, 256, generator=g)
    # training-mode forward on both sides with the same frame offsets -> updated running statistics
    new_buf = {}
    O.gen_forward(sd, z, cond, [1, 0, 1], True, 16, new_buf)
    for k, v in new_buf.items():
        sd[k] = v
    gen = gen.cuda()
    draws = iter([1, 0, 1])
    gen.subsample.draw = lambda: next(draws)
    gen.train()
    with torch.no_grad():
        gen(z.cuda(), cond=cond.cuda())
    # eval-mode generation
    z2, cond2 = torch.randn(B, 256, generator=g), torch.randn(B, 256, generator=g)
    with torch.no_grad():
        ref = O.gen_forward(sd, z2, cond2, None, False, 16)
    gen.eval()
    with torch.no_grad():
        got = gen(z2.cuda(), cond=cond2.cuda())
    assert len(got) == len(ref) == 1 and tuple(got[0].shape) == tuple(ref[0].shape) == (B, 3, 16, 64, 64)
    err = float((got[0].float().cpu() - ref[0]).norm() / ref[0].norm())
    print("eval-mode generation, relative L2 vs oracle: %.3e" % err)
    assert err < 6e-2
