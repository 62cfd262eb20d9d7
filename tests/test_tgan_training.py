"""TGAN trained through train(), CondGan and the command line with its WGAN-GP recipe (scripts/run_tgan.sh:17: WGAN
loss, gradient penalty lambda = 10, 5 critic steps per generator step, Adam 1e-4, betas (0.5, 0.9)).

Covers the penalty kernels (t2v_gp_norm_fwd / _bwd) against their executable spec (tests/gp_norm_spec.py), CondGan's
single-scale critic path, whole recipe iterations through trainer.train_iteration against the fp64 oracle
(tests/tgan_train_oracle.py), the CUDA-graph replay of the 5-critic-step iteration against eager iterations, and the
command line.
"""
import json
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn as nn

import bn_double_backward_spec as BNS
import cpu_kernels
import gp_norm_spec as GNS
import test_families as TF
import tgan_train_oracle as TO
from helpers import ROOT, golden, l2rel
from test_product_vs_oracle_cpu import adam_update_stats

LAMBDA = 10.0
STEPS = 5
LR, BETAS = 1e-4, (0.5, 0.9)
SEED = 4321
F64 = torch.float64


@pytest.fixture()
def emulated_fp32(monkeypatch):
    """product ops and FusedAdam on the CPU spec, fp32 storage"""
    from txt2vid_b200 import ops, optim
    monkeypatch.setattr(ops, "K", cpu_kernels)
    monkeypatch.setattr(optim, "K", cpu_kernels)
    BNS.install(monkeypatch)
    GNS.install(monkeypatch)
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


def recipe_params(**kw):
    """train()'s params for the recipe at one 64x64 level (the CLI defaults for everything else)"""
    p = SimpleNamespace(data_is_imgs=False, img_model=False, frame_sizes=[64], subsample_input=False,
                        discrim_steps=STEPS, gen_steps=1, gp_lambda=LAMBDA, no_mean_discrim_loss=True,
                        no_mean_gen_loss=True)
    p.__dict__.update(kw)
    return p


def recipe_gan(gen, dis):
    from txt2vid_b200.gan import CondGan, MixedGanLoss, WassersteinGanLoss
    from txt2vid_b200.optim import FusedAdam
    gan = CondGan(gen=gen, discrims=[dis], discrim_names=["video"])
    losses = MixedGanLoss(g_loss=WassersteinGanLoss(), d_loss=WassersteinGanLoss())
    return gan, losses, FusedAdam(dis.parameters(), lr=LR, betas=BETAS), FusedAdam(gen.parameters(), lr=LR, betas=BETAS)


def _params_of(module):
    return {k: p.detach().float().cpu().clone() for k, p in module.named_parameters()}


def _buffers(module):
    return {k: v.detach().float().cpu() for k, v in module.state_dict().items() if "running_" in k}


# ------------------------------------------------------------------------------------- product and oracle
def product_recipe_iteration(gen, dis, x, z, device, monkeypatch):
    """one trainer.train_iteration of the recipe; x (B, 3, T, H, W).  Records every critic step's lossD and penalty,
    and the first critic step's D gradients."""
    from txt2vid_b200 import gan as G
    from txt2vid_b200 import trainer
    gan, losses, optD, optG = recipe_gan(gen, dis)
    rec = {"steps": [], "gp": [], "params0D": _params_of(dis), "params0G": _params_of(gen)}
    d_phase, penalty = trainer._d_phase, G._gradient_penalty

    def spy_d_phase(*a, **kw):
        st = d_phase(*a, **kw)
        rec["steps"].append(float(st["lossD"]))
        if len(rec["steps"]) == 1:
            rec["gD_first"] = TF._grads(dis)
        return st

    def spy_penalty(*a, **kw):
        gp = penalty(*a, **kw)
        rec["gp"].append(float(gp))
        return gp
    monkeypatch.setattr(trainer, "_d_phase", spy_d_phase)
    monkeypatch.setattr(G, "_gradient_penalty", spy_penalty)
    torch.manual_seed(SEED)                    # the penalty's alphas: the CPU generator, one draw per critic step
    ld, lg, fake, xs, _ = trainer.train_iteration(gan, x.permute(0, 2, 1, 3, 4).contiguous(), [], device, optD, optG,
                                                  recipe_params(), losses, end2end=False, z=z)
    rec.update(lossD=float(ld), lossG=float(lg), fake=fake[0].detach().float().cpu(), gD=TF._grads(dis),
               gG=TF._grads(gen), paramsD=_params_of(dis), paramsG=_params_of(gen), buffers_D=_buffers(dis),
               buffers_G=_buffers(gen))
    assert len(fake) == 1 and len(xs) == 1
    return rec


def oracle_recipe_iteration(gen, dis, x, z, dtype=F64):
    import oracle.families_oracle as O
    torch.manual_seed(SEED)
    alphas = [torch.rand(x.shape[0]).to(dtype) for _ in range(STEPS)]
    return TO.recipe_iteration(O.leaves(gen.state_dict(), dtype), O.leaves(dis.state_dict(), dtype), x.to(dtype),
                               z.to(dtype), alphas, LAMBDA, LR, BETAS)


def oracle_sensitivity(gen, dis, x, z, orc, rel=2.0 ** -20):
    """recipe_deviation of the fp64 oracle from `orc` when every weight and the input clip are scaled by
    (1 + rel N(0, 1)) (seeded)"""
    import copy
    g = torch.Generator().manual_seed(5)
    gen2, dis2 = copy.deepcopy(gen), copy.deepcopy(dis)
    with torch.no_grad():
        for p in list(gen2.parameters()) + list(dis2.parameters()):
            p.mul_(1 + rel * torch.randn(p.shape, generator=g))
    x2 = x * (1 + rel * torch.randn(x.shape, generator=g))
    return recipe_deviation(orc, oracle_recipe_iteration(gen2, dis2, x2, z))


def _worst_grad(ref, mine):
    """worst per-tensor relative L2 over the tensors with a significant gradient (test_families._compare)"""
    scale = max(float(v.norm()) for v in ref.values())
    w = 0.0
    for k, g in ref.items():
        assert k in mine, k
        if float(g.norm()) < TF.ZERO_GRAD * scale:
            assert float(mine[k].norm()) < 100 * TF.ZERO_GRAD * scale, k
            continue
        w = max(w, l2rel(mine[k], g))
    return w


def recipe_deviation(orc, got):
    """worst gradient tensor of the first critic step, of the last one and of the G step; relative L2 of the Adam
    updates of D and G over the iteration; worst BatchNorm running statistic after it"""
    rep = {"gradD_first": _worst_grad(orc["gD_first"], got["gD_first"]),
           "gradD_last": _worst_grad(orc["gD"], got["gD"]), "gradG": _worst_grad(orc["gG"], got["gG"]),
           "updateD": adam_update_stats(orc, got, "D"), "updateG": adam_update_stats(orc, got, "G")}
    for n in ("D", "G"):
        assert set(got["buffers_" + n]) == set(orc["buffers_" + n]), n
    rep["buffers"] = max(l2rel(got["buffers_" + n][k], v) for n in ("D", "G") for k, v in orc["buffers_" + n].items())
    return rep


# Bars after the five critic steps.  Adam moves every weight by about lr whatever the size of its gradient, so an
# element whose gradient is near zero takes either sign on the slightest change; the following critic steps and the G
# step then see slightly different critics.  The fp64 oracle itself moves that way when every weight and the input clip
# are scaled by (1 + 2^-20 N(0, 1)), a perturbation below the operand precision of the fp32 mode (bf16 hi / lo splits,
# 2^-16): at B = 8 by 2.9e-3 on the first critic step's gradients, 5.7e-2 on the last one's, 0.10 on the G step's,
# 1.9e-2 / 0.30 on the Adam updates of D / G and 3.6e-3 on the running statistics.  The one-step bars (1e-2 gradients,
# 2e-2 first Adam update, 1e-3 statistics) hold for the first critic step; after it the bar is FLOOR_FACTOR x that
# sensitivity where it is larger, measured on the same inputs in the same test.  Measured on a B200 in fp32 mode at
# B = 8: 1.1e-4 / 2.2e-2 / 4.2e-2 on those gradients, 3.5e-3 / 0.20 on the updates, 6.6e-4 on the statistics.
FLOOR_FACTOR = 2.0
ONE_STEP_BARS = {"gradD_first": 1e-2, "gradD_last": 1e-2, "gradG": 1e-2, "updateD": 2e-2, "updateG": 2e-2,
                 "buffers": 1e-3}


def compare_recipe(orc, got, floor, loss_tol=1e-3):
    """every critic step's lossD on the critic scale lambda |gp| + |D(real)| + |D(fake)| of that step
    (test_critic_gradient_penalty._compare_gp), lossG on the G phase's critic scale |D(real)| + |D(fake)|; then
    recipe_deviation against ONE_STEP_BARS, or FLOOR_FACTOR x the oracle's sensitivity where that is larger (the first
    critic step always at the one-step bar)"""
    assert len(got["steps"]) == len(orc["steps"]) == STEPS
    for j, (o, g) in enumerate(zip(orc["steps"], got["steps"])):
        scale = LAMBDA * abs(o["gp"]) + abs(o["d_real"]) + abs(o["d_fake"])
        assert abs(g - o["lossD"]) <= loss_tol * scale, (j, g, o["lossD"], scale)
    assert abs(got["lossD"] - orc["lossD"]) <= loss_tol * sum(LAMBDA * abs(o["gp"]) + abs(o["d_real"]) +
                                                              abs(o["d_fake"]) for o in orc["steps"])
    g_scale = abs(orc["real_pred"]) + abs(orc["lossG"])
    assert abs(got["lossG"] - orc["lossG"]) <= loss_tol * g_scale, (got["lossG"], orc["lossG"])
    rep = recipe_deviation(orc, got)
    bars = {k: v if k == "gradD_first" else max(v, FLOOR_FACTOR * floor[k]) for k, v in ONE_STEP_BARS.items()}
    print("recipe iteration: lossD steps %s (oracle %s) lossG %.6f (oracle %.6f)"
          % (got["steps"], [s["lossD"] for s in orc["steps"]], got["lossG"], orc["lossG"]))
    print("  deviation %s\n  sensitivity %s\n  bars %s" % tuple(json.dumps({k: float("%.3g" % v) for k, v in d.items()})
                                                            for d in (rep, floor, bars)))
    for k, bar in bars.items():
        assert rep[k] <= bar, (k, rep[k], bar)
    return rep


def _tgan_setup(B):
    fx = golden("tgan_B8.json")
    gen, dis = TF.build_tgan()
    return gen, dis, TF._synth(B, 16, 64, fx["input_seed"]), torch.tensor(fx["z"])[:B]


# ------------------------------------------------------------------------------------- CPU
def test_gp_norm_spec_matches_autograd():
    """the spec of the penalty kernels in fp64 == torch autograd of mean((g.norm(dim=1) - 1)^2), a zero row included
    (torch's norm takes the zero subgradient there; the spec and the kernel write dg = 0)"""
    gen = torch.Generator().manual_seed(3)
    for B, S in ((1, 4), (3, 20), (6, 300)):
        g = torch.randn(B, S, generator=gen, dtype=F64) * torch.linspace(0.02, 0.2, B, dtype=F64).view(B, 1)
        if B > 1:
            g[1] = 0
        gr = g.clone().requires_grad_(True)
        ref = ((gr.norm(dim=1) - 1) ** 2).mean()
        gout = torch.tensor(0.7, dtype=F64)
        (dref,) = torch.autograd.grad(ref, gr, gout)
        val, norms = GNS.gp_norm_fwd(g)
        dg = GNS.gp_norm_bwd(g, norms, gout)
        assert val.dtype == F64 and dg.dtype == F64 and dg.shape == g.shape
        assert abs(float(val - ref)) <= 1e-10 * max(1.0, abs(float(ref)))
        assert float((dg - dref).norm()) <= 1e-10 * max(1.0, float(dref.norm()))
        if B > 1:
            assert float(norms[1]) == 0 and torch.all(dg[1] == 0) and torch.all(dref[1] == 0)


def test_gp_norm_entry_points_reject_bad_shapes():
    """T2V_ERR_ARG before any CUDA call: S % 4 != 0, B < 1"""
    from txt2vid_b200 import _lib
    lib = _lib.lib()
    ERR_ARG = -1                                      # T2V_ERR_ARG of include/t2v.h
    for B, S in ((2, 6), (3, 5), (0, 8)):
        assert lib.t2v_gp_norm_fwd(None, None, None, None, B, S, 1, None) == ERR_ARG
        assert lib.t2v_gp_norm_bwd(None, None, None, None, B, S, None) == ERR_ARG


def test_single_scale_critic_with_captions_is_refused():
    from txt2vid_b200.gan import CondGan, WassersteinGanLoss
    from txt2vid_b200.tgan import Discrim
    dis = Discrim(cond_dim=0)
    gan = CondGan(gen=nn.Linear(1, 1), discrims=[dis])
    x, cond = torch.zeros(2, 3, 16, 64, 64), torch.zeros(2, 8)
    loss = WassersteinGanLoss()
    with pytest.raises(ValueError, match="conditional single-scale critics"):
        gan.discrim_step(real=[x], fake=[x], cond=[cond], loss=loss.discrim_loss, gp_lambda=LAMBDA)
    with pytest.raises(ValueError, match="conditional single-scale critics"):
        gan.gen_step(fake=[x], real_pred=[torch.zeros(())], cond=[cond], loss=loss.gen_loss)


def test_recipe_iteration_cpu(emulated_fp32, monkeypatch):
    """the whole recipe iteration (5 penalised critic steps, real_pred, G step, FusedAdam on both) through
    trainer.train_iteration at B = 4, product ops on the CPU spec in fp32 storage, against the fp64 oracle"""
    gen, dis, x, z = _tgan_setup(4)
    orc = oracle_recipe_iteration(gen, dis, x, z)
    floor = oracle_sensitivity(gen, dis, x, z, orc)
    got = product_recipe_iteration(gen, dis, x, z, "cpu", monkeypatch)
    compare_recipe(orc, got, floor)


# ------------------------------------------------------------------------------------- GPU: the kernels
_GP_CASES = [(B, S) for B in (1, 3, 64) for S in (4, 3 * 16 * 64 * 64, 3 * 8 * 32 * 32)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,S", _GP_CASES)
def test_gp_norm_kernels_vs_spec(B, S):
    """t2v_gp_norm_fwd / _bwd against the spec in fp64 on the same input: 1e-5 relative on the penalty, the norms and
    dg; two calls bit-identical (fixed reduction order)"""
    from txt2vid_b200 import kernels
    gen = torch.Generator(device="cuda").manual_seed(B * 7 + S)
    g = torch.randn(B, S, device="cuda", generator=gen)
    # row norms 0.5, 1.5, 2.5: away from 1, where (n - 1)^2 cancels and no fp32 reduction meets 1e-5
    g = g / g.norm(dim=1, keepdim=True) * (0.5 + torch.arange(B, device="cuda").view(B, 1) % 3)
    if B == 3:
        g[1] = 0
    gout = torch.tensor(10.0, device="cuda")
    out, norms = kernels.gp_norm_fwd(g)
    dg = kernels.gp_norm_bwd(g, norms, gout)
    out2, norms2 = kernels.gp_norm_fwd(g)
    dg2 = kernels.gp_norm_bwd(g, norms2, gout)
    assert torch.equal(out, out2) and torch.equal(norms, norms2) and torch.equal(dg, dg2)
    rv, rn = GNS.gp_norm_fwd(g.double().cpu())
    rdg = GNS.gp_norm_bwd(g.double().cpu(), rn, gout.double().cpu())
    assert abs(float(out) - float(rv)) <= 1e-5 * abs(float(rv)), (float(out), float(rv))
    assert float((norms.double().cpu() - rn).norm()) <= 1e-5 * float(rn.norm())
    assert float((dg.double().cpu() - rdg).norm()) <= 1e-5 * float(rdg.norm())
    if B == 3:
        assert torch.all(dg[1] == 0)


@pytest.mark.gpu
def test_penalty_kernels_match_aten_composition_on_tgan_critic(fp32_mode):
    """_gradient_penalty on the TGAN critic, fp32 mode: the fused penalty and the ATen composition it replaces give
    the same penalty and critic gradients within 1e-5"""
    from txt2vid_b200 import gan as G
    from txt2vid_b200 import ops
    gen, dis, x, z = _tgan_setup(8)
    gen, dis, x, z = gen.cuda(), dis.cuda(), x.cuda(), z.cuda()
    with torch.no_grad():
        fake = gen(z)
    res = []
    for combine in (torch.mean, lambda n: torch.mean(n)):        # not torch.mean itself: the ATen composition
        ops.zero_grads(dis)
        torch.manual_seed(SEED)
        gp = G._gradient_penalty(dis, real_x=x, fake_x=fake, combine=combine)
        gp.backward()
        res.append((float(gp), TF._grads(dis)))
    (gp_f, g_f), (gp_a, g_a) = res
    print("penalty fused %.8f aten %.8f" % (gp_f, gp_a))
    assert abs(gp_f - gp_a) <= 1e-5 * abs(gp_a)
    assert max(l2rel(g_f[k], g_a[k]) for k in g_a) <= 1e-5


# ------------------------------------------------------------------------------------- GPU: the recipe iteration
@pytest.mark.gpu
def test_recipe_iteration_gpu_fp32_mode(fp32_mode, monkeypatch):
    """B = 8 on the B200 in fp32 storage against the fp64 oracle: the penalties and the critic-step losses and lossG
    at 1e-3, gradients, Adam updates and BatchNorm running statistics at the bars of compare_recipe"""
    gen, dis, x, z = _tgan_setup(8)
    orc = oracle_recipe_iteration(gen, dis, x, z)
    floor = oracle_sensitivity(gen, dis, x, z, orc)
    got = product_recipe_iteration(gen.cuda(), dis.cuda(), x.cuda(), z.cuda(), "cuda", monkeypatch)
    for j, (o, g) in enumerate(zip(orc["steps"], got["gp"])):
        assert abs(g - o["gp"]) <= 1e-3 * abs(o["gp"]), (j, g, o["gp"])
    compare_recipe(orc, got, floor)


def _floor_gp(family):
    with open(os.path.join(ROOT, "profiles", "r03_bf16_floor_families_gp.json")) as f:
        for line in f:
            if line.strip() and json.loads(line)["family"] == family:
                return json.loads(line)
    raise KeyError(family)


@pytest.mark.gpu
def test_recipe_iteration_gpu_bf16(monkeypatch):
    """bf16 storage: finite losses; the first critic step's penalty and D gradients within 1.5x the measured bf16
    floor of the penalised step (profiles/r03_bf16_floor_families_gp.json, tgan_B8_gp) against the fp32 oracle"""
    fl = _floor_gp("tgan_B8_gp")
    gen, dis, x, z = _tgan_setup(8)
    orc = oracle_recipe_iteration(gen, dis, x, z, dtype=torch.float32)
    got = product_recipe_iteration(gen.cuda(), dis.cuda(), x.cuda(), z.cuda(), "cuda", monkeypatch)
    assert all(math.isfinite(v) for v in got["steps"] + [got["lossD"], got["lossG"]])
    gp_err = abs(got["gp"][0] - orc["steps"][0]["gp"]) / abs(orc["steps"][0]["gp"])
    grad_err = _worst_grad(orc["gD_first"], got["gD_first"])
    print("recipe bf16: first-step gp %.6f (oracle %.6f, rel %.2e, bar %.2e); worst D grad %.3f (bar %.3f)"
          % (got["gp"][0], orc["steps"][0]["gp"], gp_err, 1.5 * fl["gp_rel"], grad_err, 1.5 * fl["gradD_worst"]))
    assert gp_err <= 1.5 * fl["gp_rel"]
    assert grad_err <= 1.5 * fl["gradD_worst"]


# ------------------------------------------------------------------------------------- GPU: graph and command line
def _graph_setup(B):
    from txt2vid_b200 import ops
    ops.PACKS.clear()
    gen, dis = TF.build_tgan()
    gen, dis = gen.cuda(), dis.cuda()
    torch.manual_seed(7)
    torch.cuda.manual_seed(7)
    np.random.seed(7)
    gan, losses, optD, optG = recipe_gan(gen, dis)
    g = torch.Generator().manual_seed(11)
    batches = [(torch.rand(B, 16, 3, 64, 64, generator=g) * 2 - 1).cuda() for _ in range(6)]
    return gan, losses, optD, optG, batches


@pytest.mark.gpu
def test_graph_with_five_critic_steps_matches_eager():
    """GraphedTrainStep with discrim_steps = 5 against eager train_iteration over 6 iterations from the same seeds
    (losses at the bars of test_graphed_step_gpu.test_graph_replay_matches_eager); step counts after
    sync_optimizer_state; one row of staged bias corrections per captured critic step; 5 penalty alphas per
    iteration in the host-RNG call sequence; a ragged batch between replays"""
    from txt2vid_b200.trainer import GraphedTrainStep, train_iteration
    B, dev = 8, torch.device("cuda", 0)
    params = recipe_params()
    gan, losses, optD, optG, batches = _graph_setup(B)
    eager = []
    for x in batches:
        ld, lg, _, _, _ = train_iteration(gan, x, [], dev, optD, optG, params, losses, end2end=False)
        eager.append((float(ld), float(lg)))
    gan, losses, optD, optG, batches = _graph_setup(B)
    step = GraphedTrainStep(gan, optD, optG, params, losses, dev, warmup=2)
    graphed = []
    for x in batches:
        ld, lg = step(x, [])
        graphed.append((float(ld), float(lg)))
    print("eager  ", eager)
    print("graphed", graphed)
    assert step.graphs is not None and step.draws.calls == [("alpha", B)] * STEPS
    for i, ((a, b), (c, d)) in enumerate(zip(eager, graphed)):
        tol = 3e-2 if i < 3 else 1.5e-1
        assert abs(a - c) < tol * max(1.0, abs(a)) and abs(b - d) < tol * max(1.0, abs(b)), (i, eager, graphed)
    assert all(np.isfinite(v) for pair in graphed for v in pair)
    assert len({round(p[0], 4) for p in graphed}) > 2
    torch.cuda.synchronize()
    b1, b2 = BETAS
    want = torch.tensor([[LR / (1 - b1 ** t), 1 / (1 - b2 ** t) ** 0.5] for t in range(26, 31)], dtype=torch.float32)
    assert optD.dyn.shape == (STEPS, 2) and torch.equal(optD.dyn.cpu(), want), (optD.dyn, want)
    step.sync_optimizer_state()
    assert {st["step"] for st in optD.state.values()} == {STEPS * 6}
    assert {st["step"] for st in optG.state.values()} == {6}
    # a ragged last batch runs eagerly between replays; the counts keep advancing by 5 and 1 per iteration
    step.begin_eager_step()
    train_iteration(gan, batches[0][:4].contiguous(), [], dev, optD, optG, params, losses, end2end=False)
    step.end_eager_step()
    ld, lg = step(batches[1], [])
    assert math.isfinite(float(ld)) and math.isfinite(float(lg))
    step.sync_optimizer_state()
    assert {st["step"] for st in optD.state.values()} == {STEPS * 8}
    assert {st["step"] for st in optG.state.values()} == {8}


_CLI = ["--cuda", "--seed", "100", "--G", "txt2vid.models.tgan.gen.Gen", "--D", "txt2vid.models.tgan.discrim.Discrim",
        "--D_loss", "txt2vid.gan.losses.WassersteinGanLoss", "--gp_lambda", "10", "--discrim_steps", "5",
        "--dont_use_sent", "--frame_sizes", "64", "--cuda_graphs", "--epochs", "1", "--batch_size", "8"]


@pytest.mark.gpu
def test_cli_trains_tgan_with_its_recipe(tmp_path, capsys):
    """the recipe's command line through txt2vid.train.gan.main on the on-device moving-digits clips (batch 8, 6
    batches, CUDA graphs): losses logged, a checkpoint with 20 critic Adam steps after iteration 4, samples written;
    then --test on the same model writes its 64x64 sample"""
    from txt2vid.train.gan import build_parser, main
    data_path, out, samples = tmp_path / "data.json", tmp_path / "out", tmp_path / "samples"
    with open(data_path, "w") as f:
        json.dump({"class": "txt2vid.data.MovingDigitsDataset",
                   "args": {"batch_size": 8, "num_batches": 6, "seed": 300}}, f)
    paths = ["--data", str(data_path), "--out", str(out), "--out_samples", str(samples)]
    main(build_parser().parse_args(_CLI + paths + ["--log_period", "2", "--save_example_period", "4",
                                                "--save_model_period", "4"]))
    text = capsys.readouterr().out
    assert "Iter 6, Loss_D:" in text and "Loss_G:" in text
    ckpts = [p for p in out.iterdir() if p.name.startswith("iter_4_")]
    assert len(ckpts) == 1
    saved = torch.load(ckpts[0], weights_only=False)
    assert {"gen", "optD", "optG", "discrim-0"} <= set(saved.keys())
    assert {st["step"] for st in saved["optD"]["state"].values()} == {20}
    names = {p.name for p in samples.iterdir()}
    assert any(n.startswith("fake_samples_epoch_000_iter_000004_64x64") and n.endswith(".png") for n in names)
    main(build_parser().parse_args(_CLI + paths + ["--test", "--weights", str(ckpts[0])]))
    assert (samples / "64x64_0_0.jpg").exists()
