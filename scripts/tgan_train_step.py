"""Time one training iteration of TGAN's WGAN-GP recipe (scripts/run_tgan.sh:17: 5 penalised critic steps, lambda 10,
then one generator step; FusedAdam 1e-4, betas (0.5, 0.9)) through trainer.train_iteration (eager) and
trainer.GraphedTrainStep (one CUDA graph per iteration) at b = 64, 256 and 1024 clips of 3x16x64x64 (each size that
fits), with CUDA events; then the fused penalty kernels (t2v_gp_norm_fwd / _bwd) against the ATen composition they
replace, forward + backward on a (256, 196608) fp32 gradient (200 MB, larger than L2), over many launches, alternating.
Prints the card's name and power limit and appends one JSON line with everything to --out.

Usage: python scripts/tgan_train_step.py [--out profiles/r03_tgan_train_step.json] [--steps 10] [--warmup 3]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from critic_gp_step import card  # noqa: E402
from txt2vid_b200 import kernels as K  # noqa: E402
from txt2vid_b200 import ops  # noqa: E402
from txt2vid_b200.gan import CondGan, MixedGanLoss, WassersteinGanLoss  # noqa: E402
from txt2vid_b200.optim import FusedAdam  # noqa: E402
from txt2vid_b200.tgan import Discrim, Gen  # noqa: E402
from txt2vid_b200.trainer import GraphedTrainStep, train_iteration  # noqa: E402
from txt2vid_b200.util import init  # noqa: E402


class Params(object):
    data_is_imgs = img_model = subsample_input = False
    frame_sizes = [64]
    discrim_steps, gen_steps, gp_lambda = 5, 1, 10.0
    no_mean_discrim_loss = no_mean_gen_loss = True


def setup(b):
    ops.PACKS.clear()
    torch.manual_seed(100)
    gen, dis = Gen().cuda(), Discrim(cond_dim=0).cuda()
    init(gen, "xavier")
    init(dis, "xavier")
    gan = CondGan(gen=gen, discrims=[dis])
    losses = MixedGanLoss(g_loss=WassersteinGanLoss(), d_loss=WassersteinGanLoss())
    optD = FusedAdam(dis.parameters(), lr=1e-4, betas=(0.5, 0.9))
    optG = FusedAdam(gen.parameters(), lr=1e-4, betas=(0.5, 0.9))
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.rand(b, 16, 3, 64, 64, device="cuda", generator=g) * 2 - 1      # loader order (B, T, C, H, W)
    return gan, losses, optD, optG, x


def time_calls(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def iteration_ms(b, graphed, steps, warmup):
    gan, losses, optD, optG, x = setup(b)
    dev = torch.device("cuda", 0)
    if graphed:
        step = GraphedTrainStep(gan, optD, optG, Params(), losses, dev)
        fn = lambda: step(x, [])                                     # noqa: E731
        warmup = max(warmup, step.warmup + 1)                        # eager warm-ups and the capture are untimed
    else:
        fn = lambda: train_iteration(gan, x, [], dev, optD, optG, Params(), losses, end2end=False)   # noqa: E731
    return time_calls(fn, steps, warmup)


def penalty_us(b, S, launches):
    """fwd + bwd of mean_b (||g_b|| - 1)^2: the kernels against pow / sum / sqrt / mean and their autograd backward"""
    g = torch.randn(b, S, device="cuda") / S ** 0.5
    gout = torch.tensor(10.0, device="cuda")

    def fused():
        out, norms = K.gp_norm_fwd(g)
        K.gp_norm_bwd(g, norms, gout)

    def aten():
        gr = g.detach().requires_grad_(True)
        p = ((gr.pow(2).sum(dim=1).sqrt() - 1) ** 2).mean()
        torch.autograd.grad(p, gr, gout)
    res = {"fused": [], "aten": []}
    for _ in range(3):                                               # alternate, three rounds each
        res["fused"].append(1000.0 * time_calls(fused, launches, 10))
        res["aten"].append(1000.0 * time_calls(aten, launches, 10))
    return {k: min(v) for k, v in res.items()}, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_tgan_train_step.json"))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batches", default="64,256,1024")
    ap.add_argument("--penalty-batch", type=int, default=256)
    ap.add_argument("--launches", type=int, default=200)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit))
    rows = []
    for b in [int(s) for s in a.batches.split(",")]:
        row = {"b": b}
        try:
            for graphed in (False, True):
                row["ms_graph" if graphed else "ms_eager"] = iteration_ms(b, graphed, a.steps, a.warmup)
                torch.cuda.empty_cache()
        except torch.cuda.OutOfMemoryError:
            row["oom"] = True
            torch.cuda.empty_cache()
        for k in ("eager", "graph"):
            if "ms_" + k in row:
                row["videos_per_s_" + k] = 1000.0 * b / row["ms_" + k]
        print(json.dumps(row))
        rows.append(row)
    S = 3 * 16 * 64 * 64
    best, rounds = penalty_us(a.penalty_batch, S, a.launches)
    pen = {"b": a.penalty_batch, "S": S, "us_fused": best["fused"], "us_aten": best["aten"],
           "aten_over_fused": best["aten"] / best["fused"], "rounds_us": rounds, "launches_per_round": a.launches,
           "fused_GBps": 3 * a.penalty_batch * S * 4 / (best["fused"] * 1e-6) / 1e9}
    print(json.dumps(pen))
    rec = {"what": "TGAN WGAN-GP recipe iteration (5 penalised critic steps + 1 G step, FusedAdam), eager vs one CUDA "
                   "graph, 3x16x64x64 clips; fused penalty kernels vs the ATen composition (fwd + bwd, best of 3 "
                   "alternating rounds)",
           "card": name, "power_limit": limit, "steps": a.steps, "warmup": a.warmup, "rows": rows,
           "largest_b": max([r["b"] for r in rows if "ms_graph" in r] or [0]), "penalty": pen}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    print("wrote %s" % a.out)


if __name__ == "__main__":
    main()
