"""Time one TGAN critic step (scripts/run_tgan.sh:17: WGAN loss, FusedAdam) with and without the gradient penalty
(lambda = 10) on one GPU, at b = 64, 256 and 1024 clips of 3x16x64x64 (each size that fits), with CUDA events; then,
in a separate run, a torch.profiler breakdown of the penalised step by kernel.  Prints the card's name and power
limit, and appends one JSON line with everything to --out.

Usage: python scripts/critic_gp_step.py [--out profiles/r03_critic_gp_step.json] [--steps 10] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from txt2vid_b200.gan import WassersteinGanLoss, _gradient_penalty  # noqa: E402
from txt2vid_b200.optim import FusedAdam  # noqa: E402
from txt2vid_b200.tgan import Discrim  # noqa: E402
from txt2vid_b200.util import init  # noqa: E402

LAMBDA = 10.0


def card():
    name, limit = torch.cuda.get_device_name(0), None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        if out:
            name, limit = [s.strip() for s in out.split(",")[:2]]
    except (OSError, subprocess.SubprocessError):
        pass
    return name, limit


def make_step(dis, opt, real, fake, gp):
    loss = WassersteinGanLoss()

    def step():
        dis.zero_grad()
        lossD = loss.discrim_loss(fake=dis(x=fake), real=dis(x=real))
        if gp:
            lossD = lossD + LAMBDA * _gradient_penalty(dis, real_x=real, fake_x=fake)
        lossD.backward()
        opt.step()
        return lossD
    return step


def time_step(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def setup(b):
    torch.manual_seed(100)
    dis = Discrim(cond_dim=0).cuda()
    init(dis, "xavier")
    opt = FusedAdam(dis.parameters(), lr=1e-4, betas=(0.0, 0.9))
    g = torch.Generator(device="cuda").manual_seed(7)
    real = torch.rand(b, 3, 16, 64, 64, device="cuda", generator=g) * 2 - 1
    fake = torch.rand(b, 3, 16, 64, 64, device="cuda", generator=g) * 2 - 1
    return dis, opt, real, fake


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_critic_gp_step.json"))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batches", default="64,256,1024")
    ap.add_argument("--profile-batch", type=int, default=256)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    name, limit = card()
    print("card: %s, power limit %s" % (name, limit))
    rows = []
    for b in [int(s) for s in a.batches.split(",")]:
        row = {"b": b}
        try:
            for gp in (False, True):
                dis, opt, real, fake = setup(b)
                ms = time_step(make_step(dis, opt, real, fake, gp), a.steps, a.warmup)
                row["ms_gp" if gp else "ms_plain"] = ms
                del dis, opt, real, fake
                torch.cuda.empty_cache()
        except torch.cuda.OutOfMemoryError:
            row["oom"] = True
            torch.cuda.empty_cache()
        if "ms_gp" in row:
            row["gp_over_plain"] = row["ms_gp"] / row["ms_plain"]
            row["clips_per_s_gp"] = 1000.0 * b / row["ms_gp"]
        print(json.dumps(row))
        rows.append(row)
    # kernel breakdown of the penalised step, profiler on, in a run of its own
    from torch.profiler import ProfilerActivity, profile
    dis, opt, real, fake = setup(a.profile_batch)
    step = make_step(dis, opt, real, fake, True)
    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize()
    n = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            step()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t > 0:
            per[ev.key] = per.get(ev.key, 0.0) + t / 1000.0 / n
    top = sorted(per.items(), key=lambda kv: -kv[1])[:20]
    for k, ms in top:
        print("%9.3f ms/step  %s" % (ms, k[:110]))
    rec = {"what": "TGAN critic step (WGAN, FusedAdam) with / without the gradient penalty, lambda 10, 3x16x64x64 clips",
           "card": name, "power_limit": limit, "steps": a.steps, "warmup": a.warmup, "rows": rows,
           "profile_batch": a.profile_batch, "profile_ms_per_step": {k: round(v, 4) for k, v in top}}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    print("wrote %s" % a.out)


if __name__ == "__main__":
    main()
