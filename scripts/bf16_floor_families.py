"""bf16 floor of the TGAN / TCWYT direct-drive iterations: oracle/families_oracle.py under torch.autocast(bfloat16)
against the same oracle in fp32 (TF32 off) on the same weights and inputs (see scripts/bf16_floor.py).
Usage: python scripts/bf16_floor_families.py [device] [--gp] -> one JSON line per family; with --gp, one more line
per family for the same step with the video critic's gradient penalty (lambda = 10, tests/families_gp_oracle.py):
the floor of tests/test_critic_gradient_penalty.py (profiles/r03_bf16_floor_families_gp.json)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import families_gp_oracle as GP  # noqa: E402
import oracle.families_oracle as O  # noqa: E402
import test_families as T  # noqa: E402
from helpers import golden, l2rel  # noqa: E402


def worst_grad(ref, low):
    scale = max(float(v.norm()) for v in ref.values())
    w = 0.0
    for k, g in ref.items():
        if float(g.norm()) < T.ZERO_GRAD * scale:
            continue
        w = max(w, l2rel(low[k].float().cpu(), g.float().cpu()))
    return w


def gp_floors(device, dev_sd, ac, lam=10.0, gp_seed=4321):
    """the WGAN-GP TGAN step and the TCWYT step with the video critic's penalty, autocast(bf16) vs fp32"""
    fx = golden("tgan_B8.json")
    gen, dis = T.build_tgan()
    x, z = T._synth(fx["B"], 16, 64, fx["input_seed"]).to(device), torch.tensor(fx["z"]).to(device)
    torch.manual_seed(gp_seed)
    alpha = GP.draw_gp_alpha(fx["B"])
    runs = []
    for on in (False, True):
        with ac(on):
            runs.append(GP.tgan_iteration(O.leaves(dev_sd(gen)), O.leaves(dev_sd(dis)), x, z, lam, alpha))
    ref, low = runs
    mag = abs(ref["d_real"]) + abs(ref["d_fake"])
    wgan = lambda o: o["lossD"] - lam * o["gp"]
    print(json.dumps({"family": "tgan_B8_gp", "what": "oracle autocast(bf16) vs fp32 on %s, lambda %g" % (device, lam),
                      "gp_rel": abs(low["gp"] - ref["gp"]) / abs(ref["gp"]),
                      "lossD_over_critic_scale": abs(wgan(low) - wgan(ref)) / mag,
                      "lossG_over_critic_scale": abs(low["lossG"] - ref["lossG"]) / mag,
                      "fake": l2rel(low["fake"].float().cpu(), ref["fake"].cpu()),
                      "gradD_worst": worst_grad(ref["gD"], low["gD"]), "gradG_worst": worst_grad(ref["gG"], low["gG"])}))
    fx = golden("tcwyt_B4.json")
    mods = T.build_tcwyt()
    x = T._synth(fx["B"], 16, 48, fx["input_seed"]).to(device)
    z, cond = torch.tensor(fx["z"]).to(device), torch.tensor(fx["cond"]).to(device)
    torch.manual_seed(gp_seed)
    alpha = GP.draw_gp_alpha(fx["B"])
    runs = []
    for on in (False, True):
        with ac(on):
            runs.append(GP.tcwyt_iteration(*[O.leaves(dev_sd(m)) for m in mods], x, z, cond, lam, alpha))
    ref, low = runs
    rep = {"family": "tcwyt_B4_gp", "what": "oracle autocast(bf16) vs fp32 on %s, lambda %g" % (device, lam),
           "gp_rel": abs(low["gp"] - ref["gp"]) / abs(ref["gp"]),
           "lossD_rel": abs(low["lossD"] - ref["lossD"]) / abs(ref["lossD"]),
           "lossG_rel": abs(low["lossG"] - ref["lossG"]) / abs(ref["lossG"]),
           "fake": l2rel(low["fake"].float().cpu(), ref["fake"].cpu()),
           "gradG_worst": worst_grad(ref["gG"], low["gG"])}
    for n in ("video", "frame", "motion", "map"):
        rep["gradD_%s_worst" % n] = worst_grad(ref["gD"][n], low["gD"][n])
    print(json.dumps(rep))


def main():
    args = [a for a in sys.argv[1:] if a != "--gp"]
    device = args[0] if args else "cpu"
    if device != "cpu":
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    dev_sd = lambda m: {k: v.to(device) for k, v in m.state_dict().items()}
    ac = lambda on: torch.autocast(torch.device(device).type, dtype=torch.bfloat16, enabled=on, cache_enabled=False)
    # ---- TGAN
    fx = golden("tgan_B8.json")
    gen, dis = T.build_tgan()
    x, z = T._synth(fx["B"], 16, 64, fx["input_seed"]).to(device), torch.tensor(fx["z"]).to(device)
    runs = []
    for on in (False, True):
        with ac(on):
            runs.append(O.tgan_iteration(O.leaves(dev_sd(gen)), O.leaves(dev_sd(dis)), x, z))
    ref, low = runs
    mag = abs(ref["d_real"]) + abs(ref["d_fake"])
    print(json.dumps({"family": "tgan_B8", "what": "oracle autocast(bf16) vs fp32 on %s" % device,
                      "lossD_rel": abs(low["lossD"] - ref["lossD"]) / abs(ref["lossD"]),
                      "lossG_rel": abs(low["lossG"] - ref["lossG"]) / abs(ref["lossG"]),
                      "lossD_over_critic_scale": abs(low["lossD"] - ref["lossD"]) / mag,
                      "lossG_over_critic_scale": abs(low["lossG"] - ref["lossG"]) / mag,
                      "d_real_rel": abs(low["d_real"] - ref["d_real"]) / abs(ref["d_real"]),
                      "fake": l2rel(low["fake"].float().cpu(), ref["fake"].cpu()),
                      "gradD_worst": worst_grad(ref["gD"], low["gD"]), "gradG_worst": worst_grad(ref["gG"], low["gG"])}))
    # ---- TCWYT
    fx = golden("tcwyt_B4.json")
    mods = T.build_tcwyt()
    x = T._synth(fx["B"], 16, 48, fx["input_seed"]).to(device)
    z, cond = torch.tensor(fx["z"]).to(device), torch.tensor(fx["cond"]).to(device)
    runs = []
    for on in (False, True):
        with ac(on):
            runs.append(O.tcwyt_iteration(*[O.leaves(dev_sd(m)) for m in mods], x, z, cond))
    ref, low = runs
    rep = {"family": "tcwyt_B4", "what": "oracle autocast(bf16) vs fp32 on %s" % device,
           "lossD_rel": abs(low["lossD"] - ref["lossD"]) / abs(ref["lossD"]),
           "lossG_rel": abs(low["lossG"] - ref["lossG"]) / abs(ref["lossG"]),
           "fake": l2rel(low["fake"].float().cpu(), ref["fake"].cpu()),
           "gradG_worst": worst_grad(ref["gG"], low["gG"])}
    for n in ("video", "frame", "motion", "map"):
        rep["gradD_%s_worst" % n] = worst_grad(ref["gD"][n], low["gD"][n])
    print(json.dumps(rep))
    if "--gp" in sys.argv[1:]:
        gp_floors(device, dev_sd, ac)


if __name__ == "__main__":
    main()
