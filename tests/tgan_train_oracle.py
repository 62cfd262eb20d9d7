"""TEST INFRASTRUCTURE ONLY -- one train() iteration of TGAN's WGAN-GP recipe (scripts/run_tgan.sh:17: WGAN loss,
gradient penalty lambda = 10, 5 critic steps per generator step, Adam) in plain functional PyTorch on state dicts, on
top of oracle/families_oracle.py, tests/families_gp_oracle.py and oracle.txt2vid_oracle.Adam.  Any float dtype; the
tests run it in fp64.

The calls follow gan/trainer.py:199-267 with CondGan's single-scale critic path:
  G forward, once (the fake clip every critic step reuses);
  discrim_steps times: D(real), D(fake.detach()), the penalty at a fresh alpha, backward, Adam on D;
  D(real) once more: the G phase's real_pred (no gradient; only the BatchNorm buffers move);
  D(fake), lossG = -D(fake), backward, Adam on G.
Every BatchNorm call updates its running statistics in that order.  The mean over critic steps is off
(--no_mean_discrim_loss defaults to True, trainer.py:27-28), so lossD is the sum of the critic steps' losses.
"""
import torch

import families_gp_oracle as GP
import oracle.families_oracle as O
from oracle.txt2vid_oracle import Adam


def _params(sd):
    return [k for k, v in sd.items() if v.requires_grad]


def _snapshot(sd):
    return {k: sd[k].detach().clone() for k in _params(sd)}


def recipe_iteration(sd_g, sd_d, x, z, alphas, gp_lambda=10.0, lr=1e-4, betas=(0.5, 0.9), opt_d=None, opt_g=None):
    """alphas: one (B,) draw per critic step (the CPU generator's torch.rand(B) at each penalty).  sd_* are updated in
    place (parameters by Adam, running statistics as the calls make them).  Returns per-critic-step losses, the first
    and the last critic step's and the G step's gradients, the parameters before / after and the buffers after the
    iteration."""
    opt_d = opt_d or Adam(_params(sd_d), lr, betas)
    opt_g = opt_g or Adam(_params(sd_g), lr, betas)
    params0D, params0G = _snapshot(sd_d), _snapshot(sd_g)
    g, d = GP._Chain(sd_g, True), GP._Chain(sd_d, True)
    fake = g.call(O.tgan_gen, z)
    steps = []
    gD = gD_first = None
    for alpha in alphas:
        for v in d.sd.values():
            v.grad = None
        d_real = d.call(O.video_discrim, x)
        d_fake = d.call(O.video_discrim, fake.detach())
        a = alpha.reshape(-1, 1, 1, 1, 1)
        gp = d.call(lambda sd, nb=None: GP.video_discrim_gp(sd, x, fake.detach(), None, a, nb=nb))
        lossD = O.wgan_d(d_fake, d_real) + gp_lambda * gp
        lossD.backward()
        gD = {k: v.clone() for k, v in O.grads_of(d.sd).items()}
        gD_first = gD_first if steps else gD
        opt_d.step(d.sd, gD)
        steps.append({"lossD": float(lossD), "d_real": float(d_real), "d_fake": float(d_fake), "gp": float(gp)})
    with torch.no_grad():
        d_real = d.call(O.video_discrim, x)
    for v in d.sd.values():
        v.grad = None
    lossG = O.wgan_g(d.call(O.video_discrim, fake))
    lossG.backward()
    gG = {k: v.clone() for k, v in O.grads_of(g.sd).items()}
    opt_g.step(g.sd, gG)
    return {"steps": steps, "lossD": sum(s["lossD"] for s in steps), "lossG": float(lossG), "real_pred": float(d_real),
            "fake": fake.detach(), "gD": gD, "gD_first": gD_first, "gG": gG, "params0D": params0D, "params0G": params0G,
            "paramsD": _snapshot(d.sd), "paramsG": _snapshot(g.sd), "buffers_D": d.buffers(), "buffers_G": g.buffers()}
