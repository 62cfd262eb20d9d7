"""TEST INFRASTRUCTURE ONLY -- the gradient penalty of the TGAN / TCWYT video critic on top of
oracle/families_oracle.py (plain functional PyTorch, CPU or any device, any float dtype).

The reference's only TGAN recipe (scripts/run_tgan.sh:17) is the WGAN loss with a gradient penalty, lambda = 10.
At HEAD the reference cannot run it: its _gradient_penalty unpacks `u, c, _ = discrim(...)` and VideoDiscrim returns
a 0-d tensor (models/tcwyt/video_discrim.py:57).  So the penalty here is RESTATED from the reference source
(gan/losses.py:135-186 with a scalar critic as the only output) and is not pinned by a live-reference golden
fixture, unlike the penalty-free iterations of oracle/families_oracle.py, which these functions reproduce exactly
when gp_lambda == 0.

Running statistics: every BatchNorm call updates its buffers in the order the iteration makes the calls (G forward,
D(fake), D(real), D(x_hat) of the penalty, D(fake) of the G phase); the updated buffers are returned.
"""
import torch

import oracle.families_oracle as O


def draw_gp_alpha(B):
    """gan/losses.py:140-145 (oracle.txt2vid_oracle.draw_gp_alphas for one level): torch.rand(B,1,1,1,1) on the
    CPU generator"""
    return torch.rand(B, 1, 1, 1, 1)


class _Chain(object):
    """state dict whose BatchNorm buffers follow the calls made with it (nb=None: buffers are not tracked)"""

    def __init__(self, sd, track):
        self.sd, self.track = sd, track

    def call(self, fn, *args):
        nb = {} if self.track else None
        out = fn(self.sd, *args, nb=nb)
        if nb:
            self.sd = dict(self.sd)
            self.sd.update(nb)
        return out

    def buffers(self):
        return {k: v.detach().clone() for k, v in self.sd.items() if "running_" in k}


def video_discrim_gp(sd, real, fake, cond=None, alpha=None, nb=None):
    """gan/losses.py:135-186 for the scalar VideoDiscrim: x_hat = alpha * real + (1 - alpha) * fake per sample (the
    caption too, with the same alpha, when the critic is conditional: both pairs carry the same caption here), d D /
    d x_hat with create_graph=True (only the clip's gradient is kept, :178), non-zero-centred
    mean_b (||g_b|| - 1)^2.  alpha: (B,1,1,1,1), drawn by draw_gp_alpha when None."""
    B = real.size(0)
    if alpha is None:
        alpha = draw_gp_alpha(B)
    a = alpha.to(device=real.device, dtype=real.dtype).clone().requires_grad_(True)
    ax = a.expand_as(real)
    xh = ax * real + (1 - ax) * fake
    ins, ch = [xh], None
    if cond is not None:
        ac = a.view(-1, 1).expand_as(cond)
        ch = ac * cond + (1 - ac) * cond
        ins.append(ch)
    out = O.video_discrim(sd, xh, ch, nb=nb)
    g = torch.autograd.grad([out], ins, [torch.ones_like(out)], create_graph=True, retain_graph=True)[0]
    return torch.mean((g.reshape(B, -1).norm(2, dim=1) - 1) ** 2)


def tgan_iteration(sd_g, sd_d, x, z, gp_lambda=0.0, alpha=None, track_buffers=False):
    """oracle.families_oracle.tgan_iteration plus the video critic's gradient penalty (lossD += gp_lambda * gp);
    gp_lambda = 0 gives that function's results bit for bit."""
    g, d = _Chain(sd_g, track_buffers), _Chain(sd_d, track_buffers)
    fake = g.call(O.tgan_gen, z)
    d_fake, d_real = d.call(O.video_discrim, fake.detach()), d.call(O.video_discrim, x)
    lossD = O.wgan_d(d_fake, d_real)
    gp = None
    if gp_lambda:
        gp = d.call(lambda sd, nb=None: video_discrim_gp(sd, x, fake.detach(), None, alpha, nb=nb))
        lossD = lossD + gp_lambda * gp
    lossD.backward()
    gD = {k: v.clone() for k, v in O.grads_of(sd_d).items()}
    for v in sd_d.values():
        v.grad = None
    lossG = O.wgan_g(d.call(O.video_discrim, fake))
    lossG.backward()
    out = {"lossD": float(lossD), "lossG": float(lossG), "fake": fake.detach(), "gD": gD, "gG": O.grads_of(sd_g),
           "d_real": float(d_real), "d_fake": float(d_fake), "gp": None if gp is None else float(gp)}
    if track_buffers:
        out["buffers_D"], out["buffers_G"] = d.buffers(), g.buffers()
    return out


def tcwyt_iteration(sd_g, sd_v, sd_f, sd_m, sd_map, x, z, cond, gp_lambda=0.0, alpha=None):
    """oracle.families_oracle.tcwyt_iteration plus the video critic's gradient penalty.  As in the reference's
    discrim_forward (cond_gan.py:34-87), the penalty joins that critic's own loss before the average over the three
    critics: lossD = (l_video + gp_lambda * gp + l_frame + l_motion) / 3.  The frame and motion critics read FrameMap
    features, not the interpolated clip, and take no penalty (the reference cannot penalise them either)."""
    fake = O.tcwyt_gen(sd_g, z, cond)

    def d_all(vid):
        m = O.frame_map(sd_map, vid)
        return [O.video_discrim(sd_v, vid, cond), O.frame_discrim(sd_f, cond, m), O.motion_discrim(sd_m, cond, m)]
    real_o, fake_o = d_all(x), d_all(fake.detach())
    terms = [O.ralsgan_d(f, r) for f, r in zip(fake_o, real_o)]
    gp = None
    if gp_lambda:
        gp = video_discrim_gp(sd_v, x, fake.detach(), cond, alpha)
        terms[0] = terms[0] + gp_lambda * gp
    lossD = sum(terms) / 3
    lossD.backward()
    gD = {}
    for name, sd in (("video", sd_v), ("frame", sd_f), ("motion", sd_m), ("map", sd_map)):
        gD[name] = {k: v.clone() for k, v in O.grads_of(sd).items()}
        for v in sd.values():
            v.grad = None
    fake_o2 = d_all(fake)
    lossG = sum(O.ralsgan_g(f, r.detach()) for f, r in zip(fake_o2, real_o)) / 3
    lossG.backward()
    return {"lossD": float(lossD), "lossG": float(lossG), "fake": fake.detach(), "gD": gD, "gG": O.grads_of(sd_g),
            "gp": None if gp is None else float(gp)}
