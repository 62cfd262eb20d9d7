"""GAN orchestration and losses: mirror of txt2vid/gan/cond_gan.py and txt2vid/gan/losses.py.

Same classes, method names, keyword arguments and loss arithmetic.  What differs is underneath: the
discriminator / generator calls run on the sm_100a kernels, and the conditional D step reuses the real
trunk features for the mismatched-caption pair (the reference's `computed_features` shortcut is dead
code, tganv2_cond/discrim.py:35,40-41, so it recomputes an identical trunk pass).
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import hostrng, ops


def get_labels_for(x, label):
    """gan/losses.py:4-5 with the float fill torch >= 2 needs (SURVEY 8c shim 2)."""
    return torch.full(x.size(), float(label), device=x.device)


class MixedGanLoss(object):
    def __init__(self, g_loss=None, d_loss=None):
        self.g_loss = g_loss
        self.d_loss = d_loss

    def discrim_loss(self, fake=None, real=None):
        return self.d_loss.discrim_loss(fake=fake, real=real)

    def gen_loss(self, fake=None, real=None):
        return self.g_loss.gen_loss(fake=fake, real=real)


class LabelledGanLoss(object):
    """NOTE: the reference assigns fake_label <- real_label and real_label <- fake_label
    (gan/losses.py:26-27); kept, because it is the behaviour users of VanillaGanLoss / HingeGanLoss get."""

    def __init__(self, real_label=None, fake_label=None, underlying_loss=None):
        assert real_label is not None and fake_label is not None and underlying_loss is not None
        self.loss = underlying_loss
        self.fake_label = real_label
        self.real_label = fake_label

    def _compute_loss(self, x, label):
        return self.loss(x, get_labels_for(x, label))

    def discrim_loss(self, fake=None, real=None):
        return self._compute_loss(fake, self.fake_label) + self._compute_loss(real, self.real_label)

    def gen_loss(self, fake=None, real=None):
        return self._compute_loss(fake, self.real_label)


class VanillaGanLoss(LabelledGanLoss):
    def __init__(self, bce_loss=True, reduction='mean'):
        loss = nn.BCEWithLogitsLoss(reduction=reduction) if bce_loss else nn.CrossEntropyLoss(reduction=reduction)
        super().__init__(underlying_loss=loss, real_label=1, fake_label=0)


class HingeGanLoss(LabelledGanLoss):
    def __init__(self, margin=2.0):
        super().__init__(underlying_loss=nn.HingeEmbeddingLoss(margin=margin), real_label=1, fake_label=-1)


class WassersteinGanLoss(object):
    def discrim_loss(self, fake=None, real=None):
        if real.numel() == fake.numel():
            return ops.rel_loss([(real, fake, 1.0)], 1)          # mean(fake - real), one reduction kernel
        return -(real.mean() - fake.mean())

    def gen_loss(self, fake=None, real=None):
        return -fake.mean()


class RSGANLoss(object):
    """Relativistic standard GAN (gan/losses.py:74-85): BCE-with-logits against ones of (r - f) / (f - r),
    i.e. mean softplus(-(r - f))."""

    def __init__(self, bce_loss=True):
        self.bce = bce_loss
        if not bce_loss:
            self.loss = nn.CrossEntropyLoss()

    def _rel(self, a, b):
        if self.bce:
            return ops.rel_loss([(a, b, 1.0)], 0)                # mean softplus(b - a), one reduction kernel
        return self.loss(a - b, get_labels_for(a, 1))

    def discrim_loss(self, fake=None, real=None):
        return self._rel(real, fake)

    def gen_loss(self, fake=None, real=None):
        return self._rel(fake, real)


class RaSGANLoss(object):
    """The reference's RaSGANLoss reads self.fake_labels / self.real_labels, which it never defines
    (gan/losses.py:91-96): every call raises AttributeError.  Same here, with a clearer message."""

    def __init__(self, bce_loss=True):
        self.loss = nn.BCEWithLogitsLoss() if bce_loss else nn.CrossEntropyLoss()
        self.fake_label = 0
        self.real_label = 1

    def _broken(self):
        raise AttributeError("'RaSGANLoss' object has no attribute 'fake_labels' (unusable in the reference too: "
                             "txt2vid/gan/losses.py:95-96)")

    def discrim_loss(self, fake=None, real=None):
        self._broken()

    def gen_loss(self, fake=None, real=None):
        self._broken()


class RaLSGANLoss(object):
    """Relativistic average LSGAN (gan/losses.py:113-133)."""

    def discrim_loss(self, fake=None, real=None):
        return (torch.mean((real - torch.mean(fake) - 1) ** 2) + torch.mean((fake - torch.mean(real) + 1) ** 2)) / 2

    def gen_loss(self, fake=None, real=None):
        return (torch.mean((real - torch.mean(fake) + 1) ** 2) + torch.mean((fake - torch.mean(real) - 1) ** 2)) / 2


def fused_loss_mode(loss, which):
    """0 (RSGAN, BCE form) when `loss` -- the bound discrim_loss / gen_loss of a loss object (train/gan.py:156) --
    can be evaluated over all pyramid levels and prediction pairs by ONE reduction kernel (ops.rel_loss); None
    otherwise (the generic per-level composition of gan/cond_gan.py:51-61 is used)."""
    obj = getattr(loss, "__self__", None)
    if isinstance(obj, MixedGanLoss):
        obj = obj.d_loss if which == "d" else obj.g_loss
    if isinstance(obj, RSGANLoss) and obj.bce and getattr(loss, "__name__", "") == ("discrim_loss" if which == "d"
                                                                                   else "gen_loss"):
        return 0
    return None


def _gradient_penalty(discrim, real_x=None, real_xbar=None, fake_x=None, fake_xbar=None, real_cond=None,
                      fake_cond=None, zero_center=False, combine=torch.mean):
    """gan/losses.py:135-186.  alpha ~ U(0,1) per sample from the CPU generator (created on CPU, then moved,
    :140-145); only d/dx_hat is kept (:178); the second derivative runs through ops.Conv*F etc.  A critic that
    returns one tensor instead of the (uncond, cond, features) tuple (TGAN / TCWYT VideoDiscrim: the scalar mean
    of its output map) has that tensor as its only output."""
    B = real_x.size(0)
    assert real_x.dim() in (4, 5)
    alpha = hostrng.CURRENT.alpha(B, real_x.device)            # B draws from the CPU generator, as the reference

    def lerp(r, f):
        if not (r.requires_grad or f.requires_grad) and r.dtype == torch.float32:
            return ops.K.lerp_rows(r.contiguous(), f.contiguous(), alpha.reshape(-1).contiguous()).requires_grad_(True)
        a = alpha.view([B] + [1] * (r.dim() - 1))
        return (a * r + (1 - a) * f).requires_grad_(True)
    xh = lerp(real_x, fake_x)
    xbarh = None
    if real_xbar is not None and fake_xbar is not None:
        xbarh = lerp(real_xbar, fake_xbar)
    ch = None
    if real_cond is not None and fake_cond is not None:
        ch = lerp(real_cond, fake_cond)
    out = discrim(x=xh, cond=ch, xbar=xbarh)
    if isinstance(out, torch.Tensor):
        outs = [out]
    else:
        u, c, _ = out
        outs = [u] + ([c] if c is not None else [])
    ins = [xh] + ([ch] if ch is not None else []) + ([xbarh] if xbarh is not None else [])
    g = torch.autograd.grad(outputs=outs, inputs=ins, grad_outputs=[torch.ones_like(o) for o in outs],
                            create_graph=True, retain_graph=True, only_inputs=True)[0]
    if zero_center and combine is torch.sum and g.numel() % 8 == 0:
        return ops.DotF.apply(g.contiguous(), g.contiguous())        # sum_b ||g_b||^2, one reduction kernel
    # mean_b (||g_b|| - 1)^2 on the penalty kernels; ops.K lacks them only where tests put ops on a CPU spec
    if not zero_center and combine is torch.mean and g.dtype == torch.float32 and (g.numel() // B) % 4 == 0 \
            and hasattr(ops.K, "gp_norm_fwd"):
        return ops.GradNormPenaltyF.apply(g.contiguous())
    n2 = g.reshape(B, -1).pow(2).sum(dim=1)
    return combine(n2) if zero_center else combine((n2.sqrt() - 1) ** 2)


def gradient_penalty(discrim, real_x=None, real_xbar=None, fake_x=None, fake_xbar=None, real_cond=None,
                     fake_cond=None):
    """gan/losses.py:188-209: multi-scale D -> zero-centred penalty summed over samples and levels."""
    if not hasattr(discrim, 'sub_discrims'):
        return _gradient_penalty(discrim, real_x=real_x, real_xbar=real_xbar, fake_x=fake_x, fake_xbar=fake_xbar,
                                 real_cond=real_cond, fake_cond=fake_cond)
    total = []
    for i in range(len(real_x)):
        rc = fc = rxb = fxb = None
        if real_cond is not None:
            rc, fc = real_cond[i], fake_cond[i]
            rxb = real_xbar[i] if real_xbar is not None else None
            fxb = fake_xbar[i] if fake_xbar is not None else None
        total.append(_gradient_penalty(discrim.sub_discrims[i], real_x=real_x[i], real_xbar=rxb, real_cond=rc,
                                       fake_x=fake_x[i], fake_xbar=fxb, fake_cond=fc, zero_center=True,
                                       combine=torch.sum))
    out = total[0]
    for t in total[1:]:
        out = out + t
    return out


def _zero_grad(module):
    """module.zero_grad() of cond_gan.py:91,157; the product modules' conv weights keep persistent gradient buffers
    that the weight-gradient kernels accumulate into (ops.zero_grads)."""
    from . import ops
    ops.zero_grads(module)


class CondGan(object):
    """gan/cond_gan.py:7-217."""

    def __init__(self, gen=None, discrims=None, cond_encoder=None, discrim_names=None, sample_mapping=None,
                 discrim_lambdas=None):
        assert gen is not None and discrims is not None and len(discrims) >= 1
        if discrim_names is None:
            discrim_names = ['discrim-%d' % i for i in range(len(discrims))]
        self.gen = gen
        self.discrims = discrims
        self.sample_mapping = sample_mapping
        self.cond_encoder = cond_encoder
        self.discrim_names = discrim_names
        self.discrim_lambdas = discrim_lambdas

    def _map_input(self, x):
        return self.sample_mapping(x) if self.sample_mapping is not None and x is not None else None

    def _discrim_weighted_sum(self, losses):
        if isinstance(losses, (list, tuple)):
            if len(losses) == 1 and self.discrim_lambdas is None:
                return losses[0]                       # mean of one element
            losses = torch.stack(list(losses))
        if self.discrim_lambdas is None:
            return torch.mean(losses)
        return torch.sum(torch.tensor(self.discrim_lambdas, device=losses.device) * losses)

    @staticmethod
    def _mean_over_levels(loss, fakes, reals, idx):
        return torch.stack([loss(fake=f[idx], real=r[idx]) for f, r in zip(fakes, reals)]).mean()

    @staticmethod
    def _check_single_scale(discrim, cond, mapping):
        if cond is not None:
            raise ValueError("conditional single-scale critics (TCWYT) are not supported: %s was given captions"
                             % type(discrim).__name__)
        if mapping is not None:
            raise ValueError("single-scale critics with a sample mapping (TCWYT's FrameMap) are not supported")

    def _single_scale_forward(self, discrim, real, fake, loss, gp_lambda):
        """A critic without `sub_discrims` (TGAN's VideoDiscrim: one scalar per call) on the one-level lists
        multiscale_data gives.  D(real) runs before D(fake), as in the reference's discrim_forward: the BatchNorm
        running statistics see the calls in that order.  The penalty is the non-zero-centred mean of
        gan/losses.py:135-186."""
        real_pred = discrim(x=real[0]) if real is not None else None
        fake_pred = discrim(x=fake[0]) if fake is not None else None
        l = None
        if loss is not None and real_pred is not None and fake_pred is not None:
            l = loss(fake=fake_pred, real=real_pred)
            if gp_lambda > 0:
                l = l + gp_lambda * _gradient_penalty(discrim, real_x=real[0], fake_x=fake[0])
        return l, fake_pred, real_pred

    def discrim_forward(self, name=None, discrim=None, real=None, real_mapping=None, fake=None, fake_mapping=None,
                        real_cond=None, fake_cond=None, loss=None, gp_lambda=-1):
        """(x_r,c_r) / (x_r,c_f) / (x_f,c_r) pairs and their per-level loss average (cond_gan.py:34-87)."""
        if not hasattr(discrim, "sub_discrims"):
            self._check_single_scale(discrim, real_cond, real_mapping if real_mapping is not None else fake_mapping)
            return self._single_scale_forward(discrim, real, fake, loss, gp_lambda)
        fake_pred = real_pred = l = None
        if real_cond is not None and fake_cond is not None:
            pair = loss is not None and hasattr(discrim, "forward_pair") and real_mapping is None \
                and fake_mapping is None
            if pair:       # (x_r, c_r) and (x_f, c_r) through the shared trunk in one pass (no normalisation in D)
                real_cc, fake_cc = discrim.forward_pair(x_a=real, x_b=fake, cond_a=real_cond, cond_b=real_cond)
            else:
                real_cc = discrim(x=real, cond=real_cond, xbar=real_mapping)
            real_pred = real_cc
            if loss is not None:
                real_ic = discrim(x=real, cond=fake_cond, xbar=real_mapping,
                                  computed_features=[t[-1] for t in real_cc])
                if not pair:
                    fake_cc = discrim(x=fake, cond=real_cond, xbar=fake_mapping)
                mode = fused_loss_mode(loss, "d")
                if mode is not None:
                    # (mean_i L(f_u, r_u) + (mean_i L(f_c, r_c) + mean_i L(ric_c, r_c)) / 2) / 2 in one kernel
                    n = float(len(real_cc))
                    pairs = [(r[0], f[0], 0.5 / n) for f, r in zip(fake_cc, real_cc)]
                    pairs += [(r[1], f[1], 0.25 / n) for f, r in zip(fake_cc, real_cc)]
                    pairs += [(r[1], f[1], 0.25 / n) for f, r in zip(real_ic, real_cc)]
                    l = ops.rel_loss(pairs, mode)
                else:
                    l_u = self._mean_over_levels(loss, fake_cc, real_cc, 0)
                    l_c = (self._mean_over_levels(loss, fake_cc, real_cc, 1) +
                           self._mean_over_levels(loss, real_ic, real_cc, 1)) / 2
                    l = (l_u + l_c) / 2.0
        else:
            if real is not None and fake is not None and loss is not None and hasattr(discrim, "forward_pair") \
                    and real_mapping is None and fake_mapping is None:
                ra, fa = discrim.forward_pair(x_a=real, x_b=fake)
                real_pred, fake_pred = [r[0] for r in ra], [f[0] for f in fa]
            else:
                if real is not None:
                    real_pred = [r[0] for r in discrim(x=real, cond=None, xbar=real_mapping)]
                if fake is not None:
                    fake_pred = [f[0] for f in discrim(x=fake, cond=None, xbar=fake_mapping)]
            if loss is not None and fake_pred is not None and real_pred is not None:
                mode = fused_loss_mode(loss, "d")
                if mode is not None:
                    n = float(len(real_pred))
                    l = ops.rel_loss([(r, f, 1.0 / n) for f, r in zip(fake_pred, real_pred)], mode)
                else:
                    l = torch.stack([loss(fake=f, real=r) for f, r in zip(fake_pred, real_pred)]).mean()
        if l is not None and gp_lambda > 0:
            l = l + gp_lambda * gradient_penalty(discrim, real_x=real, real_xbar=real_mapping, fake_x=fake,
                                                 fake_xbar=fake_mapping, real_cond=real_cond, fake_cond=fake_cond)
        return l, fake_pred, real_pred

    def gen_step(self, fake=None, real_pred=None, cond=None, loss=None):
        """cond_gan.py:90-118 (unconditional branch: element [0] of each tuple -- the reference passes the
        tuples themselves and raises, cond_gan.py:102-106; documented adapter, SURVEY 8c.4)."""
        _zero_grad(self.gen)
        if self.cond_encoder is not None:
            self.cond_encoder.zero_grad()
        fake_mapping = self._map_input(fake)
        losses = []
        for r, name, discrim in zip(real_pred, self.discrim_names, self.discrims):
            if not hasattr(discrim, "sub_discrims"):
                self._check_single_scale(discrim, cond, fake_mapping)
                losses.append(loss(fake=discrim(x=fake[0]), real=r))
                continue
            fake_cc = discrim(x=fake, cond=cond, xbar=fake_mapping)
            mode = fused_loss_mode(loss, "g")
            pick = lambda t: t[0] if isinstance(t, (tuple, list)) else t
            fused = mode is not None
            n = float(len(fake_cc))
            if cond is None:
                if fused:        # RSGAN generator loss: softplus(real - fake): a = fake, b = real
                    losses.append(ops.rel_loss([(pick(ff), pick(rr), 1.0 / n) for ff, rr in zip(fake_cc, r)], mode))
                else:
                    losses.append(torch.stack([loss(fake=pick(ff), real=pick(rr))
                                               for ff, rr in zip(fake_cc, r)]).mean())
            elif fused:
                pairs = [(ff[0], rr[0], 0.5 / n) for ff, rr in zip(fake_cc, r)]
                pairs += [(ff[1], rr[1], 0.5 / n) for ff, rr in zip(fake_cc, r)]
                losses.append(ops.rel_loss(pairs, mode))
            else:
                l_u = self._mean_over_levels(loss, fake_cc, r, 0)
                l_c = self._mean_over_levels(loss, fake_cc, r, 1)
                losses.append((l_c + l_u) / 2.0)
        return self._discrim_weighted_sum(losses)

    def all_discrim_forward(self, fake=None, real=None, cond=None, loss=None, gp_lambda=-1):
        """cond_gan.py:121-154: mismatched captions = a non-identity permutation of the level-0 captions
        (numpy RNG), truncated per level."""
        losses, real_pred, fake_pred = [], [], []
        real_mapping, fake_mapping = self._map_input(real), self._map_input(fake)
        for name, discrim in zip(self.discrim_names, self.discrims):
            fake_cond = None
            if cond is not None:
                perm = hostrng.CURRENT.perm(cond[0].size(0), cond[0].device)
                shuffled = cond[0][perm]
                fake_cond = [shuffled[0:r.size(0)] for r in cond]
            l, f, r = self.discrim_forward(name=name, discrim=discrim, real=real, real_cond=cond,
                                           real_mapping=real_mapping, fake=fake, fake_cond=fake_cond,
                                           fake_mapping=fake_mapping, loss=loss, gp_lambda=gp_lambda)
            losses.append(l)
            fake_pred.append(f)
            real_pred.append(r)
        return losses, fake_pred, real_pred

    def discrim_step(self, real=None, fake=None, cond=None, loss=None, gp_lambda=-1):
        for discrim in self.discrims:
            _zero_grad(discrim)
        if self.cond_encoder is not None:
            self.cond_encoder.zero_grad()
        losses, _, _ = self.all_discrim_forward(real=real, fake=fake, cond=cond, loss=loss, gp_lambda=gp_lambda)
        return self._discrim_weighted_sum(losses)

    def count_params(self):
        from .util import count_params
        n = int(np.sum([count_params(d) for d in self.discrims])) + count_params(self.gen)
        if self.cond_encoder is not None:
            n += count_params(self.cond_encoder)
        if self.sample_mapping is not None:
            n += count_params(self.sample_mapping)
        return n

    def __call__(self, *args, **kwargs):
        return self.gen(*args, **kwargs)

    @property
    def discrims_params(self):
        return [d.parameters() for d in self.discrims]

    def save_dict(self):
        res = {'gen': self.gen.state_dict()}
        if self.cond_encoder is not None:
            res['cond'] = self.cond_encoder.state_dict()
        if self.sample_mapping is not None:
            res['sample_mapping'] = self.sample_mapping.state_dict()
        for name, discrim in zip(self.discrim_names, self.discrims):
            res[name] = discrim.state_dict()
        return res

    def load_from_dict(self, to_load):
        self.gen.load_state_dict(to_load['gen'])
        if 'cond' in to_load:
            assert self.cond_encoder is not None
            self.cond_encoder.load_state_dict(to_load['cond'])
        if 'sample_mapping' in to_load:
            assert self.sample_mapping is not None
            self.sample_mapping.load_state_dict(to_load['sample_mapping'])
        for name, discrim in zip(self.discrim_names, self.discrims):
            if name in to_load:
                discrim.load_state_dict(to_load[name])
