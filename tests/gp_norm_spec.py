"""TEST-ONLY executable specification of txt2vid_b200/kernels.py::gp_norm_fwd / gp_norm_bwd (t2v_gp_norm_fwd / _bwd) in
plain PyTorch, a companion of tests/cpu_kernels.py: same arguments and results.  Math in fp32, or in fp64 when g is
fp64.  Tests that put the product's ops on the CPU spec install it into cpu_kernels (see install()).  The product never
imports this file.
"""
import torch

import cpu_kernels

F32 = torch.float32


def gp_norm_fwd(g):
    """g (B, ...) -> (0-d mean_b (||g_b||_2 - 1)^2, norms (B,))"""
    B = g.shape[0]
    norms = g.to(torch.promote_types(g.dtype, F32)).reshape(B, -1).pow(2).sum(1).sqrt()
    return ((norms - 1) ** 2).mean(), norms


def gp_norm_bwd(g, norms, gout):
    """dg = gout * 2 (n_b - 1) / (n_b B) * g_b, zero on rows with n_b = 0"""
    B = g.shape[0]
    safe = torch.where(norms > 0, norms, torch.ones_like(norms))
    c = torch.where(norms > 0, gout.reshape(()) * 2 * (norms - 1) / (safe * B), torch.zeros_like(norms))
    return (c.view(B, 1) * g.reshape(B, -1)).reshape(g.shape).to(g.dtype)


def install(monkeypatch):
    """make cpu_kernels answer ops.K.gp_norm_fwd / gp_norm_bwd for the duration of a test"""
    monkeypatch.setattr(cpu_kernels, "gp_norm_fwd", gp_norm_fwd, raising=False)
    monkeypatch.setattr(cpu_kernels, "gp_norm_bwd", gp_norm_bwd, raising=False)
