"""TEST-ONLY executable specification of txt2vid_b200/kernels.py::bn_backward_backward (t2v_bn_bwd_bwd) in plain
PyTorch, a companion of tests/cpu_kernels.py: same argument meaning, layouts and rounding point (outputs rounded to
cpu_kernels.STORE).  Tests that put the product's ops on the CPU spec install it as
cpu_kernels.bn_backward_backward (see install()).  The product never imports this file.
"""
import torch

import cpu_kernels

F32 = torch.float32


def bn_backward_backward(dy, x, mean_invstd, scale_shift, ggx, ggamma, ggbeta, relu, up):
    """(dy, x, gamma) -> (dx, dgamma, dbeta) of bn_backward differentiated once more (up == 1), in the same
    sum-based form as the CUDA kernel; math in fp32, or in fp64 when the inputs are fp64."""
    assert up == 1
    C = x.shape[-1]
    dt = torch.promote_types(x.dtype, F32)
    mean, invstd = mean_invstd[:C].to(dt), mean_invstd[C:].to(dt)
    scale, shift = scale_shift[:C].to(dt), scale_shift[C:].to(dt)
    xf, q = x.to(dt).reshape(-1, C), ggx.to(dt).reshape(-1, C)
    m = torch.ones_like(xf)
    if relu:
        m = torch.where(xf * scale + shift > 0, m, m * (0.0 if relu == 1 else 0.2))
    g = dy.to(dt).reshape(-1, C) * m
    xhat = (xf - mean) * invstd
    P = xf.shape[0]
    sg, sgx = g.sum(0), (g * xhat).sum(0)
    sq, sqx, sqg = q.sum(0), (q * xhat).sum(0), (q * g).sum(0)
    gga = torch.zeros_like(sg) if ggamma is None else ggamma.to(dt)
    ggb = torch.zeros_like(sg) if ggbeta is None else ggbeta.to(dt)
    gdy = m * (scale * (q - sq / P - xhat * sqx / P) + gga * xhat + ggb)
    t = xhat * (sq * sg / P - sqg + 3 * sgx * sqx / P) + sqx * (sg / P - g) + sgx * (sq / P - q)
    gx = scale * invstd / P * t + gga * invstd * (g - sg / P - xhat * sgx / P)
    dgamma = invstd * (sqg - sq * sg / P - sqx * sgx / P)
    return gx.reshape(x.shape).to(cpu_kernels.STORE), gdy.reshape(x.shape).to(cpu_kernels.STORE), dgamma


def install(monkeypatch):
    """make cpu_kernels answer ops.K.bn_backward_backward for the duration of a test"""
    monkeypatch.setattr(cpu_kernels, "bn_backward_backward", bn_backward_backward, raising=False)
