"""The rotation trick's gradient w.r.t. x, restated in numpy float32 in the order include/vqseg.h pins for
vqseg_rotate_bwd_f32, and the paper's transform in float64 autograd (Fifty et al., arXiv 2410.06424, §4.2).

Opt-in extension without a reference counterpart (parity unpinned): tests/test_rotation_trick.py checks the restatement
against the float64 transform, the GPU tests check the kernels bit for bit against the restatement."""
import numpy as np
import torch

F32 = np.float32


def _rows(t):
    """(N, D) float32 numpy rows of a (B, P, D) tensor (any strides, any device)"""
    return t.detach().cpu().float().reshape(-1, t.shape[-1]).numpy().astype(F32)


def _sum8(p):
    """row sums of (N, D) float32 products: eight chains a_l over d = l, l + 8, ... ascending, then
    ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7))"""
    n, d = p.shape
    a = np.zeros((8, n), F32)
    for j0 in range(0, d, 8):
        w = min(8, d - j0)
        a[:w] = a[:w] + p[:, j0:j0 + w].T
    return ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]))


def coefficients(x, c, g, lam):
    """(alpha, beta, gamma, t) per row of (N, D) float32 arrays; lam a float32 scalar"""
    lam = F32(lam)
    xx, cc, xc = _sum8(x * x), _sum8(c * c), _sum8(x * c)
    xg, cg = _sum8(x * g), _sum8(c * g)
    with np.errstate(all="ignore"):
        nx, nc = np.sqrt(xx), np.sqrt(cc)
        s = nc / nx
        rho = (xc / nx) / nc
        a, b = xg / nx, cg / nc
        t = F32(1) + rho
        h = np.where(t > 0, (a + b) / t, F32(0)).astype(F32)
        beta = ((s * ((F32(2) * b) - h)) / nx) + lam
        gamma = (-((s * h) / nc)) - lam
    deg = (xx == 0) | (cc == 0)
    alpha = np.where(deg, F32(1), s).astype(F32)
    beta = np.where(deg, lam, beta).astype(F32)
    gamma = np.where(deg, -lam, gamma).astype(F32)
    return alpha, beta, gamma, t


def rotate_grad(x, c, g, lam):
    """gx for (B, P, D) tensors x, c (the forward's quantize) and g (None: zeros); lam = coef_scale * coef in float32.
    Returns a float32 CPU tensor of x's shape (contiguous)."""
    xr, cr = _rows(x), _rows(c)
    gr = np.zeros_like(xr) if g is None else _rows(g)
    alpha, beta, gamma, _ = coefficients(xr, cr, gr, lam)
    gx = ((alpha[:, None] * gr) + (beta[:, None] * xr)) + (gamma[:, None] * cr)
    return torch.from_numpy(gx.astype(F32)).reshape(x.shape)


def lam_of(coef_scale, grad_mse):
    """the kernels' lam = fl(coef_scale * grad_mse), both rounded to float32 first (coef_scale travels as a C float)"""
    return F32(coef_scale) * F32(grad_mse)


def paper_grad_f64(x, c, g, lam):
    """float64 autograd through quantize = s (x - 2 (x.w) w + 2 (x.u) q^) with u, q^, w, s detached, plus
    0.5 lam |x - c|^2: rows of (N, D) tensors"""
    x = x.detach().double().clone().requires_grad_(True)
    c, g = c.detach().double(), g.detach().double()
    nx = x.detach().norm(dim=-1, keepdim=True)
    nc = c.norm(dim=-1, keepdim=True)
    u, qh = x.detach() / nx, c / nc
    w = (u + qh) / (u + qh).norm(dim=-1, keepdim=True)
    s = nc / nx
    rot = s * (x - 2 * (x * w).sum(-1, keepdim=True) * w + 2 * (x * u).sum(-1, keepdim=True) * qh)
    out = (rot * g).sum() + 0.5 * float(lam) * ((x - c) ** 2).sum()
    out.backward()
    return x.grad, rot.detach()
