"""CPU transcription of the residual VQ restatement in include/vqseg.h (vqseg_rvq_stage_f32), on top of oracle.vq_oracle's
assignment -- the checker of vq_seg_b200.ResidualVectorQuantizer.

Opt-in extension without a reference counterpart (parity unpinned): every elementwise operation is one separately
rounded fp32 torch CPU operation, the gradient's fused multiply-add is rounded once (numpy float64 with round-to-odd,
then float32), and m_l is torch's mean, which the GPU's fixed two-stage reduction matches within the tolerance of the
existing mse checks."""
from typing import Optional, Sequence

import numpy as np
import torch

from oracle import vq_oracle as O


def nchw(t: torch.Tensor) -> torch.Tensor:
    """t's values in a (B, P, D) tensor of NCHW memory order (the strides the module's residual buffers have, which fix
    the summation order of l2norm)"""
    b, p, d = t.shape
    out = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32)
    out.copy_(t)
    return out


def round_code(c: torch.Tensor, amp: Optional[torch.dtype]) -> torch.Tensor:
    return c if amp is None else c.to(amp).to(torch.float32)


def fma32(a, b, c) -> np.ndarray:
    """fl(a * b + c) with ONE rounding, for float32 arrays: the product is exact in float64, the float64 sum is turned
    into round-to-odd (exact with TwoSum), which makes the final rounding to float32 the correctly rounded result"""
    a, b, c = (np.asarray(v, dtype=np.float64) for v in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    bits = s.view(np.int64)
    inexact_even = (err != 0) & ((bits & 1) == 0) & np.isfinite(s)
    toward = np.where(err > 0, np.inf, -np.inf)
    s = np.where(inexact_even, np.nextafter(s, toward), s)
    return s.astype(np.float32)


def rvq_forward(x: torch.Tensor, codebooks: Sequence[torch.Tensor], training: bool, commitment_weight: float = 1.0,
                distance: str = "euclidean", amp: Optional[torch.dtype] = None):
    """The restatement on CPU.  x (B, C, H, W); codebooks: Q (K, D) weights (cosine: renormalised here, as the module
    does in place every forward).  Returns a dict: quantize (B,C,H,W), S (B,P,D), idx (Q,B,P), loss (1,), usage (),
    layer_mse (Q,), layer_usage (Q,), A (B,P,D) or None (training), residuals [r_0 .. r_{Q-1}], codebooks (as used)."""
    x = x.to(torch.float32)
    b, c, h, w = x.shape
    xv = x.reshape(b, c, h * w).permute(0, 2, 1)
    r, s, a = xv, None, None
    idxs, mses, usages, counts_all, residuals, used = [], [], [], [], [], []
    for l, e in enumerate(codebooks):
        e = e.detach().float()
        residuals.append(r)
        if distance == "cosine":
            e = O.l2norm(e)
            idx = O.assign_cosine(r, e)
        else:
            idx = O.assign_euclidean(r, e)
        used.append(e)
        k = e.shape[0]
        cl = round_code(e[idx], amp)
        s = cl if l == 0 else s + cl
        if training:
            ql = r + (cl - r)
            mses.append(torch.nn.functional.mse_loss(ql, r).reshape(1))
            d = r - ql
            a = d if l == 0 else a + d
        counts = torch.bincount(idx.reshape(-1), minlength=k)
        counts_all.append(counts)
        usages.append(O.code_usage_from_counts(counts, k))
        idxs.append(idx)
        if l < len(codebooks) - 1:
            r = nchw(r - cl)
    q = xv + (s - xv) if training else s
    wt = torch.tensor(commitment_weight, dtype=torch.float32)
    loss = torch.zeros(1, dtype=torch.float32)
    layer_mse = torch.cat(mses) if training else torch.zeros(len(codebooks))
    if training and commitment_weight > 0:
        loss = mses[0] * wt
        for m in mses[1:]:
            loss = loss + m * wt
    allc = torch.stack(counts_all)
    usage = 100 * ((allc == 0).sum() / allc.numel())
    return dict(quantize=q.permute(0, 2, 1).reshape(b, c, h, w), S=s, idx=torch.stack(idxs), loss=loss, usage=usage,
                layer_mse=layer_mse, layer_usage=torch.stack(usages), A=a if training else None, residuals=residuals,
                codebooks=used)


def rvq_backward(a: torch.Tensor, grad_q: Optional[torch.Tensor], grad_loss: Optional[torch.Tensor],
                 commitment_weight: float) -> torch.Tensor:
    """gx = fma(coef, A, g), coef = fl(fl(2 / numel) * fl(g_loss * w)) (the arithmetic of vqseg_ste_bwd_f32 with a null
    q_ste and VectorQuantizer's autograd of `mse * w`), as a (B, P, D) tensor"""
    g = np.zeros(a.shape, np.float32) if grad_q is None else grad_q.detach().float().numpy()
    if grad_loss is None or not commitment_weight > 0:
        return torch.from_numpy(g.copy())
    gl = np.float32(grad_loss.reshape(()).item())
    gm = gl if commitment_weight == 1 else np.float32(gl * np.float32(commitment_weight))
    coef = np.float32(np.float32(2.0 / a.numel()) * gm)
    return torch.from_numpy(fma32(np.float32(coef), a.detach().numpy(), g))


def rvq_decode(idx: torch.Tensor, codebooks: Sequence[torch.Tensor], amp: Optional[torch.dtype] = None) -> torch.Tensor:
    """S from (Q, B, P) indices"""
    s = None
    for l, e in enumerate(codebooks):
        c = round_code(e.detach().float()[idx[l]], amp)
        s = c if l == 0 else s + c
    return s
