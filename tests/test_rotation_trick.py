"""CPU tests of the rotation trick (opt-in extension, no reference counterpart): the float32 restatement of
tests/rotation_oracle.py against float64 autograd through the paper's transform, its rules for degenerate rows, and the
module surface of VectorQuantizer.rotation_trick."""
import inspect

import numpy as np
import pytest
import torch

from rotation_oracle import F32, coefficients, paper_grad_f64, rotate_grad


def _rows(n, d, seed, spread=0.3):
    """x, c near x (a code the row was assigned to), g: (N, D) float32"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g) * (1 + torch.rand(n, 1, generator=g) * 4)
    c = x * (0.5 + torch.rand(n, 1, generator=g)) + spread * x.norm(dim=-1, keepdim=True) / d ** 0.5 * torch.randn(n, d, generator=g)
    c[: n // 4] = torch.randn(n // 4, d, generator=g)                 # unrelated codes: any angle
    m = n // 3 - n // 4                                                # nearly opposite codes: t around 0.08
    c[n // 4: n // 3] = -0.8 * x[n // 4: n // 3] + 0.35 * x[n // 4: n // 3].norm(dim=-1, keepdim=True) / d ** 0.5 * torch.randn(m, d, generator=g)
    return x, c, torch.randn(n, d, generator=g)


@pytest.mark.parametrize("d", [3, 64, 256, 2048])
@pytest.mark.parametrize("lam", [0.0, 0.37])
def test_restatement_matches_float64_autograd(d, lam):
    n = 400 if d < 2048 else 64
    x, c, g = _rows(n, d, 10 + d)
    got = rotate_grad(x.unsqueeze(0), c.unsqueeze(0), g.unsqueeze(0), F32(lam))[0].double()
    want, rot = paper_grad_f64(x, c, g, lam)
    assert (rot - c.double()).abs().max() <= 1e-12 * c.abs().max()       # the transform's forward value is c
    xd, cd = x.double(), c.double()
    t = 1 + (xd * cd).sum(-1) / (xd.norm(dim=-1) * cd.norm(dim=-1))
    s = cd.norm(dim=-1) / xd.norm(dim=-1)
    scale = s * g.double().abs().amax(-1) + lam * (xd.abs().amax(-1) + cd.abs().amax(-1))
    keep = t >= 0.05
    assert keep.sum() >= n // 2
    err = (got - want).abs().amax(-1) / scale
    assert err[keep].max().item() <= 1e-4, err[keep].max().item()


def test_degenerate_rows_follow_the_pinned_rules():
    """zero x rows and zero c rows take the straight-through gradient (alpha 1, beta lam, gamma -lam); c = -2x rows (t
    at or next to 0: a + b is then exactly 0) take h = 0, the reflection s (g - 2 (u.g) u) + lam (x - c); all finite"""
    d, lam = 37, F32(0.25)
    x, c, g = _rows(12, d, 5)
    x[0:3] = 0
    c[3:6] = 0
    c[6:12] = -2 * x[6:12]
    xr, cr, gr = (t.numpy().astype(F32) for t in (x, c, g))
    alpha, beta, gamma, t = coefficients(xr, cr, gr, lam)
    assert (alpha[:6] == 1).all() and (beta[:6] == lam).all() and (gamma[:6] == -lam).all()
    assert (np.abs(t[6:]) <= 2 ** -22).all()
    gx = rotate_grad(x.unsqueeze(0), c.unsqueeze(0), g.unsqueeze(0), lam)[0]
    assert torch.isfinite(gx).all()
    ste = (g + lam * x) - lam * c
    assert torch.equal(gx[:6], ste[:6].float())
    xd, gd = x[6:].double(), g[6:].double()
    u = xd / xd.norm(dim=-1, keepdim=True)
    refl = 2 * (gd - 2 * (u * gd).sum(-1, keepdim=True) * u) + float(lam) * (xd - c[6:].double())
    torch.testing.assert_close(gx[6:].double(), refl, rtol=1e-5, atol=1e-5)


def test_null_gradient_and_no_loss_term():
    x, c, g = (t.unsqueeze(0) for t in _rows(40, 9, 3))
    assert torch.equal(rotate_grad(x, c, None, F32(0)), torch.zeros_like(x).abs())
    assert torch.equal(rotate_grad(x, c, None, F32(0.5)), rotate_grad(x, c, torch.zeros_like(x), F32(0.5)))


# ---- module surface --------------------------------------------------------------------------------------------------
def test_rotation_trick_is_a_plain_attribute_off_by_default():
    import vq_seg_b200 as V
    params = list(inspect.signature(V.VectorQuantizer.__init__).parameters)
    assert params == ["self", "dim", "num_embeddings", "embedding_dim", "decay", "eps", "kmeans_init", "kmeans_iters",
                      "distance", "commitment_weight", "num_codebook"]
    with pytest.raises(TypeError):
        V.VectorQuantizer(dim=8, num_embeddings=16, rotation_trick=True)
    for distance in ("euclidean", "cosine"):
        m = V.VectorQuantizer(dim=8, num_embeddings=16, distance=distance)
        assert m.rotation_trick is False
        keys = list(m.state_dict())
        m.rotation_trick = True
        assert list(m.state_dict()) == keys
        m2 = V.VectorQuantizer(dim=8, num_embeddings=16, distance=distance)
        m2.load_state_dict(m.state_dict())
        assert m2.rotation_trick is False                    # not carried by the state_dict


def test_cpu_input_still_raises():
    import vq_seg_b200 as V
    m = V.VectorQuantizer(dim=16, num_embeddings=8).train()
    m.rotation_trick = True
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 16, 4, 4, requires_grad=True))


def test_gather_mode_carries_the_flag_in_training_only():
    from vq_seg_b200 import ops
    assert ops.gather_mode(True, None, True) == ops.MODE_TRAIN | ops.MODE_ROTATE
    assert ops.gather_mode(True, torch.float16, True) == ops.MODE_TRAIN_AMP | ops.MODE_ROTATE
    assert ops.gather_mode(True, torch.bfloat16, True) == ops.MODE_TRAIN_AMP_BF16 | ops.MODE_ROTATE
    assert ops.gather_mode(True, torch.bfloat16) == ops.MODE_TRAIN_AMP_BF16
    with pytest.raises(ValueError, match="training"):
        ops.gather_mode(False, None, True)
