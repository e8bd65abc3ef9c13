"""Residual vector quantization without a GPU: the CPU restatement (tests/rvq_oracle.py) against VectorQuantizer's oracle
at Q = 1 and against float64 autograd through the mathematical definition, and the module's surface (constructor,
state_dict keys, make_vq_module's num_quantizers key, the custom ops' fake implementations, no CPU fallback)."""
import pytest
import torch

import rvq_oracle as R
from oracle import vq_oracle as O


def _setup(q, k=40, shape=(2, 16, 4, 8), seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g)
    cbs = [torch.randn(k, shape[1], generator=g) * scale * 0.5 ** l for l in range(q)]
    return x, cbs


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("amp", [None, torch.float16, torch.bfloat16])
def test_q1_is_vector_quantizer(distance, training, amp):
    x, (e,) = _setup(1)
    got = R.rvq_forward(x, [e], training, 0.7, distance, amp)
    want = O.vq_forward(x, O.l2norm(e) if distance == "cosine" else e, training, 0.7, distance)
    assert torch.equal(got["idx"][0], want["embed_index"].reshape(2, -1))
    assert torch.equal(got["usage"], want["code_usage"])
    if amp is None:
        assert torch.equal(got["quantize"], want["quantize"])
        assert torch.equal(got["loss"], want["loss"])


@pytest.mark.parametrize("w", [1.0, 0.5])
def test_q1_backward_is_vector_quantizer(w):
    """numel a power of two and g_loss = 1: the coefficient is exact, so the fused multiply-add and vq_backward's two
    roundings agree"""
    x, (e,) = _setup(1, shape=(2, 16, 4, 8))
    f = R.rvq_forward(x, [e], True, w)
    g = torch.randn(f["S"].shape, generator=torch.Generator().manual_seed(5))
    gl = torch.ones(1)
    got = R.rvq_backward(f["A"], g, gl, w)
    xv = x.reshape(2, 16, -1).permute(0, 2, 1)
    want = O.vq_backward(xv, f["quantize"].reshape(2, 16, -1).permute(0, 2, 1), g, gl, w)
    assert torch.equal(got, want)


@pytest.mark.parametrize("q", [1, 2, 3, 8])
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_gradient_matches_float64_autograd(q, distance):
    """one straight-through over the sum of the codes plus each layer's commitment loss w * mse(q_l.detach(), r_l),
    differentiated in float64: the restated gx within 1e-6 of the row scale"""
    w, gl = 0.8, torch.tensor([1.3])
    x, cbs = _setup(q, shape=(2, 12, 5, 3), seed=q)
    f = R.rvq_forward(x, cbs, True, w, distance)
    g = torch.randn(f["S"].shape, generator=torch.Generator().manual_seed(7))
    got = R.rvq_backward(f["A"], g, gl, w)

    xv = x.reshape(2, 12, -1).permute(0, 2, 1).double().requires_grad_(True)
    cs = [f["codebooks"][l][f["idx"][l]].double() for l in range(q)]
    prev = torch.zeros_like(xv)
    s = sum(cs[1:], cs[0])
    quant = xv + (s - xv).detach()
    loss = 0
    for l in range(q):
        r = xv - prev
        ql = r + (cs[l] - r)
        loss = loss + w * torch.nn.functional.mse_loss(ql.detach(), r)
        prev = prev + cs[l]
    (quant * g.double()).sum().add(loss * gl.double().item()).backward()
    scale = xv.detach().abs().amax(-1, keepdim=True).clamp_min(1.0)
    assert ((got.double() - xv.grad).abs() / scale).max() < 1e-6


def test_decode_is_the_eval_sum():
    x, cbs = _setup(3)
    f = R.rvq_forward(x, cbs, False)
    assert torch.equal(R.rvq_decode(f["idx"], cbs), f["S"])


def test_fma32_rounds_once():
    import numpy as np
    a = np.float32(1 + 2 ** -12)
    b = np.float32(1 + 2 ** -12)
    c = np.float32(-1)
    exact = 2 ** -11 + 2 ** -24                 # a b + c, representable in float32
    assert R.fma32(a, b, c) == np.float32(exact)
    assert np.float32(a * b) + c != np.float32(exact)


def test_constructor_and_state_dict():
    import vq_seg_b200 as V
    torch.manual_seed(3)
    m = V.ResidualVectorQuantizer(16, 32, 3, commitment_weight=0.5, distance="cosine")
    assert [k for k in m.state_dict()] == [f"layers.{l}.codebook.embedding.weight" for l in range(3)]
    torch.manual_seed(3)
    singles = [V.VectorQuantizer(16, 32) for _ in range(3)]
    for l in range(3):
        assert torch.equal(m.layers[l].codebook.embedding.weight, singles[l].codebook.embedding.weight)
    assert isinstance(m.layers[0].codebook, V.CosinesimCodebook)
    assert m.num_quantizers == 3 and m.commitment_weight == 0.5 and m.amp_compat
    with pytest.raises(ValueError):
        V.ResidualVectorQuantizer(16, 32, 0)
    with pytest.raises(ValueError):
        m(torch.randn(2, 16, 4))


def test_factory_key():
    import vq_seg_b200 as V
    cfg = {"num_embeddings": [0, 16, 8], "distance": "euclidean", "num_quantizers": 4}
    mods = V.make_vq_module(cfg, [3, 8, 16, 32], 3)
    assert isinstance(mods[0], V.Identity)
    assert [type(m) for m in mods[1:]] == [V.ResidualVectorQuantizer] * 2
    assert mods[2].num_quantizers == 4 and mods[2].num_embeddings == 8
    assert cfg["num_quantizers"] == 4                          # the caller's config is left as it was
    plain = V.make_vq_module({"num_embeddings": 8}, [3, 8, 16], 2)
    assert all(type(m) is V.VectorQuantizer for m in plain)


def test_custom_ops_have_fake_impls():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from vq_seg_b200 import ops
    with FakeTensorMode():
        idx = torch.empty(3, 2, 20, dtype=torch.int64)
        out = ops.rvq_decode(idx, torch.empty(3, 8, 16), ops.MODE_EVAL)
        assert out.shape == (2, 20, 16) and out.stride() == (16 * 20, 1, 20)
        r = torch.empty(2, 16, 20).permute(0, 2, 1)
        q = torch.empty(2, 16, 20).permute(0, 2, 1)
        assert ops.rvq_stage(r, None, torch.empty(8, 16), None, r, q, None, None, idx, torch.empty(3, 8, dtype=torch.int64),
                             torch.empty(3), torch.empty(3), torch.empty(1), torch.empty(()), 2, ops.MODE_EVAL, 0,
                             1.0) is None


def test_no_cpu_fallback():
    import vq_seg_b200 as V
    m = V.ResidualVectorQuantizer(16, 8, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 16, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.get_output_from_indices(torch.zeros(1, 4, 4, 2, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        V.ops.rvq_decode(torch.zeros(2, 1, 4, dtype=torch.int64), torch.randn(2, 8, 16))
