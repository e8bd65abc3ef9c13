"""The rule the bf16 gather modes reproduce, pinned on the CPU: under bf16 autocast the reference's one-hot gather
`matmul(one_hot(idx).float(), weight)` (vq_img.py:169-170) is a bf16 matmul, so its code is bf16(E[idx]) rounded to
nearest even, the straight-through output is x + (float(bf16(E[idx])) - x) and the commitment loss is the fp32 mse
of that output.  cdist is on autocast's fp32 list: the indices are the fp32 ones."""
import pytest
import torch
import torch.nn.functional as F

from oracle import vq_oracle as O


def inputs(seed, b=2, c=64, h=9, w=7, k=150):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, c, h, w, generator=g), torch.randn(k, c, generator=g)


def bf16_rule(x, e, idx, training):
    """(quantize (B,C,H,W) fp32, loss (1,)) of the bf16-autocast forward, given the fp32 indices"""
    b, c, h, w = x.shape
    xv = x.reshape(b, c, h * w).permute(0, 2, 1)
    code = e[idx.reshape(b, -1)].bfloat16().float()
    q = xv + (code - xv) if training else code
    loss = F.mse_loss(q, xv).reshape(1) if training else torch.zeros(1)
    return q.permute(0, 2, 1).reshape(b, c, h, w), loss


def check(module, x, e, training):
    module.codebook.embedding.weight.data.copy_(e)
    module.train(training)
    with torch.autocast("cpu", dtype=torch.bfloat16):
        q, idx, loss, usage = module(x)
    ref = O.vq_forward(x, e, training)                       # fp32, no autocast
    assert torch.equal(idx, ref["embed_index"])
    assert torch.equal(usage, ref["code_usage"])
    want_q, want_loss = bf16_rule(x, e, ref["embed_index"], training)
    assert q.dtype == (torch.float32 if training else torch.bfloat16)   # eval: the matmul's own dtype
    assert torch.equal(q.detach().float(), want_q)
    assert loss.dtype == torch.float32 and torch.equal(loss.detach(), want_loss)
    # the rounding is visible at this scale: the rule is not the fp32 result under another name
    assert not torch.equal(want_q, ref["quantize"])


@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_oracle_one_hot_matmul_under_bf16_autocast(training):
    x, e = inputs(31)
    m = O.OracleVectorQuantizer(dim=x.shape[1], num_embeddings=e.shape[0])
    m.faithful_ops = True                                    # the literal one_hot + matmul of vq_img.py:169-170
    check(m, x, e, training)


@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_live_reference_under_bf16_autocast(ref_vq, training):
    if ref_vq is None:
        pytest.skip("no reference checkout (VQSEG_REF)")
    x, e = inputs(32)
    check(ref_vq.VectorQuantizer(dim=x.shape[1], num_embeddings=e.shape[0]), x, e, training)


def test_gather_mode_follows_the_autocast_dtype():
    from vq_seg_b200 import ops
    assert ops.gather_mode(True, None) == ops.gather_mode(True, False) == ops.MODE_TRAIN
    assert ops.gather_mode(False, None) == ops.MODE_EVAL
    assert ops.gather_mode(True, torch.float16) == ops.gather_mode(True, True) == ops.MODE_TRAIN_AMP
    assert ops.gather_mode(False, torch.float16) == ops.gather_mode(False, True) == ops.MODE_EVAL_AMP
    assert ops.gather_mode(True, torch.bfloat16) == ops.MODE_TRAIN_AMP_BF16
    assert ops.gather_mode(False, torch.bfloat16) == ops.MODE_EVAL_AMP_BF16
    with pytest.raises(ValueError):
        ops.gather_mode(True, torch.float32)
