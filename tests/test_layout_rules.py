"""The ATen behaviour the kernels' layout-dependent choices restate, pinned over the layout catalogue (tests/layouts.py)
on the CPU, so that a torch release that changes it is noticed before any GPU run:

  (a) F.normalize(x, dim=-1) takes its summation order from the reduced dim's stride alone: a view with sD == 1 gives
      the result of its packed copy (ATen's vectorised last-dim order) whatever sB and sP are; any other stride gives
      one sequential chain acc = fl(acc + fl(v * v)) in channel order.  vqseg_l2norm_f32 chooses by the same rule.
  (b) torch.cdist of a batch of B >= 2 views equals cdist of the packed copy bit for bit (ATen copies both operands
      to contiguous memory first), so every Euclidean result may be compared with the same call on the packed copy.
  (c) layouts.make returns views of one storage with the documented strides, never a copy.
"""
import pytest
import torch
import torch.nn.functional as F

import layouts

CASES = layouts.cases()


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_catalogue_builds_views_with_the_documented_strides(case):
    layout, s = case
    shape = layouts.SHAPES[s][0]
    full, x = layouts.make(layout, shape, 1)
    v = layouts.bpd(x, full, layout)
    assert v.shape == (shape[0], shape[2] * shape[3], shape[1])
    # the same construction on the same seed gives the same values
    assert torch.equal(layouts.bpd(layouts.make(layout, shape, 1)[1]), v)
    # the view reads the seeded storage: writing through the storage shows up in the view
    before = v.clone()
    full.add_(1.0)
    assert torch.equal(v, before + 1.0)


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_normalize_order_follows_the_reduced_dims_stride(case):
    layout, s = case
    full, x = layouts.make(layout, layouts.SHAPES[s][0], 2)
    v = layouts.bpd(x, full, layout)
    got = F.normalize(v, p=2, dim=-1)
    if v.stride(2) == 1:
        assert torch.equal(got, F.normalize(v.contiguous(), p=2, dim=-1)), "sD == 1: the packed copy's result"
    else:
        assert torch.equal(got, layouts.seq_chain_normalize(v)), "sD != 1: one sequential chain"


def test_the_two_normalize_orders_differ_on_the_catalogue():
    """(a) is not vacuous: on these inputs the vectorised and the sequential order disagree for many rows, so a kernel
    that used the wrong one would fail the bit-exact l2norm tests"""
    full, x = layouts.make("nhwc_batch_step", layouts.SHAPES["odd"][0], 2)
    v = layouts.bpd(x, full, "nhwc_batch_step")
    vec, seq = F.normalize(v, p=2, dim=-1), layouts.seq_chain_normalize(v)
    assert (vec != seq).any(-1).sum().item() > v.shape[0] * v.shape[1] // 8
    full, x = layouts.make("map_1x1", layouts.SHAPES["px1"][0], 2)
    v = layouts.bpd(x, full, "map_1x1")
    assert not torch.equal(F.normalize(v, p=2, dim=-1), layouts.seq_chain_normalize(v))


@pytest.mark.parametrize("case", [c for c in CASES if layouts.SHAPES[c[1]][0][0] >= 2], ids=layouts.case_id)
def test_cdist_of_a_batch_equals_cdist_of_the_packed_copy(case):
    layout, s = case
    shape, k = layouts.SHAPES[s]
    full, x = layouts.make(layout, shape, 3)
    v = layouts.bpd(x, full, layout)
    e = torch.randn(k, shape[1], generator=torch.Generator().manual_seed(4))
    assert torch.equal(torch.cdist(v, e, p=2), torch.cdist(v.contiguous(), e, p=2))
