"""The segmentation head beyond the per-pixel kernels' limits (K > 32 classes, D > 382 features): the register-tiled
map and backward kernels (csrc/seghead_tiled.cu) behind vqseg_seghead_map_f32 / vqseg_seghead_map_bwd_f32.
Bars: the Euclidean map bit-equal to the exact scorer's distance for every class (so within 1 ulp of CPU torch.cdist
for B >= 2), indices and counts equal to the exact scorer, the tiled and per-pixel kernels identical where both apply,
gradients no further from a float64 evaluation than max(1e-5, 2 x CPU fp32 autograd), and the module against the
CPU oracle."""
import os
import sys

import pytest
import torch
from torch import nn

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import cases  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


def rel_to_max(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def ulp_close(a, b, n_ulp):
    return ((a - b).abs() <= n_ulp * torch.finfo(torch.float32).eps * b.abs()).all().item()


def squares_close(dist, live, xv, e, n_eps):
    """|dist^2 - live^2| <= n_eps * eps * (|x|^2 + |e|^2): the two augmented chains a few roundings apart"""
    scale = xv.double().pow(2).sum(-1, keepdim=True) + e.double().pow(2).sum(-1)
    diff = (dist.double().pow(2) - live.double().pow(2)).abs()
    return (diff <= n_eps * torch.finfo(torch.float32).eps * scale).all().item()


def features(seed, b, c, p, k, nchw=True):
    """post-ReLU decoder features as a (B, P, C) view (NCHW map or packed rows) and prototypes near feature rows,
    with one pixel equal to a prototype and, for K > 1, two identical prototypes"""
    g = torch.Generator().manual_seed(seed)
    x = torch.relu(torch.randn(b, c, p, generator=g))
    rows = x.permute(0, 2, 1).reshape(-1, c)
    e = rows[torch.randint(0, rows.shape[0], (k,), generator=g)] + 0.1 * torch.rand(k, c, generator=g)
    if k > 1:
        e[k - 1] = e[0]
    x[b - 1, :, p // 2] = e[k // 2]
    xv = x.permute(0, 2, 1) if nchw else x.permute(0, 2, 1).contiguous()
    return xv, e


def cpu_sim(xn, w):
    """the oracle's similarity map: einsum('n d, e d -> n e') over the flattened rows on the CPU"""
    b, p, d = xn.shape
    return torch.einsum("n d, e d -> n e", xn.cpu().contiguous().view(b * p, d), w.cpu()).view(b, p, -1)


EUCLID_K = (1, 33, 150, 1000)
EUCLID_D = (1, 382, 383, 766, 767, 768, 1024, 2048)


@pytest.mark.parametrize("d", EUCLID_D)
@pytest.mark.parametrize("k", EUCLID_K)
def test_tiled_euclidean_map_is_the_exact_scorer(dev, k, d):
    from vq_seg_b200 import ops
    nchw = (EUCLID_K.index(k) + EUCLID_D.index(d)) % 2 == 0
    b, p = (2, 181) if k * d <= 150 * 1024 else (2, 67)          # pixel counts that are not a multiple of the tile
    xv, e = features(1000 + k + d, b, d, p, k, nchw)
    xg, eg = xv.to(dev), e.to(dev)
    dist, idx, counts = ops.seghead_map(xg, eg, False, ops.SEGHEAD_TILED)
    assert dist.shape == (b, p, k) and dist.stride() == (k * p, 1, p)
    i_ex, c_ex = ops.assign(xg, eg, None, ops.ALGO_EXACT)
    assert torch.equal(idx, i_ex) and torch.equal(counts, c_ex)
    assert torch.equal(counts.cpu(), torch.bincount(idx.cpu().reshape(-1), minlength=k))
    g = torch.Generator().manual_seed(k * d)
    cols = sorted(set([0, k // 2, k - 1] + torch.randint(0, k, (4,), generator=g).tolist()))
    for j in cols:
        keys = ops.assign_keys(xg, eg[j:j + 1].contiguous(), None, 0, ops.ALGO_EXACT)
        _, dj, _ = ops.unpack_keys(keys, 1)
        assert torch.equal(dist[:, :, j], dj), (j, (dist[:, :, j] != dj).sum().item())
    # against torch.cdist itself.  Up to 768 augmented terms MKL's K-blocking is the same for every GEMM shape: 1 ulp
    # (ATen's CPU sqrt is MKL VML), except where the pixel sits on a prototype and both sides are cancellation noise of
    # the augmented form.  Beyond, MKL picks its blocking by the shape of the product (384-term blocks, what the exact
    # scorer restates, with >= 512 codes; other splits with fewer codes): the squared distances then differ by a few
    # roundings at the magnitude of |x|^2 + |e|^2, which is many ulp of a small distance
    live = torch.cdist(xv.contiguous(), e, p=2)
    if d + 2 <= 768:
        far = live > 1e-3 * live.max()
        assert ulp_close(dist.cpu()[far], live[far], 1)
    assert squares_close(dist.cpu(), live, xv, e, 8)


def test_tiled_euclidean_map_single_image_within_4_ulp(dev):
    from vq_seg_b200 import ops
    xv, e = features(5, 1, 300, 257, 70)
    dist, idx, _ = ops.seghead_map(xv.to(dev), e.to(dev), False, ops.SEGHEAD_AUTO)
    # B == 1: ATen skips cdist's contiguous copy and sums |x|^2 of the strided rows in another order: a few roundings
    # of |x|^2 apart, i.e. a few ulp of the distance except for pixels close to a prototype
    live = torch.cdist(xv, e, p=2)
    far = live > 0.5 * live.max()
    assert ulp_close(dist.cpu()[far], live[far], 4)
    assert squares_close(dist.cpu(), live, xv, e, 8)
    assert torch.equal(idx, ops.assign(xv.to(dev), e.to(dev), None, ops.ALGO_EXACT)[0])


@pytest.mark.parametrize("k,d", [(1, 5), (40, 64), (150, 383), (64, 512), (33, 1024), (1000, 256)])
def test_tiled_cosine_map_is_the_exact_ip_scorer(dev, k, d):
    from vq_seg_b200 import ops
    xv, e = features(77 + k + d, 2, d, 150, k, nchw=k % 2 == 0)
    xn = ops.l2norm_rows(xv.to(dev))
    w = e.to(dev).contiguous()
    ops.l2norm_rows_(w)
    sim, idx, counts = ops.seghead_map(xn, w, True, ops.SEGHEAD_TILED)
    i_ex, c_ex = ops.assign(xn, w, None, ops.ALGO_EXACT | ops.METRIC_IP)
    assert torch.equal(idx, i_ex) and torch.equal(counts, c_ex)
    assert rel_to_max(sim.cpu(), cpu_sim(xn, w)) <= 1e-6


@pytest.mark.parametrize("name", ["cos2_d512", "cos2_d1024"])
def test_tiled_cosine_map_matches_golden_indices(dev, name):
    from vq_seg_b200 import ops
    x, e = cases.COSINE2_CASES[name]()
    rec = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_cosine_v2.pt"),
                     weights_only=False)["cosine2"][name]
    b, c = x.shape[:2]
    xn = ops.l2norm_rows(x.to(dev).reshape(b, c, -1).permute(0, 2, 1))
    w = e.to(dev).contiguous()
    ops.l2norm_rows_(w)
    sim, idx, _ = ops.seghead_map(xn, w, True, ops.SEGHEAD_TILED)
    assert torch.equal(idx.cpu().reshape(-1), rec["idx_train"].to(torch.int64).reshape(-1))
    assert rel_to_max(sim.cpu(), cpu_sim(xn, w)) <= 1e-6


@pytest.mark.parametrize("k,d", [(1, 1), (3, 32), (7, 100), (32, 382), (20, 255)])
def test_tiled_and_per_pixel_kernels_agree(dev, k, d):
    from vq_seg_b200 import ops
    xv, e = features(300 + k + d, 3, d, 211, k, nchw=d % 2 == 0)
    xg, eg = xv.to(dev), e.to(dev)
    a = ops.seghead_score_map(xg, eg, ops.SEGHEAD_TILED)
    p = ops.seghead_score_map(xg, eg, ops.SEGHEAD_PIXEL)
    assert torch.equal(a[0], p[0]) and torch.equal(a[2], p[2]) and torch.equal(a[3], p[3])
    # (one class and a pixel on its prototype: 1 - 0 / 0 is NaN for both kernels, as for the reference's torch ops)
    nan = a[1].isnan()
    assert torch.equal(nan, p[1].isnan()) and rel_to_max(a[1][~nan], p[1][~nan]) <= 1e-6
    xn = ops.l2norm_rows(xg)
    w = eg.clone()
    ops.l2norm_rows_(w)
    a = ops.seghead_map(xn, w, True, ops.SEGHEAD_TILED)
    p = ops.seghead_map(xn, w, True, ops.SEGHEAD_PIXEL)
    assert all(torch.equal(u, v) for u, v in zip(a, p))
    # backward: the tiled kernels against float64 of the same mathematics, bar max(1e-5, 2 x the CPU fp32 error) (the
    # two kernels sum x sum_k w - sum_k w e in different orders, so they are not compared with each other bit for bit)
    g = torch.randn(a[0].shape, generator=torch.Generator().manual_seed(k))
    dm, sc, _, _ = ops.seghead_score_map(xg, eg)
    runs = [("dist", xg, eg, dm, None), ("score", xg, eg, dm, sc), ("cosine", xn, w, a[0], None)]
    if k == 1:
        runs.pop(1)          # one class on its prototype: the score is NaN (1 - 0 / 0) and so is every gradient
    for kind, xx, ww, m, s_ in runs:
        (gx64, ge64), (gx32, ge32) = _grad_bar(kind, xx.cpu(), ww.cpu(), g)
        gx, ge = ops.seghead_map_bwd(g.to(dev), m, xx, ww, kind == "cosine", s_, ops.SEGHEAD_TILED)
        for ours, ref32, ref64 in ((gx, gx32, gx64), (ge, ge32, ge64)):
            bar = max(1e-5, 2 * rel_to_max(ref32.double(), ref64))
            assert rel_to_max(ours.cpu().double(), ref64) <= bar, (kind, rel_to_max(ours.cpu().double(), ref64), bar)


def _grad_bar(kind, xv, e, gout):
    """(float64 gradients, CPU fp32 autograd gradients) of sum(gout * map) for the three head maps"""
    def run(x, w):
        x = x.clone().requires_grad_(True)
        w = w.clone().requires_grad_(True)
        if kind == "cosine":
            m = torch.einsum("bpd,kd->bpk", torch.nn.functional.normalize(x, dim=-1), w)
        else:
            m = torch.cdist(x, w, p=2)
            if kind == "score":
                m = torch.softmax(1 - m / m.sum(-1, keepdim=True), dim=-1)
        (m * gout.to(m.dtype)).sum().backward()
        return x.grad, w.grad
    return run(xv.double(), e.double()), run(xv.contiguous(), e)


@pytest.mark.parametrize("kind", ["dist", "score", "cosine"])
@pytest.mark.parametrize("k,d", [(150, 256), (64, 512), (33, 767), (1000, 64)])
def test_tiled_gradients(dev, kind, k, d):
    from vq_seg_b200 import ops
    xv, e = features(900 + k + d, 2, d, 140, k, nchw=d != 512)
    if kind == "cosine":
        e = torch.nn.functional.normalize(e, dim=-1)
    gout = torch.randn(2, 140, k, generator=torch.Generator().manual_seed(d))
    (gx64, ge64), (gx32, ge32) = _grad_bar(kind, xv, e, gout)
    xg, eg = xv.to(dev), e.to(dev)
    if kind == "cosine":
        m, _, _ = ops.seghead_map(ops.l2norm_rows(xg), eg, True)
        gx, ge = ops.seghead_map_bwd(gout.to(dev), m, xg, eg, True, None, ops.SEGHEAD_TILED)
    elif kind == "score":
        dm, sc, _, _ = ops.seghead_score_map(xg, eg)
        gx, ge = ops.seghead_map_bwd(gout.to(dev), dm, xg, eg, False, sc, ops.SEGHEAD_TILED)
    else:
        dm, _, _ = ops.seghead_map(xg, eg)
        gx, ge = ops.seghead_map_bwd(gout.to(dev), dm, xg, eg, False, None, ops.SEGHEAD_TILED)
    for ours, ref32, ref64 in ((gx, gx32, gx64), (ge, ge32, ge64)):
        bar = max(1e-5, 2 * rel_to_max(ref32.double(), ref64))
        assert rel_to_max(ours.cpu().double(), ref64) <= bar, (rel_to_max(ours.cpu().double(), ref64), bar)


def _head64(x, w, variant, idx):
    """the oracle head's training forward in float64 (quantize, score, loss) with the indices given"""
    b, c, h, wd = x.shape
    xv = x.reshape(b, c, h * wd).permute(0, 2, 1)
    if variant == "cosine":
        score = torch.einsum("bpd,kd->bpk", torch.nn.functional.normalize(xv, dim=-1), w)
    else:
        score = torch.cdist(xv, w, p=2)
        score = 1 - score / score.sum(-1, keepdim=True)
    score = score.permute(0, 2, 1).reshape(b, -1, h, wd)
    score = torch.sigmoid(score) if variant == "sigmoid" else torch.softmax(score, dim=1)
    q = w.detach()[idx.reshape(b, -1)]
    loss = torch.nn.functional.mse_loss(q, xv).reshape(1)
    quantize = (xv + (q - xv).detach()).permute(0, 2, 1).reshape(b, c, h, wd)
    return quantize, score, loss


@pytest.mark.parametrize("k,d", [(150, 256), (64, 512)])
@pytest.mark.parametrize("variant", ["softmax2d", "sigmoid", "cosine"])
def test_wide_module_against_oracle(dev, k, d, variant):
    import vq_seg_b200 as V
    from oracle.seghead_oracle import OracleVQSegmentationHead
    kw = dict(dim=d, num_embeddings=k)
    if variant == "sigmoid":
        kw["activation"] = nn.Sigmoid
    if variant == "cosine":
        kw["distance"] = "cosine"
    g = torch.Generator().manual_seed(k + d)
    x = torch.relu(torch.randn(2, d, 12, 10, generator=g))
    e = x.permute(0, 2, 3, 1).reshape(-1, d)[torch.randperm(240, generator=g)[:k]] + 0.05 * torch.rand(k, d, generator=g)
    m = V.VQSegmentationHead(**kw).to(dev)
    o = OracleVQSegmentationHead(**kw)
    m.codebook.embedding.weight.data.copy_(e.to(dev))
    o.embedding.weight.data.copy_(e)
    m.train(); o.train()
    xg = x.to(dev).requires_grad_(True)
    xc = x.clone().requires_grad_(True)
    a, b = m(xg), o(xc)
    gs = torch.randn(b[1].shape, generator=g)
    gq = torch.randn(b[0].shape, generator=g)
    ((a[1] * gs.to(dev)).sum() + (a[0] * gq.to(dev)).sum() + a[3].sum()).backward()
    ((b[1] * gs).sum() + (b[0] * gq).sum() + b[3].sum()).backward()
    assert torch.equal(a[2].cpu(), b[2]) and torch.equal(a[0].detach().cpu(), b[0].detach())
    assert a[4].item() == b[4].item()
    assert rel_to_max(a[1].detach().cpu(), b[1].detach()) <= 1e-5
    assert abs(a[3].item() - b[3].item()) <= 1e-5 * max(abs(b[3].item()), 1e-30)
    # gradients against float64 of the same mathematics, bar max(1e-5, 2 x the CPU fp32 error)
    x64 = x.double().requires_grad_(True)
    w64 = o.embedding.weight.detach().double().requires_grad_(True)     # (renormalised in place for cosine)
    r = _head64(x64, w64, variant, b[2])
    ((r[1] * gs.double()).sum() + (r[0] * gq.double()).sum() + r[2].sum()).backward()
    for ours, ref32, ref64 in ((xg.grad, xc.grad, x64.grad),
                               (m.codebook.embedding.weight.grad, o.embedding.weight.grad, w64.grad)):
        bar = max(1e-5, 2 * rel_to_max(ref32.double(), ref64))
        assert rel_to_max(ours.cpu().double(), ref64) <= bar, (rel_to_max(ours.cpu().double(), ref64), bar)
    m.eval(); o.eval()
    with torch.no_grad():
        a, b = m(x.to(dev)), o(x)
    assert torch.equal(a[2].cpu(), b[2])
    assert torch.equal(a[0].cpu(), b[0]) if variant != "cosine" else rel_to_max(a[0].cpu(), b[0]) <= 1e-6
    assert rel_to_max(a[1].cpu(), b[1]) <= 1e-5


def test_wide_kmeans_init_matches_oracle(dev):
    import vq_seg_b200 as V
    from oracle.seghead_oracle import OracleVQSegmentationHead
    g = torch.Generator().manual_seed(64)
    x = torch.relu(torch.randn(2, 96, 24, 20, generator=g))
    init = torch.randperm(960, generator=g)[:64]
    m = V.VQSegmentationHead(dim=96, num_embeddings=64, kmeans_init=True, kmeans_iters=5).to(dev)
    o = OracleVQSegmentationHead(dim=96, num_embeddings=64, kmeans_init=True, kmeans_iters=5)
    m.codebook.kmeans_init_indices = init.to(dev)
    o.kmeans_init_indices = init
    m.train(); o.train()
    a = m(x.to(dev)); b = o(x)
    assert m.codebook.initted and torch.equal(m.codebook.embedding.weight.detach().cpu(), o.embedding.weight.detach())
    assert torch.equal(a[2].cpu(), b[2]) and torch.equal(a[0].detach().cpu(), b[0].detach())


def test_seghead_custom_ops_opcheck(dev):
    from vq_seg_b200 import ops
    xv, e = features(8, 2, 40, 50, 37)
    xg, eg = xv.to(dev), e.to(dev)
    tu = ("test_schema", "test_faketensor")
    torch.library.opcheck(ops.seghead_map, (xg, eg, False, ops.SEGHEAD_TILED), test_utils=tu)
    torch.library.opcheck(ops.seghead_map, (ops.l2norm_rows(xg), eg, True, ops.SEGHEAD_AUTO), test_utils=tu)
    torch.library.opcheck(ops.seghead_score_map, (xg, eg, ops.SEGHEAD_AUTO), test_utils=tu)
    dm, sc, _, _ = ops.seghead_score_map(xg, eg)
    gout = torch.randn(dm.shape, device=dev)
    torch.library.opcheck(ops.seghead_map_bwd, (gout, dm, xg, eg, False, sc, ops.SEGHEAD_AUTO),
                          test_utils=tu)
    torch.library.opcheck(ops.seghead_map_bwd, (gout, dm, xg, eg, False, None, ops.SEGHEAD_TILED),
                          test_utils=tu)


def test_per_pixel_algo_still_refuses_wide_shapes(dev):
    from vq_seg_b200 import ops
    with pytest.raises(RuntimeError):
        ops.seghead_map(torch.randn(1, 64, 400, device=dev), torch.randn(3, 400, device=dev), False, ops.SEGHEAD_PIXEL)
    dist, _, _ = ops.seghead_map(torch.randn(1, 64, 400, device=dev), torch.randn(3, 400, device=dev))
    assert dist.shape == (1, 64, 3)
