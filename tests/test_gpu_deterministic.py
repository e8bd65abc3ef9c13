"""Reproducible gradients under torch.use_deterministic_algorithms(True).

The segmentation head's prototype gradient (VQSEG_SEGHEAD_DETERMINISTIC: fixed pixel slices, plain stores, a
fixed-order sum of the partials) must not change from call to call, with other work on the device, or with the
layout of the features; the eval-mode codebook gradient must equal CPU index_add_ bit for bit; and a small model
with a VectorQuantizer (k-means init, EMA) and a VQSegmentationHead must train to bit-identical parameters."""
import os
import subprocess
import sys
import textwrap

import pytest
import torch
from torch import nn

import layouts
from test_gpu_seghead_wide import _grad_bar, features, rel_to_max

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(3, 32), (32, 382), (150, 256), (64, 512), (1000, 64)]       # (classes K, features D)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


@pytest.fixture
def deterministic():
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=warn)


def _maps(kind, xv, e):
    """(e, map, score) as the head's backward receives them (cosine: unit prototypes, the similarity map)"""
    from vq_seg_b200 import ops
    if kind == "cosine":
        e = torch.nn.functional.normalize(e, dim=-1)
        m, _, _ = ops.seghead_map(ops.l2norm_rows(xv), e, True)
        return e, m, None
    if kind == "score":
        dm, sc, _, _ = ops.seghead_score_map(xv, e)
        return e, dm, sc
    dm, _, _ = ops.seghead_map(xv, e)
    return e, dm, None


def _busy(side, dev):
    """an unrelated kernel on a side stream while the backward runs: it takes SMs and shifts the block schedule"""
    with torch.cuda.stream(side):
        a = torch.randn(3072, 3072, device=dev)
        for _ in range(3):
            a = torch.tanh(a @ a * 1e-3)
    return a


@pytest.mark.parametrize("kind", ["dist", "score", "cosine"])
@pytest.mark.parametrize("k,d", SHAPES)
def test_prototype_gradient_is_reproducible(dev, kind, k, d):
    from vq_seg_b200 import ops
    shape = (2, d, 12, 13)                         # 312 pixels: several tiles and several pixel slices
    full, x = layouts.make("nhwc", shape, 500 + k + d, dev)
    views = {"nhwc": layouts.bpd(x, full, "nhwc"), "nchw": layouts.bpd(x.contiguous())}    # one data, two layouts
    views["packed"] = views["nchw"].contiguous()
    e = views["packed"].reshape(-1, d)[torch.arange(k, device=dev) * 7 % 312].clone() + 0.05
    e, m, sc = _maps(kind, views["nchw"], e)
    g = torch.randn(m.shape, generator=torch.Generator().manual_seed(k + d)).to(dev)
    cos = kind == "cosine"
    det = ops.SEGHEAD_AUTO | ops.SEGHEAD_DETERMINISTIC
    side = torch.cuda.Stream()
    ref_gx, ref_ge = ops.seghead_map_bwd(g, m, views["nchw"], e, cos, sc, det)
    for _ in range(3):
        busy = _busy(side, dev)
        gx, ge = ops.seghead_map_bwd(g, m, views["nchw"], e, cos, sc, det)
        torch.cuda.current_stream().wait_stream(side)
        del busy
        assert torch.equal(ge, ref_ge) and torch.equal(gx, ref_gx)
    for lay in ("nhwc", "packed"):
        _, ge_l = ops.seghead_map_bwd(g, m, views[lay], e, cos, sc, det)
        assert torch.equal(ge_l, ref_ge), lay
    gx_atomic, ge_atomic = ops.seghead_map_bwd(g, m, views["nchw"], e, cos, sc, ops.SEGHEAD_AUTO)
    assert torch.equal(ref_gx, gx_atomic)
    # the float64 bar of the tiled kernels' gradient test: max(1e-5, 2 x the CPU fp32 autograd error)
    xc = views["nchw"].cpu()
    (gx64, ge64), (gx32, ge32) = _grad_bar(kind, xc, e.cpu(), g.cpu())
    bar = max(1e-5, 2 * rel_to_max(ge32.double(), ge64))
    assert rel_to_max(ref_ge.cpu().double(), ge64) <= bar, (rel_to_max(ref_ge.cpu().double(), ge64), bar)


@pytest.mark.parametrize("kind", ["dist", "score", "cosine"])
def test_per_pixel_blocks_walking_several_tiles(dev, kind):
    """32 classes x 382 features over 98 304 pixels: the partials' 32 MiB bound makes each block of the per-pixel
    kernel walk two tiles (read-add-store into its own slice)"""
    from vq_seg_b200 import ops
    xv, e = features(41, 4, 382, 128 * 192, 32)
    xv, e = xv.to(dev), e.to(dev)
    e, m, sc = _maps(kind, xv, e)
    g = torch.randn(m.shape, generator=torch.Generator().manual_seed(3)).to(dev)
    cos = kind == "cosine"
    det = ops.SEGHEAD_PIXEL | ops.SEGHEAD_DETERMINISTIC
    assert ops._native.lib().vqseg_seghead_map_bwd_workspace_bytes(4 * 128 * 192, 382, 32, det) == 384 * 32 * 382 * 4
    side = torch.cuda.Stream()
    gx0, ge0 = ops.seghead_map_bwd(g, m, xv, e, cos, sc, det)
    busy = _busy(side, dev)
    gx1, ge1 = ops.seghead_map_bwd(g, m, xv, e, cos, sc, det)
    torch.cuda.current_stream().wait_stream(side)
    del busy
    _, ge2 = ops.seghead_map_bwd(g, m, xv.contiguous(), e, cos, sc, det)
    assert torch.equal(ge0, ge1) and torch.equal(gx0, gx1) and torch.equal(ge0, ge2)
    gxa, gea = ops.seghead_map_bwd(g, m, xv, e, cos, sc, ops.SEGHEAD_PIXEL)
    assert torch.equal(gx0, gxa)
    # the same sums as the atomic kernel up to fp32 reordering: against float64 of the same mathematics on the GPU
    x64, e64, g64 = xv.double(), e.double(), g.double()
    if cos:
        xn = x64 / x64.norm(dim=-1, keepdim=True).clamp_min(1e-12)
        ge64 = torch.einsum("bpk,bpd->kd", g64, xn)
    else:
        d64 = m.double()
        if sc is not None:
            s64 = sc.double()
            gt = s64 * (g64 - (g64 * s64).sum(-1, keepdim=True))
            ssum = d64.sum(-1, keepdim=True)
            g64 = ((gt * d64).sum(-1, keepdim=True) / ssum - gt) / ssum
        w = torch.where(d64 == 0, torch.zeros_like(d64), g64 / d64)
        ge64 = e64 * w.sum((0, 1))[:, None] - torch.einsum("bpk,bpd->kd", w, x64)
    assert rel_to_max(ge0.double(), ge64) <= max(1e-5, 2 * rel_to_max(gea.double(), ge64))


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("channels_last", [False, True])
def test_eval_codebook_gradient_is_cpu_index_add(dev, deterministic, distance, channels_last):
    import vq_seg_b200 as V
    torch.manual_seed(5)
    k, c = 300, 64
    m = V.VectorQuantizer(dim=c, num_embeddings=k, distance=distance).to(dev).eval()
    m.codebook.embedding.weight.data.normal_()
    x = torch.randn(2, c, 24, 20, device=dev)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    q, idx, _, _ = m(x)
    gq = torch.randn(q.shape, device=dev)
    (q * gq).sum().backward()
    rows = gq.permute(0, 2, 3, 1).reshape(-1, c).cpu()
    ref = torch.zeros(k, c).index_add_(0, idx.reshape(-1).cpu(), rows)
    assert torch.equal(m.codebook.embedding.weight.grad.cpu(), ref)


def _head_step(m, x, gs, one):
    q, s, _, loss, _ = m(x)
    torch.autograd.backward((s, loss), (gs, one))
    out = (s.detach().clone(), x.grad.clone(), m.codebook.embedding.weight.grad.clone())
    x.grad = None
    m.codebook.embedding.weight.grad = None
    return out


@pytest.mark.parametrize("variant", ["softmax", "sigmoid", "cosine"])
@pytest.mark.parametrize("k", [3, 150])
def test_head_gradients_repeat_and_graph_capture(dev, deterministic, variant, k):
    import vq_seg_b200 as V
    torch.manual_seed(17 + k)
    c = 48
    kw = {"distance": "cosine"} if variant == "cosine" else {}
    if variant == "sigmoid":
        kw["activation"] = nn.Sigmoid
    m = V.VQSegmentationHead(dim=c, num_embeddings=k, **kw).to(dev).train()
    m.codebook.embedding.weight.data.normal_()
    w0 = m.codebook.embedding.weight.detach().clone()
    x = torch.relu(torch.randn(2, c, 20, 24, device=dev)).requires_grad_(True)
    gs = torch.randn(2, k, 20, 24, device=dev)
    one = torch.ones(1, device=dev)

    def step(fn):
        m.codebook.embedding.weight.data.copy_(w0)      # the cosine head renormalises its weights in place
        return _head_step(m if fn is None else fn, x, gs, one)

    a, b = step(None), step(None)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    gm = torch.cuda.make_graphed_callables(m, (x.detach().clone().requires_grad_(True),), allow_unused_input=True)
    for _ in range(2):
        m.codebook.embedding.weight.grad = None
        graphed = step(gm)
        for u, v in zip(a, graphed):
            assert torch.equal(u, v)


_TRAIN = textwrap.dedent("""
    import sys, torch
    from torch import nn
    sys.path.insert(0, sys.argv[1])
    import vq_seg_b200 as V
    torch.use_deterministic_algorithms(True)
    torch.backends.cudnn.benchmark = False
    dev = torch.device("cuda:0")

    def run(classes):
        torch.manual_seed(123)
        conv1 = nn.Conv2d(8, 32, 3, padding=1)
        vq = V.VectorQuantizer(dim=32, num_embeddings=24, kmeans_init=True, kmeans_iters=3)
        vq.enable_ema(decay=0.9)
        conv2 = nn.Conv2d(32, 40, 3, padding=1)
        head = V.VQSegmentationHead(dim=40, num_embeddings=classes)
        model = nn.ModuleList([conv1, vq, conv2, head]).to(dev).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)
        g = torch.Generator(device="cuda").manual_seed(9)
        for _ in range(3):
            x = torch.randn(4, 8, 32, 32, device=dev, generator=g)
            tgt = torch.randn(4, classes, 32, 32, device=dev, generator=g)
            q, _, vq_loss, _ = vq(torch.relu(conv1(x)))
            _, score, _, head_loss, _ = head(torch.relu(conv2(q)))
            loss = (score * tgt).sum() + vq_loss.sum() + head_loss.sum()
            opt.zero_grad()
            loss.backward()
            opt.step()
        return [p.detach().cpu().clone() for p in model.parameters()] + [vq.codebook.embedding.weight.detach().cpu()]

    for classes in (3, 150):
        a, b = run(classes), run(classes)
        same = all(torch.equal(u, v) for u, v in zip(a, b))
        print(classes, "identical" if same else "DIFFER")
        if not same:
            sys.exit(1)
""")


def test_small_model_trains_bit_identically(dev):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    r = subprocess.run([sys.executable, "-c", _TRAIN, ROOT], env=env, capture_output=True, text=True, timeout=200)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.split() == ["3", "identical", "150", "identical"]
