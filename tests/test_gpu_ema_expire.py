"""EMA dead-code expiry on the B200 (opt-in extension, no reference counterpart; run with -m gpu): the kernels against
tests/ema_expire_oracle.py and ops.ema_update bit for bit, strided sources, the module against an oracle loop, no host
sync, CUDA-graph capture, threshold 0, opcheck and two NCCL ranks."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import layouts
from ema_expire_oracle import ema_expire
from oracle import vq_oracle as O

pytestmark = pytest.mark.gpu
EPS = torch.finfo(torch.float32).eps


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


def _ids(n, k, g=None, device="cpu"):
    """sample_vectors' rule: randperm(N)[:K] when N >= K, else randint(0, N, (K,))"""
    ids = torch.randperm(n, generator=g)[:k] if n >= k else torch.randint(0, n, (k,), generator=g)
    return ids.to(device)


# ---- the kernels ---------------------------------------------------------------------------------------------------
def _inputs(k, d, kind, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    counts = torch.randint(0, 6, (k,), device=dev, generator=g)
    counts[::5] = 0
    cs0 = torch.rand(k, device=dev, generator=g) * 3
    if kind == "tie":                                   # a third of the codes land exactly on the threshold
        cs0[::3], counts[::3] = cs0[0].clone(), counts[0].clone()
    sums = torch.randn(k, d, device=dev, generator=g) * counts.unsqueeze(1).float()
    ea0 = torch.randn(k, d, device=dev, generator=g)
    cand = torch.randn(k, d, device=dev, generator=g)
    return counts, sums, cs0, ea0, cand


def _threshold(cs, kind):
    if kind == "none":
        return float(cs.min())                          # strict comparison: the smallest code stays live
    if kind == "all":
        return float(torch.nextafter(cs.max(), torch.tensor(float("inf"), device=cs.device)))
    if kind == "tie":
        return float(cs[0])
    return float(cs.quantile(0.4))                      # "some", "reset"


@pytest.mark.parametrize("kind", ["none", "some", "all", "tie", "reset"])
@pytest.mark.parametrize("d", [1, 64, 96, 2048])
@pytest.mark.parametrize("k", [1, 7, 300, 4096, 65536])
def test_kernel_matches_oracle(dev, k, d, kind):
    from vq_seg_b200 import ops
    counts, sums, cs0, ea0, cand = _inputs(k, d, kind, dev, seed=k * 7 + d)
    decay, eps = 0.8, 1e-5
    cs1, ea1, w1 = cs0.clone(), ea0.clone(), torch.empty(k, d, device=dev)
    ops.ema_update(counts, sums, cs1, ea1, w1, decay, eps)
    thr = _threshold(cs1, kind)
    reset = 0.37 if kind == "reset" else None
    want_cs, want_ea, want_w, m = ema_expire(cs1, ea1, w1, cand, thr, reset)
    cs2, ea2 = cs0.clone(), ea0.clone()
    w2 = torch.full((k, d), float("nan"), device=dev)                   # every element must be written
    expired = torch.tensor([5, 7], dtype=torch.int64, device=dev)
    ops.ema_update_expire(counts, sums, cs2, ea2, w2, decay, eps, thr, thr if reset is None else reset, cand, expired)
    assert m == {"none": 0, "all": k}.get(kind, m)
    if kind == "tie":
        assert m < k and not (cs1[::3] < thr).any()
    assert expired.tolist() == [m, 7 + m]
    assert torch.equal(cs2, want_cs) and torch.equal(ea2, want_ea) and torch.equal(w2, want_w)
    live = cs1 >= thr
    assert torch.equal(cs2[live], cs1[live]) and torch.equal(ea2[live], ea1[live]) and torch.equal(w2[live], w1[live])


def test_threshold_zero_is_the_plain_update(dev):
    from vq_seg_b200 import ops
    counts, sums, cs0, ea0, cand = _inputs(300, 96, "some", dev, seed=3)
    a = (cs0.clone(), ea0.clone(), torch.empty(300, 96, device=dev))
    b = (cs0.clone(), ea0.clone(), torch.empty(300, 96, device=dev))
    ops.ema_update(counts, sums, *a, 0.9, 1e-5)
    expired = torch.zeros(2, dtype=torch.int64, device=dev)
    ops.ema_update_expire(counts, sums, *b, 0.9, 1e-5, 0.0, 0.0, cand, expired)
    assert all(torch.equal(x, y) for x, y in zip(a, b)) and expired.tolist() == [0, 0]
    # and through the module: enable_ema(threshold_ema_dead_code=0) is the EMA without the feature
    import vq_seg_b200 as V
    x = torch.randn(2, 64, 8, 8, device=dev)
    mods = []
    for kw in ({}, {"threshold_ema_dead_code": 0.0}):
        kw["deterministic"] = True                      # ordered statistics: two runs are bit-equal
        torch.manual_seed(0)
        m = V.VectorQuantizer(dim=64, num_embeddings=128).to(dev).enable_ema(**kw)
        m.train()
        with torch.no_grad():
            for _ in range(3):
                m(x)
        mods.append(m.codebook)
    for name in ("cluster_size", "embed_avg"):
        assert torch.equal(getattr(mods[0], name), getattr(mods[1], name))
    assert torch.equal(mods[0].embedding.weight, mods[1].embedding.weight)


def test_opcheck(dev):
    from vq_seg_b200 import ops  # noqa: F401
    counts, sums, cs0, ea0, cand = _inputs(40, 24, "some", dev, seed=4)
    args = (counts, sums, cs0, ea0, torch.empty(40, 24, device=dev), 0.8, 1e-5, 1.0, 1.0, cand,
            torch.zeros(2, dtype=torch.int64, device=dev))
    torch.library.opcheck(torch.ops.vqseg.ema_update_expire, args, test_utils=("test_schema", "test_faketensor"))


# ---- candidate sources: every layout of the catalogue, bit-equal to the packed copy --------------------------------
@pytest.mark.parametrize("case", layouts.cases(), ids=layouts.case_id)
def test_sources_over_layouts(dev, case):
    import vq_seg_b200 as V
    lay, shape_name = case
    shape, k = layouts.SHAPES[shape_name]
    _, x = layouts.make(lay, shape, seed=11, device=dev)
    v = layouts.bpd(x)
    b, c, h, w = shape
    n = b * h * w
    idx = torch.randint(0, 8, (b, h * w), device=dev, generator=torch.Generator(device=dev).manual_seed(1))      # eight codes used: the others expire
    ids = _ids(n, k, torch.Generator().manual_seed(2), dev)
    outs = []
    for src in (v, v.contiguous()):
        torch.manual_seed(0)
        cb = V.EuclideanCodebook(embedding_dim=c, num_embeddings=k, kmeans_init=False, kmeans_iters=1, decay=0.8,
                                 eps=1e-5, num_codebook=1).to(dev)
        cb.enable_ema(deterministic=True, threshold_ema_dead_code=1.0, reset_cluster_size=0.375)
        cb.expire_indices = ids
        cb._ema_step(src, idx)
        outs.append((cb.embedding.weight.detach(), cb.cluster_size, cb.embed_avg, cb.codes_expired))
    assert int(outs[0][3][0]) > 0
    for a, bb in zip(*outs):
        assert torch.equal(a, bb)
    rows = v.reshape(-1, c)[ids]
    dead = outs[0][1] == 0.375                          # no live code lands on the reset value
    slot = torch.cumsum(dead.long(), 0) - 1
    assert torch.equal(outs[0][0][dead], rows[slot[dead]])


# ---- the module against an oracle loop -----------------------------------------------------------------------------
def _far_setup(k, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(2, d, 16, 16, generator=g) + 3.0
    e = torch.randn(k, d, generator=g) + 3.0
    e[k // 2:] = -(torch.randn(k // 2, d, generator=g) + 3.0)      # codes far from every row (and opposite in angle)
    return x, e


def _euclid_tie_ok(v, e, idx, ref):
    bad = (idx != ref).nonzero()
    d = O.euclidean_dist(v, e)
    return all((d[b, p, idx[b, p]] - d[b, p, ref[b, p]]).abs() <= 2 * EPS * d[b, p, ref[b, p]].abs()
               for b, p in bad.tolist())


def _ip_tie_ok(v, e, idx, ref):
    bad = (idx != ref).nonzero()
    s = torch.einsum("bpd,kd->bpk", v, e)
    mag = torch.einsum("bpd,kd->bpk", v.abs(), e.abs())
    return all((s[b, p, ref[b, p]] - s[b, p, idx[b, p]]).abs() <= 2 * EPS * mag[b, p, ref[b, p]]
               for b, p in bad.tolist())


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_module_against_oracle_loop(dev, distance):
    import vq_seg_b200 as V
    k, d, decay, thr = 512, 64, 0.8, 1.0
    cosine = distance == "cosine"
    x, e = _far_setup(k, d, seed=8)
    m = V.VectorQuantizer(dim=d, num_embeddings=k, decay=decay, distance=distance).to(dev)
    m.codebook.embedding.weight.data.copy_(e)
    m.enable_ema(threshold_ema_dead_code=thr)
    m.train()
    cb = m.codebook
    v = x.reshape(2, d, -1).permute(0, 2, 1)
    src = O.l2norm(v) if cosine else v
    n = src.shape[0] * src.shape[1]
    far = torch.arange(k // 2, k)
    total, usage = 0, []
    for step in range(3):
        ids = _ids(n, k, torch.Generator().manual_seed(100 + step))
        cb.expire_indices = ids.to(dev)
        w0 = cb.embedding.weight.detach().cpu().clone()
        cs0, ea0 = cb.cluster_size.cpu().clone(), cb.embed_avg.cpu().clone()
        with torch.no_grad():
            _, idx, _, u = m(x.to(dev))
        usage.append(float(u))
        idx = idx.cpu().reshape(2, -1)
        if cosine:
            wn = O.l2norm(w0)
            assert _ip_tie_ok(src, wn, idx, O.assign_cosine(src, wn))
        else:
            assert _euclid_tie_ok(src, w0, idx, O.assign_euclidean(src, w0))
        flat = idx.reshape(-1)
        counts = torch.bincount(flat, minlength=k)
        sums = torch.zeros(k, d).index_add_(0, flat, src.reshape(-1, d))
        # decay as an fp32 tensor: the cluster sizes, hence the expired mask, come out in the kernel's arithmetic
        cs1, ea1, w1 = O.ema_update(counts, sums, cs0, ea0, torch.tensor(decay), 1e-5)
        want_cs, want_ea, want_w, mexp = ema_expire(cs1, ea1, w1, src.reshape(-1, d)[ids], thr)
        total += mexp
        assert cb.codes_expired.tolist() == [mexp, total]
        assert torch.equal(cb.cluster_size.cpu(), want_cs)
        assert torch.allclose(cb.embedding.weight.detach().cpu(), want_w, rtol=1e-4, atol=1e-5)
        assert torch.allclose(cb.embed_avg.cpu(), want_ea, rtol=1e-4, atol=1e-5)
        if step == 0:
            assert mexp >= k // 2
            w = cb.embedding.weight.detach().cpu()
            rows = src.reshape(-1, d)
            assert all((rows == w[j]).all(1).any() for j in far.tolist())     # every far code holds a row of x
    assert usage[1] < usage[0], usage


# ---- no host sync, CUDA-graph capture ------------------------------------------------------------------------------
@pytest.mark.parametrize("rows", [512, 100])             # N >= K: randperm; N < K: randint
def test_expiry_path_does_not_sync(dev, rows):
    import vq_seg_b200 as V
    k, d = 256, 32
    m = V.VectorQuantizer(dim=d, num_embeddings=k).to(dev).enable_ema(threshold_ema_dead_code=1.0)
    cb = m.codebook
    xv = torch.randn(1, rows, d, device=dev)
    idx = torch.randint(0, 8, (1, rows), device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.no_grad():
            cb._ema_step(xv, idx)
            cb._ema_step(xv, idx)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert int(cb.codes_expired[0]) > 0


def _graph_pair(dev, k=512, d=64, reset=None):
    import vq_seg_b200 as V
    x, e = _far_setup(k, d, seed=9)
    mods = []
    for _ in range(2):
        m = V.VectorQuantizer(dim=d, num_embeddings=k).to(dev)
        m.codebook.embedding.weight.data.copy_(e)
        m.enable_ema(threshold_ema_dead_code=1.0, reset_cluster_size=reset, deterministic=True)
        m.train()
        mods.append(m)
    return x.to(dev), mods


def _capture(m, x_static):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        m(x_static)                                       # warm-up: one real training step
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g), torch.no_grad():
        m(x_static)
    return g


def test_graph_capture_matches_eager(dev):
    x, (eager, graphed) = _graph_pair(dev)
    n, k = x.shape[0] * x.shape[2] * x.shape[3], 512
    ids_static = _ids(n, k, torch.Generator().manual_seed(0), dev)
    eager.codebook.expire_indices = ids_static.clone()
    graphed.codebook.expire_indices = ids_static
    x_static = x.clone()
    g = _capture(graphed, x_static)
    with torch.no_grad():
        eager(x)                                          # the warm-up step
    for step in range(3):
        xs = x + 0.1 * step
        ids = _ids(n, k, torch.Generator().manual_seed(step + 1), dev)
        x_static.copy_(xs)
        ids_static.copy_(ids)
        eager.codebook.expire_indices = ids
        g.replay()
        with torch.no_grad():
            eager(xs)
        a, b = eager.codebook, graphed.codebook
        assert torch.equal(a.embedding.weight, b.embedding.weight), step
        assert torch.equal(a.cluster_size, b.cluster_size) and torch.equal(a.embed_avg, b.embed_avg)
        assert torch.equal(a.codes_expired, b.codes_expired)
    assert int(a.codes_expired[1]) >= k // 2


def test_graph_capture_default_sampling(dev):
    x, (_, m) = _graph_pair(dev, reset=0.375)
    cb = m.codebook
    g = _capture(m, x)
    w_before = cb.embedding.weight.detach().clone()
    total_before = int(cb.codes_expired[1])
    g.replay()
    torch.cuda.synchronize()
    # the replay's expiry runs on the cluster sizes the warm-up step left, decayed once more
    dead = cb.codes_expired[0].item()
    assert dead > 0 and int(cb.codes_expired[1]) == total_before + dead
    rows = x.reshape(x.shape[0], x.shape[1], -1).permute(0, 2, 1).reshape(-1, x.shape[1])
    replaced = cb.cluster_size == 0.375                  # no live code lands on the reset value
    w = cb.embedding.weight.detach()
    new = w[replaced]
    assert new.shape[0] == dead
    hits = (new.unsqueeze(1) == rows.unsqueeze(0)).all(-1)                     # (dead, N)
    assert bool(hits.any(1).all()), "a replaced code is not a row of x"
    assert len(set(hits.float().argmax(1).tolist())) == dead, "replacement rows repeat although N >= K"
    assert not torch.equal(w, w_before)


# ---- two GPUs: NCCL ------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, results):
    import vq_seg_b200 as V
    from vq_seg_b200 import distributed as Dd
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    x, e = _far_setup(512, 64, seed=10)
    torch.manual_seed(1234 + rank)                        # ranks draw different candidates
    m = V.VectorQuantizer(dim=64, num_embeddings=512).to(dev)
    m.codebook.embedding.weight.data.copy_(e)
    m.enable_ema(reduce_fn=Dd.allreduce_code_stats, threshold_ema_dead_code=1.0, expire_sync_fn=Dd.broadcast_rows)
    m.train()
    xr = (x + 0.5 * rank).to(dev)                         # and hold different x
    with torch.no_grad():
        for _ in range(3):
            m(xr)
    cb = m.codebook
    results[rank] = tuple(t.cpu() for t in (cb.embedding.weight.detach(), cb.cluster_size, cb.embed_avg,
                                            cb.codes_expired))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_codebooks_stay_identical():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mgr = mp.Manager()
    results = mgr.dict()
    mp.spawn(_nccl_worker, args=(2, _free_port(), results), nprocs=2, join=True)
    for a, b in zip(results[0], results[1]):
        assert torch.equal(a, b)
    assert int(results[0][3][1]) >= 256
