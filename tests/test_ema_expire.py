"""CPU tests of the EMA dead-code expiry (opt-in extension, no reference counterpart): the restated equations of
tests/ema_expire_oracle.py against a literal transcription of lucidrains/vector-quantize-pytorch's boolean-mask
`replace`, the module surface of enable_ema(threshold_ema_dead_code=...), and the data-parallel hooks over gloo."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ema_expire_oracle import ema_expire
from oracle import vq_oracle as O


def _lucidrains_expire(cluster_size, embed_avg, embed, samples, threshold, reset, sample_fn):
    """expire_codes_ + replace of lucidrains/vector-quantize-pytorch for one codebook, transcribed"""
    cluster_size, embed_avg, embed = cluster_size.clone(), embed_avg.clone(), embed.clone()
    expired_codes = cluster_size < threshold
    if not torch.any(expired_codes):
        return cluster_size, embed_avg, embed
    mask = expired_codes
    sampled = sample_fn(samples, mask.sum().item())
    embed[mask] = sampled
    cluster_size[mask] = reset
    embed_avg[mask] = sampled * reset
    return cluster_size, embed_avg, embed


def _candidate_ids(n, k, g):
    """sample_vectors' rule: randperm(N)[:K] when N >= K, else randint(0, N, (K,))"""
    return torch.randperm(n, generator=g)[:k] if n >= k else torch.randint(0, n, (k,), generator=g)


# (K, D, N, how the cluster sizes sit against the threshold)
CASES = [(64, 16, 500, "none"), (64, 16, 500, "some"), (64, 16, 500, "all"), (64, 16, 500, "tie"),
         (300, 8, 40, "some"), (7, 3, 7, "some"), (1, 5, 3, "all")]


@pytest.mark.parametrize("k,d,n,kind", CASES)
@pytest.mark.parametrize("reset", [None, 0.25])
def test_oracle_matches_lucidrains_replace(k, d, n, kind, reset):
    g = torch.Generator().manual_seed(k * 1000 + n)
    threshold = 1.0
    cs = torch.rand(k, generator=g) * 3
    if kind == "none":
        cs = cs + threshold
    elif kind == "all":
        cs = cs * 0.3
    elif kind == "tie":
        cs[::3] = threshold                                  # exactly at the threshold: strict comparison, live
        cs[1::3] = torch.nextafter(torch.tensor(threshold), torch.tensor(0.0))
    ea = torch.randn(k, d, generator=g)
    w = torch.randn(k, d, generator=g)
    samples = torch.randn(n, d, generator=g)
    seed = 99 + k
    ids = _candidate_ids(n, k, torch.Generator().manual_seed(seed))
    got = ema_expire(cs, ea, w, samples[ids], threshold, reset)
    if n >= k:
        # lucidrains draws randperm(N)[:m] for m expired codes: the same permutation gives the same first m rows
        def sample_fn(s, m):
            return s[torch.randperm(s.shape[0], generator=torch.Generator().manual_seed(seed))[:m]]
    else:
        def sample_fn(s, m):
            return s[ids[:m]]
    want = _lucidrains_expire(cs, ea, w, samples, threshold, threshold if reset is None else reset, sample_fn)
    for a, b in zip(got[:3], want):
        assert torch.equal(a, b)
    expected_n = {"none": 0, "all": k}.get(kind)
    assert got[3] == int((cs < threshold).sum()) and (expected_n is None or got[3] == expected_n)
    if kind == "tie":
        assert torch.equal(got[0][::3], cs[::3]) and torch.equal(got[2][::3], w[::3])


def test_enable_ema_expiry_surface():
    import vq_seg_b200 as V
    m = V.VectorQuantizer(dim=8, num_embeddings=16)
    sync = lambda rows: None  # noqa: E731
    m.enable_ema(threshold_ema_dead_code=2, expire_sync_fn=sync)
    cb = m.codebook
    assert cb.ema_enabled and cb.threshold_ema_dead_code == 2.0 and cb.reset_cluster_size == 2.0
    assert cb.expire_sync_fn is sync and cb.expire_indices is None
    assert cb.codes_expired_last.dtype == torch.int64 and cb.codes_expired_last.dim() == 0
    assert int(cb.codes_expired_last) == 0 and int(cb.codes_expired_total) == 0
    m.enable_ema(threshold_ema_dead_code=1.5, reset_cluster_size=0.5)
    assert cb.threshold_ema_dead_code == 1.5 and cb.reset_cluster_size == 0.5
    assert V.VectorQuantizer(dim=8, num_embeddings=16).codebook.threshold_ema_dead_code == 0.0    # off by default
    m2 = V.VectorQuantizer(dim=8, num_embeddings=16).enable_ema()
    assert m2.codebook.threshold_ema_dead_code == 0.0


@pytest.mark.parametrize("bad", [-1.0, -1e-30, float("nan")])
def test_enable_ema_rejects_bad_threshold(bad):
    import vq_seg_b200 as V
    m = V.VectorQuantizer(dim=8, num_embeddings=16)
    with pytest.raises(ValueError, match="threshold_ema_dead_code"):
        m.enable_ema(threshold_ema_dead_code=bad)
    assert not m.codebook.ema_enabled


def test_expiry_without_ema_is_an_error():
    import vq_seg_b200 as V
    m = V.VectorQuantizer(dim=8, num_embeddings=16)
    m.codebook.threshold_ema_dead_code = 1.0
    m.train()
    with pytest.raises(ValueError, match="enable_ema"):
        m(torch.randn(1, 8, 2, 2))


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("persistent", [False, True])
def test_expiry_adds_no_state_dict_keys(distance, persistent):
    import vq_seg_b200 as V
    m = V.VectorQuantizer(dim=8, num_embeddings=16, distance=distance)
    m.enable_ema(persistent=persistent)
    keys = list(m.state_dict())
    m2 = V.VectorQuantizer(dim=8, num_embeddings=16, distance=distance)
    m2.enable_ema(persistent=persistent, threshold_ema_dead_code=1.0, reset_cluster_size=2.0)
    assert list(m2.state_dict()) == keys
    assert not [k for k in m2.state_dict() if "expired" in k]
    m2.load_state_dict(m.state_dict())
    assert "codebook.codes_expired" in dict(m2.named_buffers())      # a buffer (moves with .to()), never saved


# ---- data-parallel: gloo, world size 2, the oracle standing in for the kernels through the hooks -------------------
K, D, ROWS = 32, 12, 300


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _start():
    g = torch.Generator().manual_seed(5)
    w = torch.randn(K, D, generator=g)
    w[16:] += 40.0                                            # codes far from every row: no vector, they expire
    return w


def _step(x, w, cs, ea, reduce_fn, cand, sync_fn):
    """one training step of the EMA with expiry as vq_img._ema_step sequences it"""
    idx = torch.argmin(O.euclidean_dist(x.unsqueeze(0), w)[0], dim=-1)
    counts = torch.bincount(idx, minlength=K)
    sums = torch.zeros(K, D).index_add_(0, idx, x)
    reduce_fn(counts, sums)
    sync_fn(cand)
    cs, ea, w = O.ema_update(counts, sums, cs, ea, torch.tensor(0.8), 1e-5)
    return ema_expire(cs, ea, w, cand, 1.0)


def _worker(rank, world, port, results):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    from vq_seg_b200 import distributed as Dd
    x = torch.randn(ROWS, D, generator=torch.Generator().manual_seed(100 + rank))           # ranks hold different x
    cand = x[torch.randperm(ROWS, generator=torch.Generator().manual_seed(200 + rank))[:K]].clone()
    w = _start()
    results[rank] = {"x": x, "cand": cand.clone(),
                     "out": _step(x, w, torch.ones(K), w.clone(), Dd.allreduce_code_stats, cand, Dd.broadcast_rows)}
    dist.barrier()
    dist.destroy_process_group()


def test_world2_gloo_expiry_keeps_codebooks_identical():
    mgr = mp.Manager()
    results = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), results), nprocs=2, join=True)
    r0, r1 = results[0], results[1]
    assert not torch.equal(r0["cand"], r1["cand"])
    for a, b in zip(r0["out"][:3], r1["out"][:3]):
        assert torch.equal(a, b)                              # bit-identical codebooks and moving averages
    assert r0["out"][3] == r1["out"][3] >= 16
    w = _start()
    x = torch.cat([r0["x"], r1["x"]])
    ref = _step(x, w, torch.ones(K), w.clone(), lambda c, s: None, r0["cand"], lambda c: None)
    assert torch.equal(r0["out"][0], ref[0]) and r0["out"][3] == ref[3]
    dead = r0["out"][0] == 1.0
    assert torch.equal(r0["out"][2][dead], ref[2][dead])      # replaced rows: rank 0's candidates, exactly
    torch.testing.assert_close(r0["out"][1], ref[1], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(r0["out"][2], ref[2], rtol=1e-5, atol=1e-5)
