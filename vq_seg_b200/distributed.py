"""Multi-GPU modes of the VQ path: one process per GPU, torch.distributed (NCCL over NVLink 5 / NVSwitch).

The reference is single-GPU (SURVEY.md §2a); its single-GPU result is the oracle for both modes.

1. data-parallel over latent pixels, replicated codebook
     * lookup shards with NO data-path collective (rows are independent); only the K per-code counts
       (4 KiB at K=512) are all-reduced when a GLOBAL code usage is wanted;
     * k-means / code-stat update: every rank computes local counts[K] + sums[K,D] and ONE exchange step
       per Lloyd iteration all-reduces both; every rank then applies the identical
       `where(count==0, old, sum/count)` (vq_img.py:44-61).  Counts are bit-exact for any rank count;
       sums are fp32 and follow the all-reduce's association order (tolerance 1e-5).
2. codebook-sharded assignment for very large K: every rank scores the replicated rows against ITS slice of
   the codebook (exact distances), packs (float_bits(dist) << 32 | global index) into an int64 key and the
   ranks MIN-all-reduce the keys: distances are >= 0 so their bit patterns order like the floats, and the
   index in the low word reproduces torch.argmin's lowest-index-wins tie rule across shards.

The collectives are device-agnostic (the CPU tests drive them over gloo with the oracle standing in for the
local kernels through the `*_fn` hooks); the default local compute is the CUDA path, which has no CPU fallback.
"""
from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist


def _world(group=None) -> Tuple[int, int]:
    if not dist.is_available() or not dist.is_initialized():
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def allreduce_code_stats(counts: torch.Tensor, sums: torch.Tensor, group=None) -> None:
    """In-place SUM all-reduce of per-code counts (int64) and sums (fp32): the one exchange step of a
    data-parallel Lloyd iteration (2.1 MB at K=1024, D=512: latency-bound over NVSwitch)."""
    if _world(group)[1] == 1:
        return
    h1 = dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group, async_op=True)
    h2 = dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group, async_op=True)
    h1.wait()
    h2.wait()


def broadcast_rows(rows: torch.Tensor, group=None) -> None:
    """In-place broadcast of rank 0's packed (K, D) rows: the `expire_sync_fn` of enable_ema(threshold_ema_dead_code=...).
    Every rank draws its own dead-code candidates from its own batch; with `allreduce_code_stats` as the EMA's
    `reduce_fn` the cluster sizes, hence the expired codes, are the same on every rank, and rank 0's candidates keep
    the codebooks identical (K * D * 4 bytes per training forward)."""
    if _world(group)[1] == 1:
        return
    dist.broadcast(rows, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)


def global_code_usage(counts: torch.Tensor, group=None, usage_fn: Optional[Callable] = None) -> torch.Tensor:
    """code_usage over ALL ranks' pixels: all-reduce the K counts, then 100 * (#zero / K) (vq_img.py:173-175)."""
    counts = counts.clone()
    if _world(group)[1] > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    if usage_fn is None:
        from . import ops
        usage_fn = ops.code_usage
    return usage_fn(counts)


def shard_rows(n_rows: int, group=None) -> Tuple[int, int]:
    """Contiguous [begin, end) slice of the global row range owned by this rank."""
    rank, world = _world(group)
    per = (n_rows + world - 1) // world
    return min(rank * per, n_rows), min((rank + 1) * per, n_rows)


def dp_init_means(x_local: torch.Tensor, row_begin: int, global_init_rows: torch.Tensor, group=None,
                  gather_rows_fn: Optional[Callable] = None) -> torch.Tensor:
    """Initial k-means means (sample_vectors, vq_img.py:10-17) when the samples are sharded: rank 0's choice
    of GLOBAL row ids is broadcast, each rank fills the rows it owns, and a SUM all-reduce assembles the
    identical (K, D) start on every rank (every row has exactly one owner, so the sum is exact)."""
    rank, world = _world(group)
    ids = global_init_rows.clone()
    if world > 1:
        dist.broadcast(ids, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    n_local = x_local.shape[0] * x_local.shape[1]
    local = ids - row_begin
    own = (local >= 0) & (local < n_local)
    if gather_rows_fn is None:
        from . import ops
        gather_rows_fn = ops.gather_rows
    rows = gather_rows_fn(x_local, torch.where(own, local, torch.full_like(local, -1)))   # -1 -> zero row
    rows = rows * own.to(rows.dtype).unsqueeze(1)
    if world > 1:
        dist.all_reduce(rows, op=dist.ReduceOp.SUM, group=group)
    return rows


def dp_kmeans(x_local: torch.Tensor, num_clusters: int, num_iters: int, global_init_rows: torch.Tensor,
              row_begin: int, group=None, use_cosine_sim: bool = False, deterministic: bool = True):
    """Data-parallel Lloyd iterations (kmeans, vq_img.py:29-63) on this rank's (B, P, D) slice.
    Returns (means (1,K,D), bins (1,K)) identical on every rank."""
    from . import ops
    means = dp_init_means(x_local, row_begin, global_init_rows, group)
    bins = torch.zeros(num_clusters, dtype=torch.int64, device=x_local.device)
    for _ in range(num_iters):
        if use_cosine_sim:
            buckets, _ = ops.assign_cosine(x_local, means)
        else:
            buckets, _ = ops.assign(x_local, means, ops.prepare_codebook(means), ops.ALGO_AUTO)
        bins, sums = ops.code_stats(x_local, buckets, num_clusters, deterministic)
        allreduce_code_stats(bins, sums, group)
        ops.kmeans_finalize(sums, bins, means, use_cosine_sim)
    return means.unsqueeze(0), bins.unsqueeze(0)


def pack_keys(dist_f32: torch.Tensor, global_idx: torch.Tensor) -> torch.Tensor:
    """(float_bits(dist) << 32) | idx as int64 (dist >= 0, so the key is non-negative and MIN-reducible)."""
    bits = dist_f32.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    return (bits << 32) | (global_idx.to(torch.int64) & 0xFFFFFFFF)


def unpack_keys(keys: torch.Tensor):
    idx = keys & 0xFFFFFFFF
    d = (keys >> 32).to(torch.int32).view(torch.float32)
    return idx, d


def sharded_assign(x: torch.Tensor, codebook_shard: torch.Tensor, code_base: int, num_codes_total: int,
                   group=None, local_keys_fn: Optional[Callable] = None, unpack_fn: Optional[Callable] = None):
    """Codebook-sharded nearest-code assignment.  x: the SAME (B, P, D) rows on every rank; codebook_shard:
    this rank's contiguous slice [code_base, code_base + K_local) of the codebook.
    Returns (idx (B,P) int64 global indices, dist (B,P) fp32, counts (K_total,) int64), identical on every rank."""
    if local_keys_fn is None:
        from . import ops

        def local_keys_fn(xx, cb, base):
            return ops.assign_keys(xx, cb, ops.prepare_codebook(cb), base, ops.ALGO_AUTO)
    keys = local_keys_fn(x, codebook_shard, code_base)
    if _world(group)[1] > 1:
        dist.all_reduce(keys, op=dist.ReduceOp.MIN, group=group)       # ncclMin on 8 B per row
    if unpack_fn is None:
        from . import ops
        return ops.unpack_keys(keys, num_codes_total)
    return unpack_fn(keys, num_codes_total)
