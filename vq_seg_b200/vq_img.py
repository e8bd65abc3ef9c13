"""Drop-in replacement of VQ_SEG's vector_quantizer/vq_img.py on B200.

Same classes, constructor arguments (names, order, defaults), attributes, state_dict keys and
forward outputs as the reference:

    VectorQuantizer(dim, num_embeddings, embedding_dim=None, decay=0.8, eps=1e-5, kmeans_init=False,
                    kmeans_iters=10, distance='euclidean', commitment_weight=1, num_codebook=1)
    forward(x: (B,C,H,W)) -> (quantize (B,C,H,W) fp32, embed_index (B,H,W) int64,
                              loss (1,) fp32 [requires_grad == training], code_usage () fp32)

(reference: vq_img.py:193-244; EuclideanCodebook :133-190; CosinesimCodebook :65-130; kmeans :29-63).
The arithmetic runs in hand-written sm_100a kernels (libvqseg.so) through torch.library custom ops;
there is no CPU path: CPU tensors raise.
"""
from typing import Optional

import torch
from torch import nn

from . import ops

__all__ = ["VectorQuantizer", "EuclideanCodebook", "CosinesimCodebook", "kmeans", "sample_vectors",
           "batched_sample_vectors", "batched_bincount", "l2norm"]


def l2norm(t: torch.Tensor) -> torch.Tensor:
    """vq_img.py:7-8.  (B, P, D) -> packed unit rows."""
    lead = t.shape[:-1]
    return ops.l2norm_rows(t.reshape(1, -1, t.shape[-1]) if t.dim() != 3 else t).reshape(*lead, t.shape[-1])


def _sample_rows(x_bpd: torch.Tensor, num: int, indices: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`num` rows of the flattened (B*P, D) view of x_bpd WITHOUT flattening it (strided NCHW views stay in place):
    randperm(N)[:num] if N >= num, else randint with replacement (vq_img.py:11-15)."""
    num_samples, device = x_bpd.shape[0] * x_bpd.shape[1], x_bpd.device
    if indices is None:
        if num_samples >= num:
            indices = torch.randperm(num_samples, device=device)[:num]
        else:
            indices = torch.randint(0, num_samples, (num,), device=device)
    return ops.gather_rows(x_bpd, indices.to(device))


def sample_vectors(sample: torch.Tensor, num: int, indices: Optional[torch.Tensor] = None) -> torch.Tensor:
    """vq_img.py:10-17 for an (N, D) sample.  `indices` injects the choice (the device RNG stream differs from the
    CPU one)."""
    return _sample_rows(sample.unsqueeze(0), num, indices)


def batched_sample_vectors(samples: torch.Tensor, num: int) -> torch.Tensor:
    """vq_img.py:19-20"""
    return torch.stack([sample_vectors(s, num) for s in samples.unbind(dim=0)], dim=0)


def batched_bincount(x: torch.Tensor, minlength: int) -> torch.Tensor:
    """vq_img.py:22-27 for (1, N) int64 input -> (1, minlength) int64."""
    return torch.stack([ops.unpack_keys(row, minlength)[2] for row in x.unbind(dim=0)], dim=0)


def kmeans(flatten_x: torch.Tensor, num_clusters: int, num_iters: int, use_cosine_sim: bool = False,
           init_indices: Optional[torch.Tensor] = None, deterministic: bool = True, algo: int = ops.ALGO_AUTO,
           reduce_fn=None):
    """Lloyd iterations of vq_img.py:29-63 on the (B, P, D) view (or (N, D) samples) WITHOUT copying it.

    Per iteration: fused distance+argmin (tcgen05 filter + exact rescoring), per-code counts and
    ordered per-code sums, then means = where(count==0, means, sums/count) [l2norm if cosine].
    `reduce_fn(counts, sums)` is the data-parallel hook: it must all-reduce both in place
    (vq_seg_b200.distributed.allreduce_code_stats).  Returns (means (1,K,D), bins (1,K) int64) like the
    reference; bins belong to the LAST assignment."""
    x = flatten_x if flatten_x.dim() == 3 else flatten_x.reshape(1, -1, flatten_x.shape[-1])
    x = x.detach()
    n_rows = x.shape[0] * x.shape[1]
    means = _sample_rows(x, num_clusters, init_indices)            # batched_sample_vectors of vq_img.py:33, one codebook
    if reduce_fn is not None and init_indices is None:
        # data-parallel: every rank drew its own rows; all must iterate from ONE start (rank 0's), or the first
        # all-reduce would sum statistics of unrelated clusters under one index and the replicas would diverge
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.broadcast(means, src=0)
    bins = torch.zeros(num_clusters, dtype=torch.int64, device=x.device)
    # many samples, several iterations, a codebook that is streamed (not resident): convert the samples to the
    # filter's fp16 operand ONCE -- the conversion bounds the streaming kernel at K ~ 1024 (DESIGN.md 4.0b)
    samples = None
    if (not use_cosine_sim and algo in (ops.ALGO_AUTO, ops.ALGO_TC) and num_iters > 1 and n_rows >= 65536
            and x.shape[-1] <= 512 and 256 < num_clusters <= 65536):
        samples = ops.prepare_samples(x)
    for _ in range(num_iters):
        if use_cosine_sim:
            buckets, _ = ops.assign_cosine(x, means, None, algo)
        else:
            blob = ops.prepare_codebook(means) if algo != ops.ALGO_EXACT else None
            buckets, _ = ops.assign(x, means, blob, algo, 0, samples)
        bins, sums = ops.code_stats(x, buckets, num_clusters, deterministic)
        if reduce_fn is not None:
            reduce_fn(bins, sums)
        ops.kmeans_finalize(sums, bins, means, use_cosine_sim)
    return means.unsqueeze(0), bins.unsqueeze(0)


class _CodebookBase(nn.Module):
    """Shared constructor of EuclideanCodebook (vq_img.py:134-159) / CosinesimCodebook (:66-92)."""

    def __init__(self, embedding_dim, num_embeddings, kmeans_init, kmeans_iters, decay, eps, num_codebook):
        super().__init__()
        self.kmeans_init = kmeans_init
        self.kmeans_iters = kmeans_iters
        self.initted = False                    # plain attribute, NOT in the state_dict (like the reference)
        self.ema_enabled = False
        self.num_codebook = num_codebook
        self.decay = decay                      # accepted and stored, never read (the reference has no EMA)
        self.embedding = nn.Embedding(num_embeddings, embedding_dim)
        self.num_embeddings = num_embeddings
        self.embedding_dim = embedding_dim
        if not kmeans_init:
            self.embedding.weight.data.uniform_(-1 / self.num_embeddings, 1 / self.num_embeddings)
            self.initted = True
        # B200 knobs (not in the reference signature)
        self.algo = ops.ALGO_AUTO
        self.kmeans_init_indices = None         # test hook: inject the k-means init rows
        self.kmeans_reduce_fn = None            # data-parallel hook: all-reduce (counts, sums)
        self.threshold_ema_dead_code = 0.0      # dead-code expiry of the EMA update (enable_ema); 0 = off
        self.expire_indices = None              # test hook: inject the K candidate rows of the expiry
        self._blob = None
        self._blob_key = None

    def _prepared(self, ip=False):
        """The prepared-codebook blob (a cache: every assignment re-checks it against the live weights on the device
        and rebuilds it in place when they changed, so `weight.data.copy_()` needs no invalidate())."""
        w = self.embedding.weight
        key = (w.data_ptr(), w._version, w.device, ip)
        if self._blob is None or self._blob_key != key:
            self._blob = ops.fast_prepare_codebook(w.detach(), ip)
            self._blob_key = key
        return self._blob

    def invalidate(self):
        self._blob = None

    # ---- opt-in EMA codebook update (extension, SURVEY.md 8f-4; the reference never reads decay / eps) ----
    def enable_ema(self, decay=None, eps=1e-5, reduce_fn=None, deterministic=False, persistent=False,
                   threshold_ema_dead_code=0.0, reset_cluster_size=None, expire_sync_fn=None):
        """After every TRAINING forward move the codebook towards the per-code means of that batch with the
        standard VQ-VAE EMA rule (include/vqseg.h, vqseg_ema_update_f32), using the `decay` the constructor stored
        (VectorQuantizer.enable_ema() also passes its stored `eps`).  `reduce_fn(counts, sums)` all-reduces the statistics in data-parallel training
        (vq_seg_b200.distributed.allreduce_code_stats).  The moving averages are non-persistent buffers by default, so
        state_dict keys stay the reference's; `persistent=True` puts `cluster_size` / `embed_avg` into the state_dict so
        a resumed run continues the averages instead of restarting them.  They start as if every code had been used
        once (cluster_size = 1, embed_avg = weight): a code that gets no vector in the first steps keeps its weight
        instead of being divided by ~eps.

        `threshold_ema_dead_code > 0` replaces dead codes on the device after each EMA update (threshold_ema_dead_code
        of lucidrains/vector-quantize-pytorch): every code whose updated cluster_size is below the threshold takes a
        row of the batch (K rows drawn like sample_vectors; the r-th dead code in ascending k gets row r) as its
        weight, that row * `reset_cluster_size` (default: the threshold) as its embed_avg and `reset_cluster_size` as
        its cluster_size (vqseg_ema_update_expire_f32).  No host sync and no data-dependent shapes, so a training
        forward with expiry can be captured as a CUDA graph.  `expire_sync_fn(rows)` makes the K candidate rows
        identical on every rank in data-parallel training (vq_seg_b200.distributed.broadcast_rows).  The int64 device
        counters `codes_expired_last` / `codes_expired_total` count the replaced codes; they are not in the state_dict."""
        threshold_ema_dead_code = float(threshold_ema_dead_code)
        if not threshold_ema_dead_code >= 0:
            raise ValueError(f"threshold_ema_dead_code must be >= 0, got {threshold_ema_dead_code}")
        if decay is not None:
            self.decay = decay
        self.ema_eps = eps
        w = self.embedding.weight
        self.register_buffer("cluster_size", torch.ones(self.num_embeddings, dtype=torch.float32, device=w.device),
                             persistent=persistent)
        self.register_buffer("embed_avg", w.detach().clone().float().contiguous(), persistent=persistent)
        self.ema_reduce_fn = reduce_fn
        self.ema_deterministic = deterministic
        self.threshold_ema_dead_code = threshold_ema_dead_code
        self.reset_cluster_size = threshold_ema_dead_code if reset_cluster_size is None else float(reset_cluster_size)
        self.expire_sync_fn = expire_sync_fn
        self.register_buffer("codes_expired", torch.zeros(2, dtype=torch.int64, device=w.device), persistent=False)
        self.ema_enabled = True
        return self

    @property
    def codes_expired_last(self) -> torch.Tensor:
        """Codes replaced by the last training forward (0-d int64 on the device)."""
        return self.codes_expired[0]

    @property
    def codes_expired_total(self) -> torch.Tensor:
        """Codes replaced since enable_ema() (0-d int64 on the device)."""
        return self.codes_expired[1]

    @torch.no_grad()
    def _ema_step(self, x, idx):
        if idx.numel() == 0:
            return                              # an empty batch carries no statistics (and n = 0 would divide by zero)
        counts, sums = ops.code_stats(x, idx, self.num_embeddings, self.ema_deterministic)
        if self.ema_reduce_fn is not None:
            self.ema_reduce_fn(counts, sums)
        w = self.embedding.weight
        if self.threshold_ema_dead_code > 0:
            cand = _sample_rows(x, self.num_embeddings, self.expire_indices)
            if self.expire_sync_fn is not None:
                self.expire_sync_fn(cand)
            ops.ema_update_expire(counts, sums, self.cluster_size, self.embed_avg, w.data, self.decay, self.ema_eps,
                                  self.threshold_ema_dead_code, self.reset_cluster_size, cand, self.codes_expired)
        else:
            ops.ema_update(counts, sums, self.cluster_size, self.embed_avg, w.data, self.decay, self.ema_eps)
        self.invalidate()                       # the prepared fp16 image of the codebook is stale now

    def _kmeans_init(self, flatten_x, cosine):
        if self.initted:
            return
        embed, _ = kmeans(flatten_x, self.num_embeddings, self.kmeans_iters, use_cosine_sim=cosine,
                          init_indices=self.kmeans_init_indices, reduce_fn=self.kmeans_reduce_fn, algo=self.algo)
        self.embedding.weight.data.copy_(embed[0])
        self.invalidate()                       # .data.copy_ does not bump the version counter
        self.initted = True


class EuclideanCodebook(_CodebookBase):
    def lookup(self, x: torch.Tensor):
        """(idx (B,P) int64, counts (K,) int64) -- cdist + argmin + bincount of vq_img.py:167-168,173."""
        if x.shape[-1] != self.embedding_dim:
            raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {x.shape[-1]} X2: {self.embedding_dim}")
        blob = self._prepared() if self.algo != ops.ALGO_EXACT else None
        return ops.fast_assign(x, self.embedding.weight.detach(), blob, self.algo)

    def forward(self, x):
        """x: (B, HxW, C) -> (quantized (B,HW,C), embed_idx (B,HW), code_usage)   [vq_img.py:160-177]"""
        x = x.float()
        if x.dim() != 3:
            x = x.reshape(x.shape[0], -1, x.shape[-1])
        if self.kmeans_init and self.training:
            self._kmeans_init(x, cosine=False)
        idx, counts = self.lookup(x)
        quantized = ops.eval_gather(self.embedding.weight, x, idx)
        return quantized, idx, ops.code_usage(counts)


class CosinesimCodebook(_CodebookBase):
    def lookup(self, x: torch.Tensor):
        """(idx (B,P) int64, counts (K,) int64) of vq_img.py:97-107: l2norm(x) (ATen's arithmetic, layout kept), the
        in-place renormalisation of the weights EVERY forward (:100), einsum + argmax as the tcgen05 filter + exact
        rescoring in inner-product mode."""
        if x.shape[-1] != self.embedding_dim:
            raise RuntimeError(f"einsum(): operands do not broadcast with remapped shapes: {x.shape[-1]} vs {self.embedding_dim}")
        xn = ops.l2norm_rows(x)
        blob = self._renormalise_and_prepare()
        return ops.fast_assign(xn, self.embedding.weight.detach(), blob, self.algo | ops.METRIC_IP)

    def _renormalise_and_prepare(self):
        """The in-place renormalisation of the weights (vq_img.py:100), then the inner-product blob (None for
        ALGO_EXACT) rebuilt for the renormalised rows."""
        w = self.embedding.weight
        ops.l2norm_rows_(w.data)
        blob = None
        if self.algo != ops.ALGO_EXACT:
            had = self._blob is not None
            blob = self._prepared(ip=True)
            if had and blob is self._blob:
                # the renormalisation moves a few rows by an ulp on every forward (x / |x| is not idempotent in fp32):
                # rebuild the prepared image here with the multi-block kernels instead of leaving it to the assignment's
                # guard, which rebuilds inside a single block (measured: 360-600 us per forward against ~170)
                ops.fast_refresh_codebook(blob, w.detach(), True)
        return blob

    def forward(self, x):
        """x: (B, HxW, C) -> (quantized, embed_idx, code_usage)   [vq_img.py:93-113]"""
        x = x.float()
        if x.dim() != 3:
            x = x.reshape(x.shape[0], -1, x.shape[-1])
        if self.kmeans_init and self.training:
            self._kmeans_init(ops.l2norm_rows(x), cosine=True)
        idx, counts = self.lookup(x)
        quantized = ops.eval_gather(self.embedding.weight, x, idx)
        return quantized, idx, ops.code_usage(counts)


class CudaGraphCache(dict):
    """The opt-in CUDA-graph mode of the quantizer modules (enable_cuda_graphs): ONE captured graph of a no-grad forward
    per (input address, shape, strides, dtype, `extra`), at most `max_entries` of them (the oldest goes first)."""

    def __init__(self, max_entries: int = 16):
        super().__init__()
        self.max_entries = max_entries

    def run(self, forward, x, extra, keep):
        """forward(x)'s outputs, replayed from the entry's graph (captured on the first call).  `keep()` names what the
        graph reads beyond x and the module's parameters (the prepared codebooks): the entry holds it alive."""
        key = (x.data_ptr(), tuple(x.shape), tuple(x.stride()), x.dtype) + tuple(extra) + (torch.cuda.current_device(),)
        ent = self.get(key)
        if ent is None:
            if len(self) >= self.max_entries:
                self.pop(next(iter(self)))                        # oldest entry
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):                         # warm-up outside the capture (lazy init, allocations)
                forward(x)
            cur.wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                outs = forward(x)
            ent = (g, outs, keep())                               # what the graph reads must outlive the cache's view of it
            self[key] = ent
        ent[0].replay()
        return ent[1]


class VectorQuantizer(nn.Module):
    def __init__(self, dim, num_embeddings, embedding_dim=None, decay=0.8, eps=1e-5, kmeans_init=False,
                 kmeans_iters=10, distance='euclidean', commitment_weight=1, num_codebook=1):
        super().__init__()
        embedding_dim = embedding_dim if embedding_dim != None else dim  # noqa: E711 (reference spelling)
        self.num_embeddings = num_embeddings
        self.eps = eps
        self.commitment_weight = commitment_weight
        codebook_dict = {'euclidean': EuclideanCodebook, 'cosine': CosinesimCodebook}
        codebook_class = codebook_dict[distance]          # KeyError on anything else, like vq_img.py:217
        self.codebook = codebook_class(embedding_dim=embedding_dim, num_embeddings=num_embeddings,
                                       kmeans_init=kmeans_init, kmeans_iters=kmeans_iters, decay=decay,
                                       eps=eps, num_codebook=num_codebook)
        self.amp_compat = True    # round the gathered code through the fp16 / bf16 autocast dtype like the reference's matmul
        self.rotation_trick = False  # opt-in: carry the gradient to x by the rotation trick instead of straight-through
        self._graphs = None       # opt-in CUDA-graph cache of the no-grad forward (enable_cuda_graphs)

    def enable_cuda_graphs(self, max_entries: int = 16):
        """Opt-in: replay the no-grad forward as ONE CUDA graph per (input address, shape, strides) instead of
        enqueueing its kernels from Python -- the host cost of a forward drops from ~120 us to one graph launch, so a
        model calling `self.codebook[i](x)` per layer gets the kernels' speed without capturing graphs itself.
        Contract of a captured forward (the usual one for CUDA graphs): the four returned tensors are buffers owned by
        the cache entry and are overwritten by the next call with the same input address; the input must stay at that
        address (a reused activation buffer / a static input).  Weight updates are picked up: the kernels re-check the
        prepared codebook against the live weights on the device.  Training-mode and grad-enabled calls, the k-means
        init and the EMA update take the ordinary path."""
        self._graphs = CudaGraphCache(max_entries)
        return self

    def disable_cuda_graphs(self):
        self._graphs = None
        return self

    def _graph_forward(self, x):
        amp = ops.autocast_code_dtype(self.amp_compat)
        w = self.codebook.embedding.weight
        return self._graphs.run(self._forward_impl, x, (amp, w.data_ptr()), lambda: self.codebook._blob)

    def enable_ema(self, **kw):
        """Opt-in EMA codebook update with the stored `decay` and `eps`, optionally with dead-code expiry
        (`threshold_ema_dead_code`, `reset_cluster_size`, `expire_sync_fn`; extension; see the codebook's enable_ema)."""
        kw.setdefault("eps", self.eps)
        self.codebook.enable_ema(**kw)
        return self

    def forward(self, x):
        if x.dim() != 4:
            raise ValueError(f"VectorQuantizer expects a (B, C, H, W) tensor, got shape {tuple(x.shape)}")
        if self.training and self.codebook.threshold_ema_dead_code > 0 and not self.codebook.ema_enabled:
            raise ValueError("threshold_ema_dead_code replaces codes after the EMA update: enable it through enable_ema()")
        if not x.is_cuda:
            raise RuntimeError("vq_seg_b200.VectorQuantizer runs on a B200 GPU only (no CPU fallback); "
                               "move the module and its input to cuda")
        if (self._graphs is not None and not self.training and not torch.is_grad_enabled() and x.numel() > 0
                and not torch.cuda.is_current_stream_capturing()):
            return self._graph_forward(x)
        return self._forward_impl(x)

    def _forward_impl(self, x):
        x = x.to(torch.float32)
        b, c, h, w = x.shape
        device = x.device
        xv = x.reshape(b, c, h * w).permute(0, 2, 1)          # the 'b c h w -> b (h w) c' VIEW, no copy
        cb = self.codebook
        amp = ops.autocast_code_dtype(self.amp_compat)
        cosine = isinstance(cb, CosinesimCodebook)
        rotate = self.rotation_trick and self.training
        if cb.kmeans_init and self.training and not cb.initted:
            cb._kmeans_init(ops.l2norm_rows(xv) if cosine else xv, cosine=cosine)
        if cosine:
            idx, counts = cb.lookup(xv)
            code_usage = ops.fast_code_usage(counts)
            if self.training:
                quantize, mse = ops.straight_through(xv, cb.embedding.weight.detach(), idx, amp, rotate)
            else:
                quantize, mse = ops.eval_gather(cb.embedding.weight, xv, idx, amp), None
        else:
            # Euclidean: lookup + gather + STE + mse + usage are enqueued by one host call
            if xv.shape[-1] != cb.embedding_dim:
                raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {xv.shape[-1]} X2: {cb.embedding_dim}")
            blob = cb._prepared() if cb.algo != ops.ALGO_EXACT else None
            quantize, idx, mse, code_usage = ops.fused_forward(xv, cb.embedding.weight, blob, self.training, amp,
                                                                cb.algo, rotate)
        # loss (vq_img.py:230,239-241): [0.] + mse * w.  0 + v and v * 1 are exact in fp32, so for the default weight
        # the kernel's (1,) mse IS the loss (no fill / mul / add launches); eval: the kernel's zeroed (1,) output
        if self.training and self.commitment_weight > 0 and (mse.requires_grad or not torch.is_grad_enabled()):
            loss = mse if self.commitment_weight == 1 else mse * self.commitment_weight
        elif self.training and self.commitment_weight > 0:
            # x carries no gradient: the reference's requires_grad leaf still makes the loss require grad
            loss = torch.zeros(1, device=device, dtype=torch.float32, requires_grad=True) + mse * self.commitment_weight
        elif mse is not None and not self.training and not mse.requires_grad:
            loss = mse
        else:
            loss = torch.zeros(1, device=device, dtype=torch.float32, requires_grad=self.training)
        if self.training and cb.ema_enabled:
            if cb.embed_avg.device != device:    # enable_ema() ran before .to(device)
                cb.enable_ema(eps=cb.ema_eps, reduce_fn=cb.ema_reduce_fn, deterministic=cb.ema_deterministic,
                              threshold_ema_dead_code=cb.threshold_ema_dead_code,
                              reset_cluster_size=cb.reset_cluster_size, expire_sync_fn=cb.expire_sync_fn)
            cb._ema_step(ops.l2norm_rows(xv) if cosine else xv, idx)
        quantize = quantize.permute(0, 2, 1).reshape(b, c, h, w)     # memory is already (B, C, H*W): a view
        embed_index = idx.reshape(b, h, w)
        return quantize, embed_index, loss, code_usage
