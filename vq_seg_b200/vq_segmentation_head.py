"""B200 drop-in for the reference's VQ segmentation head (models/modules/vq_segmentation_head.py, SURVEY.md 8f-3).

Same classes, constructor arguments, attributes, state_dict keys (`codebook.embedding.weight`) and five outputs as
the reference: (quantize (B,C,H,W), score (B,K,H,W), embed_index (B,H,W) int64, loss (1,), code_usage ()).
The head is a nearest-prototype classifier: the distance (or cosine similarity) of every decoder pixel to each of
the K class prototypes is an OUTPUT (`score = activation(1 - d / sum_k d)`) and carries gradient to the features and
to the prototypes.

Euclidean: one kernel writes the exact fp32 distance map in the (B,K,H,W) score layout together with the argmin
and the class counts (bit-equal to ATen's CPU cdist); its backward is one kernel too.  Cosine: the rows are
l2-normalised by the existing kernel, the same map kernel evaluates the similarities.  Any number of classes and any
width: the per-pixel kernels (csrc/seghead.cu) serve small heads, the register-tiled ones (csrc/seghead_tiled.cu) the
rest, chosen in C (vqseg_seghead_map_f32).  GPU only: there is no CPU fallback.
"""
import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from .vq_img import kmeans


class _SegHeadBase(nn.Module):
    """Shared constructor (EuclideanSegHead :134-159 / CosinesimSegHead :66-92)."""

    def __init__(self, embedding_dim, num_embeddings, kmeans_init, kmeans_iters, decay, eps, num_codebook):
        super().__init__()
        self.kmeans_init = kmeans_init
        self.kmeans_iters = kmeans_iters
        self.initted = False                    # plain attribute, not in the state_dict (like the reference)
        self.num_codebook = num_codebook
        self.decay = decay
        self.embedding = nn.Embedding(num_embeddings, embedding_dim)
        self.num_embeddings = num_embeddings
        self.embedding_dim = embedding_dim
        if not kmeans_init:
            self.embedding.weight.data.uniform_(-1 / self.num_embeddings, 1 / self.num_embeddings)
            self.initted = True
        self.kmeans_init_indices = None         # optional (K,) int64 start rows (reproducible init; default: randperm)

    def _kmeans_init(self, flatten_x, cosine):
        if self.initted:
            return
        embed, _ = kmeans(flatten_x, self.num_embeddings, self.kmeans_iters, use_cosine_sim=cosine,
                          init_indices=self.kmeans_init_indices)
        self.embedding.weight.data.copy_(embed[0])
        self.initted = True

    @staticmethod
    def _usage(counts, k):
        return ops.fast_code_usage(counts)


class EuclideanSegHead(_SegHeadBase):
    def forward(self, x):
        """x: (B, HW, C) view.  Returns (quantized, distance (B, HW, K), embed_idx, code_usage) like :160-179."""
        x = x.float()
        if x.shape[-1] != self.embedding_dim:
            raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {x.shape[-1]} X2: {self.embedding_dim}")
        distance, embed_idx, counts = self.lookup(x)
        quantized = ops.eval_gather(self.embedding.weight, x, embed_idx)       # one_hot @ weight (:170-171)
        return quantized, distance, embed_idx, self._usage(counts, self.num_embeddings)

    def lookup(self, x):
        """k-means hook + (distance map, argmin, class counts) without the gather."""
        if self.kmeans_init and self.training:
            self._kmeans_init(x, cosine=False)
        return ops.euclidean_dist_map(x, self.embedding.weight)


class _CosineMap(torch.autograd.Function):
    """similarity = l2norm(x) @ weight^T with weight already unit-norm (:97-104); gradient through the
    normalisation to x and directly to the weight (the reference renormalises weight.data in place).  Forward: the
    map kernel on the normalised rows; backward: vqseg_seghead_map_bwd_f32 in cosine mode."""

    @staticmethod
    def forward(ctx, x, weight):
        xn = ops.l2norm_rows(x)
        sim, idx, counts = ops.fast_seghead_map(xn, weight, True)
        ctx.save_for_backward(x, sim, weight)
        ctx.mark_non_differentiable(idx, counts)
        return sim, idx, counts

    @staticmethod
    def backward(ctx, g, g_idx, g_counts):
        x, sim, weight = ctx.saved_tensors
        gx, gw = ops.fast_seghead_map_bwd(g, sim, x, weight, True)
        return (gx if ctx.needs_input_grad[0] else None), (gw if ctx.needs_input_grad[1] else None)


class CosinesimSegHead(_SegHeadBase):
    def forward(self, x):
        """x: (B, HW, C) view.  Returns (quantized, similarity (B, HW, K), embed_idx, code_usage) like :93-119."""
        x = x.float()
        sim, embed_idx, counts = self.lookup(x)
        quantized = ops.eval_gather(self.embedding.weight, x, embed_idx)
        return quantized, sim, embed_idx, self._usage(counts, self.num_embeddings)

    def lookup(self, x):
        if self.kmeans_init and self.training:
            self._kmeans_init(ops.l2norm_rows(x), cosine=True)
        w = self.embedding.weight
        ops.l2norm_rows_(w.data)                                                # in-place renormalisation (:100)
        return _CosineMap.apply(x, w)


class VQSegmentationHead(nn.Module):
    """Drop-in for vq_segmentation_head.VQSegmentationHead (:195-253): same kwargs, defaults and outputs."""

    def __init__(self, dim, num_embeddings, embedding_dim=None, decay=0.8, eps=1e-5, kmeans_init=False,
                 kmeans_iters=10, distance='euclidean', commitment_weight=1, num_codebook=1, activation=nn.Softmax2d):
        super().__init__()
        embedding_dim = embedding_dim if embedding_dim != None else dim  # noqa: E711 (reference spelling)
        self.num_embeddings = num_embeddings
        self.eps = eps
        self.commitment_weight = commitment_weight
        self.code_distance = distance
        codebook_dict = {'euclidean': EuclideanSegHead, 'cosine': CosinesimSegHead}
        codebook_class = codebook_dict[distance]           # KeyError on anything else, like :219
        self.codebook = codebook_class(embedding_dim=embedding_dim, num_embeddings=num_embeddings,
                                       kmeans_init=kmeans_init, kmeans_iters=kmeans_iters, decay=decay, eps=eps,
                                       num_codebook=num_codebook)
        self.activation = activation()

    def forward(self, x):
        if x.dim() != 4:
            raise ValueError(f"VQSegmentationHead expects a (B, C, H, W) tensor, got shape {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError("vq_seg_b200.VQSegmentationHead runs on a B200 GPU only (no CPU fallback); "
                               "move the module and its input to cuda")
        x = x.to(torch.float32)
        b, c, h, w = x.shape
        xv = x.reshape(b, c, h * w).permute(0, 2, 1)              # 'b c h w -> b (h w) c' as a view
        cb = self.codebook
        if xv.shape[-1] != cb.embedding_dim:
            raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {xv.shape[-1]} X2: {cb.embedding_dim}")
        # default configuration (Euclidean + Softmax2d): distances, normalisation and softmax in ONE kernel each way
        fused = self.code_distance == "euclidean" and type(self.activation) is nn.Softmax2d
        if fused:
            if cb.kmeans_init and self.training:
                cb._kmeans_init(xv, cosine=False)
            score_bpk, embed_idx, counts = ops.euclidean_score_map(xv, cb.embedding.weight)
        else:
            distance, embed_idx, counts = cb.lookup(xv)
        code_usage = ops.fast_code_usage(counts)
        loss = torch.zeros(1, device=x.device, dtype=torch.float32, requires_grad=self.training)
        # under fp16 / bf16 autocast the reference's one_hot @ weight is a matmul in that dtype: the gathered code is
        # E[idx] rounded through it (same switch as VectorQuantizer.amp_compat)
        amp = ops.autocast_code_dtype(getattr(self, "amp_compat", True))
        if self.training:
            # quantize = x + (quantize - x).detach(); loss = mse(quantize.detach(), x) * w   (:237-242)
            quantize, mse = ops.straight_through(xv, cb.embedding.weight.detach(), embed_idx, amp)
            if self.commitment_weight > 0:
                loss = loss + mse * self.commitment_weight
        else:
            quantize = ops.eval_gather(cb.embedding.weight, xv, embed_idx, amp)      # one_hot @ weight (:170-171)
        # the maps are stored as (B, K, HW): 'b (h w) c -> b c h w' is a view of them
        if fused:
            score = score_bpk.permute(0, 2, 1).reshape(b, -1, h, w)
        else:
            score = distance.permute(0, 2, 1).reshape(b, -1, h, w)
            if self.code_distance == "euclidean":
                score = 1 - (score / torch.sum(score, dim=1, keepdim=True))    # :245
            score = self.activation(score)
        quantize = quantize.permute(0, 2, 1).reshape(b, c, h, w)
        embed_index = embed_idx.reshape(b, h, w)
        return quantize, score, embed_index, loss, code_usage
