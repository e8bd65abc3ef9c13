"""Residual vector quantization: OPT-IN EXTENSION, no reference counterpart (ResidualVQ of
lucidrains/vector-quantize-pytorch; parity unpinned).

    ResidualVectorQuantizer(dim, num_embeddings, num_quantizers, embedding_dim=None, decay=0.8, eps=1e-5,
                            kmeans_init=False, kmeans_iters=10, distance='euclidean', commitment_weight=1,
                            num_codebook=1)
    forward(x: (B,C,H,W)) -> (quantize (B,C,H,W) fp32, embed_index (B,H,W,Q) int64, loss (1,) fp32, code_usage () fp32)

Q codebooks quantize the input, then what the first one left, and so on; quantize is the sum of the Q codes.  The
arithmetic is restated exactly in include/vqseg.h (vqseg_rvq_stage_f32); with Q = 1 every output and gradient is
bit-identical to VectorQuantizer's.  Each stage is ONE host call (the assignment's launches with the stage kernel in the
gather's place), the gradient to x is the identity plus the commitment terms of all layers (one elementwise kernel),
and the layers are ordinary VectorQuantizer modules: state_dict keys `layers.{l}.codebook.embedding.weight`, the k-means
init, the EMA update and the dead-code expiry of each layer work as they do there.
"""
import torch
from torch import nn

from . import ops
from .vq_img import CosinesimCodebook, CudaGraphCache, VectorQuantizer

__all__ = ["ResidualVectorQuantizer"]


def _nchw(b, p, d, device):
    """a (B, P, D) buffer in NCHW memory order: the layout the filters read by TMA and the module returns"""
    return torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=device)


def _stages(rvq, xv, mode, training, need_grad):
    """The Q stages on the (B, P, D) view xv: (quantize (B,P,D), idx (Q,B,P), loss (1,), usage (), layer_mse (Q,),
    layer_usage (Q,), A or None).  Layer l is k-means-initialised on r_l (training, kmeans_init) right before its
    stage, and its EMA update runs right after it."""
    b, p, d = xv.shape
    dev = xv.device
    nq, k = len(rvq.layers), rvq.num_embeddings
    weight = float(rvq.commitment_weight)
    q = _nchw(b, p, d, dev)
    idx = torch.empty((nq, b, p), dtype=torch.int64, device=dev)
    counts = torch.empty((nq, k), dtype=torch.int64, device=dev)
    layer_mse = torch.empty(nq, dtype=torch.float32, device=dev)
    layer_usage = torch.empty(nq, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)      # the last stage writes it (0 in eval)
    usage = torch.empty((), dtype=torch.float32, device=dev)
    acc = _nchw(b, p, d, dev) if need_grad else None
    bufs = [_nchw(b, p, d, dev) for _ in range(min(nq - 1, 2))]      # r_1, r_2, ... ping-pong
    stage = ops._rvq_stage_impl if ops._fast() else ops.rvq_stage
    empty = b * p == 0
    r = xv
    for l, layer in enumerate(rvq.layers):
        cb = layer.codebook
        cosine = isinstance(cb, CosinesimCodebook)
        rn = ops.l2norm_rows(r) if cosine and not empty else None
        if training and cb.kmeans_init and not cb.initted and not empty:
            cb._kmeans_init(rn if cosine else r, cosine=cosine)
        w = cb.embedding.weight
        if empty:
            blob = None
        elif cosine:
            blob = cb._renormalise_and_prepare()
        else:
            blob = cb._prepared() if cb.algo != ops.ALGO_EXACT else None
        r_next = bufs[l % 2] if l < nq - 1 else None
        stage(r, rn, w.detach(), blob, xv, q, r_next, acc, idx, counts, layer_mse, layer_usage,
              loss, usage, l, mode, cb.algo, weight)
        if training and cb.ema_enabled:
            if cb.embed_avg.device != dev:    # enable_ema() ran before .to(device)
                cb.enable_ema(eps=cb.ema_eps, reduce_fn=cb.ema_reduce_fn, deterministic=cb.ema_deterministic,
                              threshold_ema_dead_code=cb.threshold_ema_dead_code,
                              reset_cluster_size=cb.reset_cluster_size, expire_sync_fn=cb.expire_sync_fn)
            cb._ema_step(rn if cosine else r, idx[l])
        r = r_next
    return q, idx, loss, usage, layer_mse, layer_usage, acc


class _RVQTrain(torch.autograd.Function):
    """Training forward of the Q stages.  Gradient to x: gx = fma(coef, A, g) with coef = g_loss * w * 2 / numel
    (vqseg_ste_bwd_f32 with x = A and no q): the identity through the sum of the codes plus every layer's commitment
    term.  The codebooks get none, and the backward reads no weight (the EMA update may have rewritten them)."""

    @staticmethod
    def forward(ctx, xv, rvq, mode):
        q, idx, loss, usage, lm, lu, acc = _stages(rvq, xv, mode, True, True)
        ctx.save_for_backward(acc)
        ctx.weight = rvq.commitment_weight
        ctx.mark_non_differentiable(idx, usage, lm, lu)
        return q, idx, loss, usage, lm, lu

    @staticmethod
    def backward(ctx, grad_q, _gi, grad_loss, _gu, _gm, _gl):
        (acc,) = ctx.saved_tensors
        gm = None
        if grad_loss is not None and ctx.weight > 0:
            gm = grad_loss if ctx.weight == 1 else grad_loss * ctx.weight     # the autograd of `mse * w`
        gx = (ops._ste_bwd_impl if ops._fast() else ops.ste_bwd)(grad_q, acc, None, gm, 2.0 / acc.numel())
        return gx, None, None


class _RVQEval(torch.autograd.Function):
    """Eval forward of the Q stages; like VectorQuantizer's eval forward the gradient goes to the codebooks only:
    gE_l[k] = sum of g over the rows with idx_l = k (ordered under torch.use_deterministic_algorithms)."""

    @staticmethod
    def forward(ctx, xv, rvq, mode, *weights):
        q, idx, loss, usage, lm, lu, _ = _stages(rvq, xv, mode, False, False)
        ctx.save_for_backward(idx)
        ctx.num_codes = rvq.num_embeddings
        ctx.mark_non_differentiable(idx, loss, usage, lm, lu)
        return q, idx, loss, usage, lm, lu

    @staticmethod
    def backward(ctx, grad_q, *_):
        (idx,) = ctx.saved_tensors
        ge = [ops._codebook_grad(grad_q, idx[l], ctx.num_codes) if ctx.needs_input_grad[3 + l] else None
              for l in range(idx.shape[0])]
        return (None, None, None, *ge)


class ResidualVectorQuantizer(nn.Module):
    def __init__(self, dim, num_embeddings, num_quantizers, embedding_dim=None, decay=0.8, eps=1e-5, kmeans_init=False,
                 kmeans_iters=10, distance='euclidean', commitment_weight=1, num_codebook=1):
        super().__init__()
        if num_quantizers < 1:
            raise ValueError(f"num_quantizers must be >= 1, got {num_quantizers}")
        self.num_quantizers = num_quantizers
        self.num_embeddings = num_embeddings
        self.eps = eps
        self.commitment_weight = commitment_weight
        # Q consecutive constructions: a seeded init draws the codebooks in layer order
        self.layers = nn.ModuleList([
            VectorQuantizer(dim, num_embeddings, embedding_dim=embedding_dim, decay=decay, eps=eps,
                            kmeans_init=kmeans_init, kmeans_iters=kmeans_iters, distance=distance,
                            commitment_weight=commitment_weight, num_codebook=num_codebook)
            for _ in range(num_quantizers)])
        self.amp_compat = True    # round the gathered codes through the fp16 / bf16 autocast dtype, as VectorQuantizer
        self._graphs = None       # opt-in CUDA-graph cache of the no-grad forward (enable_cuda_graphs)

    def enable_cuda_graphs(self, max_entries: int = 16):
        """Opt-in: replay the no-grad forward as ONE CUDA graph per (input address, shape, strides), with
        VectorQuantizer.enable_cuda_graphs's contract: the returned tensors are buffers of the cache entry, overwritten by
        the next call with the same input address; weight updates are picked up; training-mode and grad-enabled calls,
        the k-means init and the EMA update take the ordinary path."""
        self._graphs = CudaGraphCache(max_entries)
        return self

    def disable_cuda_graphs(self):
        self._graphs = None
        return self

    def enable_ema(self, **kw):
        """Opt-in EMA update of every layer's codebook (VectorQuantizer.enable_ema: dead-code expiry, reduce / sync
        hooks).  Layer l is updated from r_l and its own indices right after its stage."""
        for layer in self.layers:
            layer.enable_ema(**kw)
        return self

    def forward(self, x, return_layer_stats=False):
        """(quantize, embed_index (B,H,W,Q), loss (1,), code_usage ()).  return_layer_stats=True returns loss and
        code_usage as (Q,) tensors instead: each layer's w * mean((q_l - r_l)^2) and its own unused-code percentage.
        These are statistics for monitoring: they carry no gradient (train with the pooled loss)."""
        if x.dim() != 4:
            raise ValueError(f"ResidualVectorQuantizer expects a (B, C, H, W) tensor, got shape {tuple(x.shape)}")
        if self.training:
            for layer in self.layers:
                cb = layer.codebook
                if cb.threshold_ema_dead_code > 0 and not cb.ema_enabled:
                    raise ValueError("threshold_ema_dead_code replaces codes after the EMA update: enable it through "
                                     "enable_ema()")
        if not x.is_cuda:
            raise RuntimeError("vq_seg_b200.ResidualVectorQuantizer runs on a B200 GPU only (no CPU fallback); "
                               "move the module and its input to cuda")
        if (self._graphs is not None and not self.training and not torch.is_grad_enabled() and x.numel() > 0
                and not torch.cuda.is_current_stream_capturing()):
            amp = ops.autocast_code_dtype(self.amp_compat)
            wptrs = tuple(layer.codebook.embedding.weight.data_ptr() for layer in self.layers)
            outs = self._graphs.run(self._forward_impl, x, (amp, wptrs),
                                    lambda: [layer.codebook._blob for layer in self.layers])
        else:
            outs = self._forward_impl(x)
        quantize, embed_index, loss, usage, layer_mse, layer_usage = outs
        if return_layer_stats:
            return quantize, embed_index, layer_mse * self.commitment_weight, layer_usage
        return quantize, embed_index, loss, usage

    def _forward_impl(self, x):
        x = x.to(torch.float32)
        b, c, h, w = x.shape
        device = x.device
        xv = x.reshape(b, c, h * w).permute(0, 2, 1)          # the 'b c h w -> b (h w) c' VIEW, no copy
        if xv.shape[-1] != self.layers[0].codebook.embedding_dim:
            raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {xv.shape[-1]} "
                               f"X2: {self.layers[0].codebook.embedding_dim}")
        mode = ops.gather_mode(self.training, ops.autocast_code_dtype(self.amp_compat))
        weights = [layer.codebook.embedding.weight for layer in self.layers]
        if self.training and torch.is_grad_enabled() and xv.requires_grad:
            q, idx, loss, usage, lm, lu = _RVQTrain.apply(xv, self, mode)
        elif not self.training and torch.is_grad_enabled() and any(wt.requires_grad for wt in weights):
            q, idx, loss, usage, lm, lu = _RVQEval.apply(xv, self, mode, *weights)
        else:
            q, idx, loss, usage, lm, lu, _ = _stages(self, xv, mode, self.training, False)
        # the loss rules of VectorQuantizer.forward (vq_img.py:230,239-241)
        if self.training and self.commitment_weight > 0 and not loss.requires_grad and torch.is_grad_enabled():
            loss = torch.zeros(1, device=device, dtype=torch.float32, requires_grad=True) + loss
        elif self.training and not self.commitment_weight > 0:
            loss = torch.zeros(1, device=device, dtype=torch.float32, requires_grad=True)
        quantize = q.permute(0, 2, 1).reshape(b, c, h, w)     # memory is already (B, C, H*W): a view
        embed_index = idx.reshape(len(self.layers), b, h, w).permute(1, 2, 3, 0)
        return quantize, embed_index, loss, usage, lm, lu

    @torch.no_grad()
    def get_output_from_indices(self, embed_index):
        """The eval quantize (B, C, H, W) of (B, H, W, Q) indices, in one launch (vqseg_rvq_decode_f32); the code is
        rounded like the forward's under autocast."""
        b, h, w, nq = embed_index.shape
        if nq != self.num_quantizers:
            raise ValueError(f"expected {self.num_quantizers} index layers, got {nq}")
        if not embed_index.is_cuda:
            raise RuntimeError("vq_seg_b200.ResidualVectorQuantizer runs on a B200 GPU only (no CPU fallback)")
        idx = embed_index.permute(3, 0, 1, 2).reshape(nq, b, h * w)
        codebooks = torch.stack([layer.codebook.embedding.weight.detach().float() for layer in self.layers])
        mode = ops.gather_mode(False, ops.autocast_code_dtype(self.amp_compat))
        out = (ops._rvq_decode_impl if ops._fast() else ops.rvq_decode)(idx, codebooks, mode)
        return out.permute(0, 2, 1).reshape(b, -1, h, w)
