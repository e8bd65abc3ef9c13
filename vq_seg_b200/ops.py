"""torch.library custom ops over the libvqseg C ABI + the straight-through autograd.Function.

Every op takes latent vectors as a logical (B, P, D) tensor with arbitrary strides -- the view
`rearrange(x, 'b c h w -> b (h w) c')` of the reference (vq_img.py:232) -- so NCHW feature maps are
consumed in place, never copied.  All ops run on the current CUDA stream and never synchronise.
"""
from typing import Optional, Tuple

import torch

from . import _native

ALGO_AUTO, ALGO_EXACT, ALGO_TC, ALGO_TC_STREAM, ALGO_TC_PAIR, ALGO_TC_TMA, ALGO_TC_STREAM_PAIR = 0, 1, 2, 3, 4, 5, 6
METRIC_IP = 0x100        # OR into an algo: first argmax of the fp32 inner product (cosine codebook) instead of cdist + argmin
MODE_EVAL, MODE_TRAIN, MODE_TRAIN_AMP, MODE_EVAL_AMP = 0, 1, 2, 3
MODE_TRAIN_AMP_BF16, MODE_EVAL_AMP_BF16 = 4, 5     # as MODE_*_AMP with E[idx] rounded through bf16 instead of fp16
MODE_ROTATE = 0x10       # OR into a train mode: quantize = E[idx] itself, gradient to x by the rotation trick (rotate_bwd)
_last_assign_ws = None


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("vq_seg_b200 kernels run on a B200 GPU only; got a CPU tensor "
                               "(there is no CPU fallback)")


def _bpd(t: torch.Tensor):
    assert t.dim() == 3, "expected a (B, P, D) view"
    return (t.shape[0], t.shape[1], t.shape[2], t.stride(0), t.stride(1), t.stride(2))


def _aligned_bytes(nbytes: int, device) -> torch.Tensor:
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    off = (-buf.data_ptr()) % 1024
    return buf[off:off + nbytes]


# -------------------------------------------------------------------------------------------------
def _prepare_codebook_impl(codebook: torch.Tensor, ip: bool = False) -> torch.Tensor:
    """fp32 |e|^2 (torch CPU summation order) + fp16 tcgen05 operand image; see vqseg.h.
    ip=True: the blob of an inner-product (cosine) lookup, whose score carries no |e|^2 term."""
    _require_cuda(codebook)
    L = _native.lib()
    cb = codebook.detach().contiguous().float()
    k, d = cb.shape
    n = L.vqseg_codebook_blob_bytes(k, d)
    blob = _aligned_bytes(n, cb.device)
    with torch.cuda.device(cb.device):
        fn = L.vqseg_codebook_prepare_ip_f32 if ip else L.vqseg_codebook_prepare_f32
        _native.check(fn(cb.data_ptr(), k, d, blob.data_ptr(), n, _stream()), "codebook_prepare")
    return blob


prepare_codebook = torch.library.custom_op("vqseg::prepare_codebook", mutates_args=())(_prepare_codebook_impl)


def _refresh_codebook_impl(blob: torch.Tensor, codebook: torch.Tensor, ip: bool = False) -> None:
    """Rebuild an existing blob (same K, D) from the current weights with the multi-block preparation kernels.  For
    callers that KNOW the weights just changed (the cosine codebook renormalises them every forward): the assignment's
    own guard would notice too, but rebuilds inside one block."""
    _require_cuda(blob, codebook)
    L = _native.lib()
    cb = codebook.detach().contiguous().float()
    k, d = cb.shape
    n = L.vqseg_codebook_blob_bytes(k, d)
    if blob.numel() < n:
        raise RuntimeError("refresh_codebook: the blob was prepared for another codebook shape")
    with torch.cuda.device(cb.device):
        fn = L.vqseg_codebook_prepare_ip_f32 if ip else L.vqseg_codebook_prepare_f32
        _native.check(fn(cb.data_ptr(), k, d, blob.data_ptr(), n, _stream()), "codebook_prepare")


refresh_codebook = torch.library.custom_op("vqseg::refresh_codebook", mutates_args=("blob",))(_refresh_codebook_impl)


@refresh_codebook.register_fake
def _(blob, codebook, ip=False):
    return None


@prepare_codebook.register_fake
def _(codebook, ip=False):
    k, d = codebook.shape
    return codebook.new_empty(_native.lib().vqseg_codebook_blob_bytes(k, d), dtype=torch.uint8)


_profile = None      # a _native.ProfileEvents while bench.py / scripts time the kernels of a call, else None


def set_profile_events(pe):
    """bench.py: hand the next assign / fused-forward calls four caller-owned CUDA events (None switches it off)."""
    global _profile
    _profile = pe


def _prof():
    return _profile.array if _profile is not None else None


def _prepare_samples_impl(x: torch.Tensor) -> torch.Tensor:
    """The fp16 operand tiles + row norms of the tensor-core filter for a (B, P, D) input that will be assigned many
    times (k-means: the same samples against new means every Lloyd iteration); pass it to assign(..., samples=)."""
    _require_cuda(x)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    b, p, d, sb, sp, sd = _bpd(x)
    n = L.vqseg_samples_blob_bytes(b * p, d)
    blob = _aligned_bytes(n, x.device)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_samples_prepare_f32(x.data_ptr(), b, p, d, sb, sp, sd, blob.data_ptr(), n, _stream()), "samples_prepare")
    return blob


prepare_samples = torch.library.custom_op("vqseg::prepare_samples", mutates_args=())(_prepare_samples_impl)


@prepare_samples.register_fake
def _(x):
    return x.new_empty(_native.lib().vqseg_samples_blob_bytes(x.shape[0] * x.shape[1], x.shape[2]), dtype=torch.uint8)


def _assign_impl(x: torch.Tensor, codebook: torch.Tensor, blob: Optional[torch.Tensor], algo: int = 0,
           kblock: int = 0, samples: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(idx (B,P) int64, counts (K,) int64): first-index argmin of the reference's fp32 cdist.
    `samples` = prepare_samples(x): the filter streams the prepared operand instead of converting x (same results)."""
    _require_cuda(x, codebook, blob, samples)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach().contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    if cb.shape[1] != d:
        raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {d} X2: {cb.shape[1]}")
    idx = torch.empty((b, p), dtype=torch.int64, device=x.device)
    counts = torch.zeros(k, dtype=torch.int64, device=x.device)
    nws = L.vqseg_assign_workspace_bytes(b * p, d, k, algo)
    ws = torch.empty(nws, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        if samples is not None and blob is not None and kblock == 0:
            _native.check(L.vqseg_assign_prepared_f32(x.data_ptr(), b, p, d, sb, sp, sd, samples.data_ptr(), cb.data_ptr(), k,
                                                      blob.data_ptr(), idx.data_ptr(), counts.data_ptr(), algo,
                                                      ws.data_ptr(), nws, _stream(), _prof()), "assign_prepared")
        else:
            _native.check(L.vqseg_assign_f32(x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k,
                                             blob.data_ptr() if blob is not None else None,
                                             idx.data_ptr(), counts.data_ptr(), None, 0, kblock, algo,
                                             ws.data_ptr(), nws, _stream(), _prof()), "assign")
    global _last_assign_ws
    _last_assign_ws = ws            # dev diagnostics: ws[0:4] = number of rows sent to the exact pass
    return idx, counts


assign = torch.library.custom_op("vqseg::assign", mutates_args=())(_assign_impl)


@assign.register_fake
def _(x, codebook, blob, algo=0, kblock=0, samples=None):
    return (x.new_empty((x.shape[0], x.shape[1]), dtype=torch.int64),
            x.new_empty((codebook.shape[0],), dtype=torch.int64))


def _assign_keys_impl(x: torch.Tensor, codebook: torch.Tensor, blob: Optional[torch.Tensor], code_base: int,
                algo: int = 0, kblock: int = 0) -> torch.Tensor:
    """Sharded mode: per row the packed key (float_bits(dist) << 32 | code_base + local idx) as int64."""
    _require_cuda(x, codebook, blob)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach().contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    keys = torch.empty((b, p), dtype=torch.int64, device=x.device)
    nws = L.vqseg_assign_workspace_bytes(b * p, d, k, algo)
    ws = torch.empty(nws, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_assign_f32(x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k,
                                         blob.data_ptr() if blob is not None else None,
                                         None, None, keys.data_ptr(), code_base, kblock, algo,
                                         ws.data_ptr(), nws, _stream(), None), "assign_keys")
    return keys


assign_keys = torch.library.custom_op("vqseg::assign_keys", mutates_args=())(_assign_keys_impl)


@assign_keys.register_fake
def _(x, codebook, blob, code_base, algo=0, kblock=0):
    return x.new_empty((x.shape[0], x.shape[1]), dtype=torch.int64)


def _unpack_keys_impl(keys: torch.Tensor, num_codes: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    _require_cuda(keys)
    L = _native.lib()
    keys = keys.contiguous()
    n = keys.numel()
    idx = torch.empty(keys.shape, dtype=torch.int64, device=keys.device)
    dist = torch.empty(keys.shape, dtype=torch.float32, device=keys.device)
    counts = torch.zeros(num_codes, dtype=torch.int64, device=keys.device)
    with torch.cuda.device(keys.device):
        _native.check(L.vqseg_unpack_keys(keys.data_ptr(), n, idx.data_ptr(), dist.data_ptr(), counts.data_ptr(),
                                          num_codes, _stream()), "unpack_keys")
    return idx, dist, counts


unpack_keys = torch.library.custom_op("vqseg::unpack_keys", mutates_args=())(_unpack_keys_impl)


@unpack_keys.register_fake
def _(keys, num_codes):
    return (keys.new_empty(keys.shape), keys.new_empty(keys.shape, dtype=torch.float32),
            keys.new_empty((num_codes,)))


def _gather_ste_impl(x: torch.Tensor, codebook: torch.Tensor, idx: torch.Tensor, mode: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(q (B,P,D) laid out like an NCHW map, mse (1,)): E[idx] (eval) or x + (E[idx] - x) (train)
    and mean((q - x)^2) in one pass."""
    _require_cuda(x, codebook, idx)
    L = _native.lib()
    cb = codebook.detach().contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    # output in the layout of the NCHW map the module returns: memory (B, D, P), logical (B, P, D)
    q = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device)
    loss = torch.zeros(1, dtype=torch.float32, device=x.device)
    nws = L.vqseg_gather_workspace_bytes(b * p, d)
    ws = torch.empty(nws, dtype=torch.uint8, device=x.device)
    idx = idx.contiguous()
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_gather_ste_f32(x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k, idx.data_ptr(),
                                             q.data_ptr(), q.stride(0), q.stride(1), q.stride(2),
                                             loss.data_ptr(), mode, ws.data_ptr(), nws, _stream()), "gather_ste")
    return q, loss


gather_ste = torch.library.custom_op("vqseg::gather_ste", mutates_args=())(_gather_ste_impl)


@gather_ste.register_fake
def _(x, codebook, idx, mode):
    b, p, d = x.shape
    return (torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device),
            x.new_empty((1,), dtype=torch.float32))


def _ste_bwd_impl(grad_q: Optional[torch.Tensor], x: torch.Tensor, q_ste: Optional[torch.Tensor],
            grad_mse: Optional[torch.Tensor], coef_scale: float) -> torch.Tensor:
    """gx = grad_q + coef_scale * grad_mse * (x - q_ste)   (coef_scale = 2 / numel).  q_ste=None stands for zeros:
    gx = fma(coef, x, grad_q), the residual quantizer's backward with x = the accumulated commitment term A."""
    _require_cuda(x, q_ste, grad_q, grad_mse)
    L = _native.lib()
    b, p, d, sb, sp, sd = _bpd(x)
    gx = torch.empty_like(x, dtype=torch.float32)      # preserve_format keeps the NCHW-view strides
    gq = grad_q
    if gq is not None and gq.dtype != torch.float32:
        gq = gq.float()
    g = (gq.data_ptr(), gq.stride(0), gq.stride(1), gq.stride(2)) if gq is not None else (None, 0, 0, 0)
    gm = grad_mse.reshape(-1)[:1].float().contiguous() if grad_mse is not None else None
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_ste_bwd_f32(g[0], g[1], g[2], g[3], x.data_ptr(), sb, sp, sd,
                                          *((q_ste.data_ptr(), *q_ste.stride()) if q_ste is not None else (None, 0, 0, 0)),
                                          gm.data_ptr() if gm is not None else None, coef_scale,
                                          gx.data_ptr(), gx.stride(0), gx.stride(1), gx.stride(2),
                                          b, p, d, _stream()), "ste_bwd")
    return gx


ste_bwd = torch.library.custom_op("vqseg::ste_bwd", mutates_args=())(_ste_bwd_impl)


@ste_bwd.register_fake
def _(grad_q, x, q_ste, grad_mse, coef_scale):
    return torch.empty_like(x, dtype=torch.float32)


def _rotate_bwd_impl(grad_q: Optional[torch.Tensor], x: torch.Tensor, q: torch.Tensor,
                     grad_mse: Optional[torch.Tensor], coef_scale: float) -> torch.Tensor:
    """The rotation trick's gradient w.r.t. x (vqseg.h, vqseg_rotate_bwd_f32): grad_q carried from q = E[idx] to x by the
    rotation taking x onto q, scaled by |q| / |x|, plus coef_scale * grad_mse * (x - q).  q is the forward's output."""
    _require_cuda(x, q, grad_q, grad_mse)
    L = _native.lib()
    b, p, d, sb, sp, sd = _bpd(x)
    gx = torch.empty_like(x, dtype=torch.float32)      # preserve_format keeps the NCHW-view strides
    gq = grad_q
    if gq is not None and gq.dtype != torch.float32:
        gq = gq.float()
    g = (gq.data_ptr(), gq.stride(0), gq.stride(1), gq.stride(2)) if gq is not None else (None, 0, 0, 0)
    gm = grad_mse.reshape(-1)[:1].float().contiguous() if grad_mse is not None else None
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_rotate_bwd_f32(g[0], g[1], g[2], g[3], x.data_ptr(), sb, sp, sd,
                                             q.data_ptr(), q.stride(0), q.stride(1), q.stride(2),
                                             gm.data_ptr() if gm is not None else None, coef_scale,
                                             gx.data_ptr(), gx.stride(0), gx.stride(1), gx.stride(2),
                                             b, p, d, _stream()), "rotate_bwd")
    return gx


rotate_bwd = torch.library.custom_op("vqseg::rotate_bwd", mutates_args=())(_rotate_bwd_impl)


@rotate_bwd.register_fake
def _(grad_q, x, q, grad_mse, coef_scale):
    return torch.empty_like(x, dtype=torch.float32)


def _x_grad(mode, grad_q, x, q, grad_mse):
    """gradient w.r.t. x of a training forward in `mode`: straight-through, or the rotation trick with MODE_ROTATE"""
    if mode & MODE_ROTATE:
        return (_rotate_bwd_impl if _fast() else rotate_bwd)(grad_q, x, q, grad_mse, 2.0 / x.numel())
    return (_ste_bwd_impl if _fast() else ste_bwd)(grad_q, x, q, grad_mse, 2.0 / x.numel())


# -------------------------------------------------------------------------------------------------
# residual vector quantization (opt-in extension, vqseg.h: vqseg_rvq_stage_f32 / vqseg_rvq_decode_f32)
def _rvq_stage_impl(r: torch.Tensor, rn: Optional[torch.Tensor], codebook: torch.Tensor, blob: Optional[torch.Tensor],
                    x: torch.Tensor, q: torch.Tensor, r_next: Optional[torch.Tensor], acc: Optional[torch.Tensor],
                    idx: torch.Tensor, counts: torch.Tensor, layer_mse: torch.Tensor, layer_usage: torch.Tensor,
                    loss: torch.Tensor, usage: torch.Tensor, layer: int, mode: int, algo: int, weight: float) -> None:
    """Stage `layer` of Q = idx.shape[0] in one host call: the lookup of r (Euclidean, or the inner product of its
    normalised rows rn for the cosine codebook), then per element S (into q), r_next = r - c, A (into acc, training)
    and, in the last training stage, quantize = x + (S - x) into q.  idx (Q, B, P) and counts (Q, K) get row `layer`;
    layer_mse / layer_usage (Q,) entry `layer`; the last stage writes the pooled loss (training) and usage."""
    _require_cuda(r, rn, codebook, blob, x, q, r_next, acc, idx, counts)
    L = _native.lib()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(r)
    k = cb.shape[0]
    if cb.shape[1] != d:
        raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {d} X2: {cb.shape[1]}")
    nq = idx.shape[0]
    for t in (q, r_next, acc):
        if t is not None and t.stride() != q.stride():
            raise RuntimeError("rvq_stage: q, r_next and acc must share strides")
    nws = L.vqseg_rvq_stage_workspace_bytes(b * p, d, k)
    ws = torch.empty(nws, dtype=torch.uint8, device=r.device)
    ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None  # noqa: E731
    rnv = (ptr(rn), *rn.stride()) if rn is not None else (None, 0, 0, 0)
    with torch.cuda.device(r.device):
        _native.check(L.vqseg_rvq_stage_f32(ptr(r), b, p, d, sb, sp, sd, *rnv, ptr(x), *x.stride(),
                                            cb.data_ptr(), k, ptr(blob), ptr(idx[layer]), counts.data_ptr(),
                                            ptr(q), *q.stride(), ptr(r_next), ptr(acc),
                                            layer_mse.data_ptr(), layer_usage.data_ptr(), ptr(loss), ptr(usage),
                                            layer, nq, float(weight), mode, algo, ws.data_ptr(), nws, _stream()),
                      "rvq_stage")


rvq_stage = torch.library.custom_op(
    "vqseg::rvq_stage",
    mutates_args=("q", "r_next", "acc", "idx", "counts", "layer_mse", "layer_usage", "loss", "usage"))(_rvq_stage_impl)


@rvq_stage.register_fake
def _(r, rn, codebook, blob, x, q, r_next, acc, idx, counts, layer_mse, layer_usage, loss, usage, layer, mode, algo,
      weight):
    return None


def _rvq_decode_impl(idx: torch.Tensor, codebooks: torch.Tensor, mode: int = 0) -> torch.Tensor:
    """S = sum over l of the rounded codes codebooks[l][idx[l]] in ascending l, from (Q, B, P) indices and (Q, K, D)
    codebooks: (B, P, D) in NCHW memory order, bit-equal to the eval forward's quantize.  mode: MODE_EVAL*."""
    _require_cuda(idx, codebooks)
    L = _native.lib()
    nq, b, p = idx.shape
    cb = codebooks.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    k, d = cb.shape[1], cb.shape[2]
    if cb.shape[0] != nq:
        raise RuntimeError(f"rvq_decode: {nq} index layers for {cb.shape[0]} codebooks")
    idx = idx.to(torch.int64).contiguous()
    out = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=idx.device)
    with torch.cuda.device(idx.device):
        _native.check(L.vqseg_rvq_decode_f32(idx.data_ptr() if idx.numel() else None, nq, b, p, cb.data_ptr(), k, d,
                                             out.data_ptr() if out.numel() else None, *out.stride(), mode, _stream()),
                      "rvq_decode")
    return out


rvq_decode = torch.library.custom_op("vqseg::rvq_decode", mutates_args=())(_rvq_decode_impl)


@rvq_decode.register_fake
def _(idx, codebooks, mode=0):
    nq, b, p = idx.shape
    d = codebooks.shape[2]
    return torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=idx.device)


def _gather_bwd_codebook_impl(grad_q: torch.Tensor, idx: torch.Tensor, num_codes: int) -> torch.Tensor:
    _require_cuda(grad_q, idx)
    L = _native.lib()
    gq = grad_q.float()
    b, p, d, sb, sp, sd = _bpd(gq)
    ge = torch.zeros((num_codes, d), dtype=torch.float32, device=gq.device)
    idx = idx.contiguous()
    with torch.cuda.device(gq.device):
        _native.check(L.vqseg_gather_bwd_codebook_f32(gq.data_ptr(), b, p, d, sb, sp, sd, idx.data_ptr(),
                                                      ge.data_ptr(), num_codes, _stream()), "gather_bwd_codebook")
    return ge


gather_bwd_codebook = torch.library.custom_op("vqseg::gather_bwd_codebook", mutates_args=())(_gather_bwd_codebook_impl)


@gather_bwd_codebook.register_fake
def _(grad_q, idx, num_codes):
    return grad_q.new_empty((num_codes, grad_q.shape[2]), dtype=torch.float32)


def _code_stats_impl(x: torch.Tensor, idx: torch.Tensor, num_codes: int, deterministic: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """(counts (K,) int64, sums (K, D) fp32) of the rows assigned to each code.  The sums are ordered (ascending rows)
    when `deterministic` is set or torch.use_deterministic_algorithms(True) is in force."""
    _require_cuda(x, idx)
    L = _native.lib()
    deterministic = deterministic or torch.are_deterministic_algorithms_enabled()
    if x.dtype != torch.float32:
        x = x.float()
    b, p, d, sb, sp, sd = _bpd(x)
    counts = torch.zeros(num_codes, dtype=torch.int64, device=x.device)
    sums = torch.zeros((num_codes, d), dtype=torch.float32, device=x.device)
    nws = L.vqseg_code_stats_workspace_bytes(b * p, d, num_codes, int(deterministic))
    ws = torch.empty(nws, dtype=torch.uint8, device=x.device)
    idx = idx.contiguous()
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_code_stats_f32(x.data_ptr(), b, p, d, sb, sp, sd, idx.data_ptr(), num_codes,
                                             counts.data_ptr(), sums.data_ptr(), int(deterministic),
                                             ws.data_ptr(), nws, _stream()), "code_stats")
    return counts, sums


code_stats = torch.library.custom_op("vqseg::code_stats", mutates_args=())(_code_stats_impl)


@code_stats.register_fake
def _(x, idx, num_codes, deterministic=True):
    return x.new_empty((num_codes,), dtype=torch.int64), x.new_empty((num_codes, x.shape[2]), dtype=torch.float32)


def _kmeans_finalize_impl(sums: torch.Tensor, counts: torch.Tensor, means: torch.Tensor, cosine: bool = False) -> None:
    _require_cuda(sums, counts, means)
    L = _native.lib()
    assert means.is_contiguous() and sums.is_contiguous() and counts.is_contiguous()
    k, d = means.shape
    with torch.cuda.device(means.device):
        _native.check(L.vqseg_kmeans_finalize_f32(sums.data_ptr(), counts.data_ptr(), means.data_ptr(), k, d,
                                                  int(cosine), _stream()), "kmeans_finalize")


kmeans_finalize = torch.library.custom_op("vqseg::kmeans_finalize", mutates_args=("means",))(_kmeans_finalize_impl)


def _code_usage_impl(counts: torch.Tensor) -> torch.Tensor:
    """0-dim fp32: percent of UNUSED codes (vq_img.py:173-175)."""
    _require_cuda(counts)
    L = _native.lib()
    counts = counts.contiguous()
    out = torch.empty((), dtype=torch.float32, device=counts.device)
    with torch.cuda.device(counts.device):
        _native.check(L.vqseg_code_usage(counts.data_ptr(), counts.numel(), out.data_ptr(), _stream()), "code_usage")
    return out


code_usage = torch.library.custom_op("vqseg::code_usage", mutates_args=())(_code_usage_impl)


@code_usage.register_fake
def _(counts):
    return counts.new_empty((), dtype=torch.float32)


def _gather_rows_impl(x: torch.Tensor, row_ids: torch.Tensor) -> torch.Tensor:
    _require_cuda(x, row_ids)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    b, p, d, sb, sp, sd = _bpd(x)
    ids = row_ids.to(torch.int64).contiguous()
    out = torch.empty((ids.numel(), d), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_gather_rows_f32(x.data_ptr(), b, p, d, sb, sp, sd, ids.data_ptr(), ids.numel(),
                                              out.data_ptr(), _stream()), "gather_rows")
    return out


gather_rows = torch.library.custom_op("vqseg::gather_rows", mutates_args=())(_gather_rows_impl)


@gather_rows.register_fake
def _(x, row_ids):
    return x.new_empty((row_ids.numel(), x.shape[2]), dtype=torch.float32)


def _dense_like(x: torch.Tensor) -> torch.Tensor:
    """an uninitialised dense tensor of x's shape whose dims are ordered like x's strides (what TensorIterator
    allocates for an elementwise result: NCHW maps viewed as (B, P, D) stay pixel-contiguous)"""
    order = sorted(range(x.dim()), key=lambda i: (x.stride(i), -i), reverse=True)
    strides, acc = [0] * x.dim(), 1
    for i in reversed(order):
        strides[i] = acc
        acc *= max(x.shape[i], 1)
    return torch.empty_strided(tuple(x.shape), tuple(strides), dtype=torch.float32, device=x.device)


def _l2norm_rows_impl(x: torch.Tensor) -> torch.Tensor:
    """F.normalize(x, p=2, dim=-1) of a (B, P, D) view in ATen's CPU arithmetic (bit-equal: the summation order
    follows the layout, see vqseg.h); the result keeps x's dim order like torch's."""
    _require_cuda(x)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    b, p, d, sb, sp, sd = _bpd(x)
    out = _dense_like(x)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_l2norm_f32(x.data_ptr(), b, p, d, sb, sp, sd, out.data_ptr(), out.stride(0), out.stride(1),
                                         out.stride(2), _stream()), "l2norm")
    return out


l2norm_rows = torch.library.custom_op("vqseg::l2norm_rows", mutates_args=())(_l2norm_rows_impl)


@l2norm_rows.register_fake
def _(x):
    return _dense_like(x)


def _l2norm_rows_inplace_impl(w: torch.Tensor) -> None:
    """w[k, :] /= max(|w[k, :]|, 1e-12) for a contiguous (K, D) codebook: `weight.data.copy_(l2norm(weight.data))`
    (vq_img.py:100) without the temporary."""
    _require_cuda(w)
    if w.dtype != torch.float32 or not w.is_contiguous() or w.dim() != 2:
        raise RuntimeError("l2norm_rows_ expects a contiguous fp32 (K, D) tensor")
    L = _native.lib()
    k, d = w.shape
    with torch.cuda.device(w.device):
        _native.check(L.vqseg_l2norm_f32(w.data_ptr(), 1, k, d, k * d, d, 1, w.data_ptr(), k * d, d, 1, _stream()), "l2norm_")


l2norm_rows_ = torch.library.custom_op("vqseg::l2norm_rows_", mutates_args=("w",))(_l2norm_rows_inplace_impl)


@l2norm_rows_.register_fake
def _(w):
    return None


def assign_cosine(xn: torch.Tensor, codebook: torch.Tensor, blob: Optional[torch.Tensor] = None, algo: int = ALGO_AUTO):
    """(idx, counts): first argmax_k <xn, e_k> as the reference's einsum + argmax computes it (vq_img.py:104-107):
    the tcgen05 filter + exact rescoring of `assign` in inner-product mode.  `blob` = prepare_codebook(e, ip=True)."""
    if blob is None and algo != ALGO_EXACT:
        blob = fast_prepare_codebook(codebook, True)
    return fast_assign(xn, codebook, blob, algo | METRIC_IP)


# -------------------------------------------------------------------------------------------------
# opt-in EMA codebook update (no reference counterpart: SURVEY.md 8f-4, parity unpinned)
def _ema_update_impl(counts: torch.Tensor, sums: torch.Tensor, cluster_size: torch.Tensor, embed_avg: torch.Tensor,
                     weight: torch.Tensor, decay: float, eps: float) -> None:
    """In place: cluster_size, embed_avg (moving averages) and weight (the new codebook)."""
    _require_cuda(counts, sums, cluster_size, embed_avg, weight)
    L = _native.lib()
    k, d = weight.shape
    assert counts.dtype == torch.int64 and counts.is_contiguous() and counts.numel() == k
    for t in (sums, cluster_size, embed_avg, weight):
        assert t.dtype == torch.float32 and t.is_contiguous()
    ws = torch.empty(4, dtype=torch.float32, device=weight.device)
    with torch.cuda.device(weight.device):
        _native.check(L.vqseg_ema_update_f32(counts.data_ptr(), sums.data_ptr(), cluster_size.data_ptr(),
                                             embed_avg.data_ptr(), weight.data_ptr(), k, d, float(decay), float(eps),
                                             ws.data_ptr(), _stream()), "ema_update")


ema_update = torch.library.custom_op("vqseg::ema_update", mutates_args=("cluster_size", "embed_avg", "weight"))(_ema_update_impl)


def _ema_update_expire_impl(counts: torch.Tensor, sums: torch.Tensor, cluster_size: torch.Tensor, embed_avg: torch.Tensor,
                            weight: torch.Tensor, decay: float, eps: float, threshold: float, reset: float,
                            cand: torch.Tensor, expired: torch.Tensor) -> None:
    """ema_update, then dead-code expiry (vqseg.h, vqseg_ema_update_expire_f32): the r-th code in ascending k whose
    updated cluster_size is < threshold takes row r of `cand` (K, D) as its weight, cand * reset as its embed_avg and
    `reset` as its cluster_size.  expired: int64 (2,) counters [last, total], updated on the device."""
    _require_cuda(counts, sums, cluster_size, embed_avg, weight, cand, expired)
    L = _native.lib()
    k, d = weight.shape
    assert counts.dtype == torch.int64 and counts.is_contiguous() and counts.numel() == k
    for t in (sums, cluster_size, embed_avg, weight, cand):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert cand.shape == (k, d), "cand must hold K packed rows"
    assert expired.dtype == torch.int64 and expired.is_contiguous() and expired.numel() == 2
    nws = L.vqseg_ema_expire_workspace_bytes(k)
    ws = torch.empty(nws, dtype=torch.uint8, device=weight.device)
    with torch.cuda.device(weight.device):
        _native.check(L.vqseg_ema_update_expire_f32(counts.data_ptr(), sums.data_ptr(), cluster_size.data_ptr(),
                                                    embed_avg.data_ptr(), weight.data_ptr(), k, d, float(decay),
                                                    float(eps), float(threshold), float(reset), cand.data_ptr(),
                                                    expired.data_ptr(), ws.data_ptr(), nws, _stream()), "ema_update_expire")


ema_update_expire = torch.library.custom_op(
    "vqseg::ema_update_expire", mutates_args=("cluster_size", "embed_avg", "weight", "expired"))(_ema_update_expire_impl)


@ema_update_expire.register_fake
def _(counts, sums, cluster_size, embed_avg, weight, decay, eps, threshold, reset, cand, expired):
    return None


# -------------------------------------------------------------------------------------------------
# distance map of the VQ segmentation head (models/modules/vq_segmentation_head.py:167-176 / :104-111)
def _dist_map_raw(x, codebook, cosine=False, with_score=False):
    """x (B, P, D) view (any strides; for cosine: rows already l2-normalised), codebook (K, D).
    Returns (dist (B, P, K) fp32 laid out as (B, K, P) in memory, idx (B, P) int64, counts (K,) int64, score or None)."""
    _require_cuda(x, codebook)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    if cb.shape[1] != d:
        raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {d} X2: {cb.shape[1]}")
    dev = x.device
    dist = torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=dev)
    idx = torch.empty((b, p), dtype=torch.int64, device=dev)
    counts = torch.empty(k, dtype=torch.int64, device=dev)
    score = torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=dev) if with_score else None
    with torch.cuda.device(dev):
        _native.check(L.vqseg_dist_map_f32(x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k, 1 if cosine else 0,
                                           dist.data_ptr(), dist.stride(0), dist.stride(1), dist.stride(2),
                                           idx.data_ptr(), counts.data_ptr(),
                                           score.data_ptr() if with_score else None, _stream()), "dist_map")
    return dist, idx, counts, score


def _dist_map_impl(x: torch.Tensor, codebook: torch.Tensor, cosine: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return _dist_map_raw(x, codebook, cosine, False)[:3]


dist_map = torch.library.custom_op("vqseg::dist_map", mutates_args=())(_dist_map_impl)


def _dist_score_map_impl(x: torch.Tensor, codebook: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Euclidean map plus the head's class scores softmax_k(1 - d_k / sum_j d_j) from the same kernel:
    (dist, score, idx, counts), dist and score (B, P, K) laid out as (B, K, P)."""
    dist, idx, counts, score = _dist_map_raw(x, codebook, False, True)
    return dist, score, idx, counts


dist_score_map = torch.library.custom_op("vqseg::dist_score_map", mutates_args=())(_dist_score_map_impl)


@dist_score_map.register_fake
def _(x, codebook):
    b, p, d = x.shape
    k = codebook.shape[0]
    mk = lambda: torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=x.device)  # noqa: E731
    return mk(), mk(), x.new_empty((b, p), dtype=torch.int64), x.new_empty((k,), dtype=torch.int64)


@dist_map.register_fake
def _(x, codebook, cosine=False):
    b, p, d = x.shape
    k = codebook.shape[0]
    return (torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=x.device),
            x.new_empty((b, p), dtype=torch.int64), x.new_empty((k,), dtype=torch.int64))


def _dist_map_bwd_impl(grad: torch.Tensor, dist: torch.Tensor, x: torch.Tensor,
                       codebook: torch.Tensor, score: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Backward of the Euclidean map (torch.cdist p=2): (gx with x's (B, P, D) shape in NCHW memory order, gE (K, D)).
    With `score` (the saved class scores) `grad` is the gradient w.r.t. those scores instead."""
    _require_cuda(grad, dist, x, codebook)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    g = grad.float()
    if g.stride() != dist.stride():
        g2 = torch.empty_strided(dist.shape, dist.stride(), dtype=torch.float32, device=dist.device)
        g2.copy_(g)
        g = g2
    gx = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device)
    ge = torch.empty((k, d), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_dist_map_bwd_f32(g.data_ptr(), dist.data_ptr(), dist.stride(0), dist.stride(1), dist.stride(2),
                                               x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k,
                                               gx.data_ptr(), gx.stride(0), gx.stride(1), gx.stride(2), ge.data_ptr(),
                                               score.data_ptr() if score is not None else None,
                                               _stream()), "dist_map_bwd")
    return gx, ge


dist_map_bwd = torch.library.custom_op("vqseg::dist_map_bwd", mutates_args=())(_dist_map_bwd_impl)


def _sim_map_bwd_impl(grad: torch.Tensor, sim: torch.Tensor, x: torch.Tensor, codebook: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Backward of the cosine similarity map l2norm(x) @ codebook^T (codebook rows already unit-norm):
    (gx with x's (B, P, D) shape in NCHW memory order, gE (K, D)).  `sim` only lends its strides to the gradient."""
    _require_cuda(grad, sim, x, codebook)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    g = grad.float()
    if g.stride() != sim.stride():
        g2 = torch.empty_strided(sim.shape, sim.stride(), dtype=torch.float32, device=sim.device)
        g2.copy_(g)
        g = g2
    gx = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device)
    ge = torch.empty((k, d), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_sim_map_bwd_f32(g.data_ptr(), g.stride(0), g.stride(1), g.stride(2),
                                              x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k,
                                              gx.data_ptr(), gx.stride(0), gx.stride(1), gx.stride(2), ge.data_ptr(),
                                              _stream()), "sim_map_bwd")
    return gx, ge


sim_map_bwd = torch.library.custom_op("vqseg::sim_map_bwd", mutates_args=())(_sim_map_bwd_impl)


@sim_map_bwd.register_fake
def _(grad, sim, x, codebook):
    b, p, d = x.shape
    return (torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device),
            x.new_empty((codebook.shape[0], d), dtype=torch.float32))


@dist_map_bwd.register_fake
def _(grad, dist, x, codebook, score=None):
    b, p, d = x.shape
    return (torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device),
            codebook.new_empty(codebook.shape, dtype=torch.float32))


# the head for any class count and width: vqseg_seghead_map_f32 picks the per-pixel kernels above where they apply
# (SEGHEAD_AUTO) and the register-tiled ones otherwise; PIXEL / TILED force one of them
SEGHEAD_AUTO, SEGHEAD_PIXEL, SEGHEAD_TILED = 0, 1, 2
SEGHEAD_DETERMINISTIC = 0x100   # OR into the algo of seghead_map_bwd: prototype gradient in a fixed summation order


def _seghead_map_raw(x, codebook, cosine=False, with_score=False, algo=SEGHEAD_AUTO):
    _require_cuda(x, codebook)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    if cb.shape[1] != d:
        raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {d} X2: {cb.shape[1]}")
    dev = x.device
    dist = torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=dev)
    idx = torch.empty((b, p), dtype=torch.int64, device=dev)
    counts = torch.empty(k, dtype=torch.int64, device=dev)
    score = torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=dev) if with_score else None
    with torch.cuda.device(dev):
        _native.check(L.vqseg_seghead_map_f32(x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k, 1 if cosine else 0,
                                              dist.data_ptr(), dist.stride(0), dist.stride(1), dist.stride(2),
                                              idx.data_ptr(), counts.data_ptr(),
                                              score.data_ptr() if with_score else None, algo, _stream()), "seghead_map")
    return dist, idx, counts, score


def _seghead_map_impl(x: torch.Tensor, codebook: torch.Tensor, cosine: bool = False,
                      algo: int = SEGHEAD_AUTO) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(map (B, P, K) laid out as (B, K, P), idx (B, P), counts (K,)) for any K and D: the Euclidean distance map
    (bit-equal to ATen's CPU cdist) + first argmin, or, with cosine=True, the similarity map of rows the caller has
    already l2-normalised + first argmax."""
    return _seghead_map_raw(x, codebook, cosine, False, algo)[:3]


seghead_map = torch.library.custom_op("vqseg::seghead_map", mutates_args=())(_seghead_map_impl)


@seghead_map.register_fake
def _(x, codebook, cosine=False, algo=SEGHEAD_AUTO):
    b, p, d = x.shape
    k = codebook.shape[0]
    return (torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=x.device),
            x.new_empty((b, p), dtype=torch.int64), x.new_empty((k,), dtype=torch.int64))


def _seghead_score_map_impl(x: torch.Tensor, codebook: torch.Tensor,
                            algo: int = SEGHEAD_AUTO) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Euclidean map plus the class scores softmax_k(1 - d_k / sum_j d_j) from the same launch, for any K and D:
    (dist, score, idx, counts)."""
    dist, idx, counts, score = _seghead_map_raw(x, codebook, False, True, algo)
    return dist, score, idx, counts


seghead_score_map = torch.library.custom_op("vqseg::seghead_score_map", mutates_args=())(_seghead_score_map_impl)


@seghead_score_map.register_fake
def _(x, codebook, algo=SEGHEAD_AUTO):
    b, p, d = x.shape
    k = codebook.shape[0]
    mk = lambda: torch.empty_strided((b, p, k), (k * p, 1, p), dtype=torch.float32, device=x.device)  # noqa: E731
    return mk(), mk(), x.new_empty((b, p), dtype=torch.int64), x.new_empty((k,), dtype=torch.int64)


def _seghead_map_bwd_impl(grad: torch.Tensor, dist: torch.Tensor, x: torch.Tensor, codebook: torch.Tensor,
                          cosine: bool = False, score: Optional[torch.Tensor] = None,
                          algo: int = SEGHEAD_AUTO) -> Tuple[torch.Tensor, torch.Tensor]:
    """Backward of seghead_map / seghead_score_map: (gx with x's (B, P, D) shape in NCHW memory order, gE (K, D)).
    `dist` is the saved map (the similarity map when cosine=True); with `score` (Euclidean only) `grad` is the
    gradient w.r.t. the class scores."""
    _require_cuda(grad, dist, x, codebook, score)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    g = grad.float()
    if g.stride() != dist.stride():
        g2 = torch.empty_strided(dist.shape, dist.stride(), dtype=torch.float32, device=dist.device)
        g2.copy_(g)
        g = g2
    gx = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device)
    ge = torch.empty((k, d), dtype=torch.float32, device=x.device)
    nws = L.vqseg_seghead_map_bwd_workspace_bytes(b * p, d, k, algo)
    ws = torch.empty(nws, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(L.vqseg_seghead_map_bwd_f32(g.data_ptr(), dist.data_ptr(), dist.stride(0), dist.stride(1),
                                                  dist.stride(2), x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k,
                                                  1 if cosine else 0, score.data_ptr() if score is not None else None,
                                                  gx.data_ptr(), gx.stride(0), gx.stride(1), gx.stride(2), ge.data_ptr(),
                                                  algo, ws.data_ptr() if nws else None, nws, _stream()), "seghead_map_bwd")
    return gx, ge


seghead_map_bwd = torch.library.custom_op("vqseg::seghead_map_bwd", mutates_args=())(_seghead_map_bwd_impl)


@seghead_map_bwd.register_fake
def _(grad, dist, x, codebook, cosine=False, score=None, algo=SEGHEAD_AUTO):
    b, p, d = x.shape
    return (torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device),
            codebook.new_empty(codebook.shape, dtype=torch.float32))


def fast_seghead_map(x, codebook, cosine=False, algo=SEGHEAD_AUTO):
    return (_seghead_map_impl if _fast() else seghead_map)(x, codebook, cosine, algo)


def fast_seghead_map_bwd(grad, dist, x, codebook, cosine=False, score=None, algo=SEGHEAD_AUTO):
    """seghead_map_bwd for the head's autograd functions: deterministic under torch.use_deterministic_algorithms(True)"""
    if torch.are_deterministic_algorithms_enabled():
        algo |= SEGHEAD_DETERMINISTIC
    return (_seghead_map_bwd_impl if _fast() else seghead_map_bwd)(grad, dist, x, codebook, cosine, score, algo)


class _EuclideanDistMap(torch.autograd.Function):
    """torch.cdist(x, weight, p=2) + argmin + bincount with the map as a differentiable output
    (vq_segmentation_head.py:167-174): gradients to the features AND to the prototypes."""

    @staticmethod
    def forward(ctx, x, weight):
        dist, idx, counts = fast_seghead_map(x, weight, False)
        ctx.save_for_backward(x, weight, dist)
        ctx.mark_non_differentiable(idx, counts)
        return dist, idx, counts

    @staticmethod
    def backward(ctx, g_dist, g_idx, g_counts):
        x, weight, dist = ctx.saved_tensors
        gx, ge = fast_seghead_map_bwd(g_dist, dist, x, weight)
        return (gx if ctx.needs_input_grad[0] else None), (ge if ctx.needs_input_grad[1] else None)


def euclidean_dist_map(x, weight):
    return _EuclideanDistMap.apply(x, weight)


class _EuclideanScoreMap(torch.autograd.Function):
    """The whole score path of the Euclidean head in one kernel each way: cdist -> 1 - d / sum(d) -> softmax
    (vq_segmentation_head.py:167,243-247).  Differentiable output: score; idx / counts are not."""

    @staticmethod
    def forward(ctx, x, weight):
        dist, score, idx, counts = (_seghead_score_map_impl if _fast() else seghead_score_map)(x, weight)
        ctx.save_for_backward(x, weight, dist, score)
        ctx.mark_non_differentiable(idx, counts)
        return score, idx, counts

    @staticmethod
    def backward(ctx, g_score, g_idx, g_counts):
        x, weight, dist, score = ctx.saved_tensors
        gx, ge = fast_seghead_map_bwd(g_score, dist, x, weight, False, score)
        return (gx if ctx.needs_input_grad[0] else None), (ge if ctx.needs_input_grad[1] else None)


def euclidean_score_map(x, weight):
    return _EuclideanScoreMap.apply(x, weight)


# -------------------------------------------------------------------------------------------------
def _vq_forward_counts(x, codebook, blob, mode, algo=0):
    """_vq_forward_impl plus the per-code counts (for a global, all-reduced code usage)."""
    return _vq_forward_raw(x, codebook, blob, mode, algo)


def _vq_forward_impl(x: torch.Tensor, codebook: torch.Tensor, blob: Optional[torch.Tensor], mode: int,
                     algo: int = 0) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    return _vq_forward_raw(x, codebook, blob, mode, algo)[:4]


def _vq_forward_raw(x, codebook, blob, mode, algo=0):
    """(q (B,P,D) in NCHW memory order, idx (B,P) int64, mse (1,), code_usage ()): the whole forward of
    vq_img.py:228-244 (minus the k-means hook) enqueued by ONE host call."""
    _require_cuda(x, codebook, blob)
    L = _native.lib()
    if x.dtype != torch.float32:
        x = x.float()
    cb = codebook.detach()
    if cb.dtype != torch.float32 or not cb.is_contiguous():
        cb = cb.contiguous().float()
    b, p, d, sb, sp, sd = _bpd(x)
    k = cb.shape[0]
    if cb.shape[1] != d:
        raise RuntimeError(f"X1 and X2 must have the same number of columns. X1: {d} X2: {cb.shape[1]}")
    dev = x.device
    idx = torch.empty((b, p), dtype=torch.int64, device=dev)
    counts = torch.empty(k, dtype=torch.int64, device=dev)
    usage = torch.empty((), dtype=torch.float32, device=dev)
    q = torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    nws = L.vqseg_forward_workspace_bytes(b * p, d, k)
    ws = torch.empty(nws, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _native.check(L.vqseg_vq_forward_f32(x.data_ptr(), b, p, d, sb, sp, sd, cb.data_ptr(), k,
                                             blob.data_ptr() if blob is not None else None,
                                             idx.data_ptr(), counts.data_ptr(), usage.data_ptr(),
                                             q.data_ptr(), q.stride(0), q.stride(1), q.stride(2), loss.data_ptr(),
                                             mode, algo, 0, ws.data_ptr(), nws, _stream(), _prof()), "vq_forward")
    return q, idx, loss, usage, counts


vq_forward = torch.library.custom_op("vqseg::vq_forward", mutates_args=())(_vq_forward_impl)


@vq_forward.register_fake
def _(x, codebook, blob, mode, algo=0):
    b, p, d = x.shape
    return (torch.empty_strided((b, p, d), (d * p, 1, p), dtype=torch.float32, device=x.device),
            x.new_empty((b, p), dtype=torch.int64), x.new_empty((1,), dtype=torch.float32),
            x.new_empty((), dtype=torch.float32))


def _fast():
    """Eager fast path: call the Python implementations directly instead of going through the
    torch.library dispatcher (saves ~20 us of host time per op); the registered custom ops are used
    whenever a graph is being traced / compiled."""
    return not torch.compiler.is_compiling()


class _StraightThrough(torch.autograd.Function):
    """Training forward of vq_img.py:235-240: q_ste = x + (E[idx] - x), mse = mean((q_ste - x)^2).
    Gradients: d q_ste / dx = I (straight-through), d mse / dx = 2 (x - q_ste) / numel; the codebook
    gets none (the reference detaches it, SURVEY.md §0).  With MODE_ROTATE in `mode`: q = E[idx] and the
    rotation trick's gradient (rotate_bwd)."""

    @staticmethod
    def forward(ctx, x, codebook, idx, mode):
        q, mse = (_gather_ste_impl if _fast() else gather_ste)(x, codebook, idx, mode)
        ctx.save_for_backward(x, q)
        ctx.mark_non_differentiable(idx)
        ctx.mode = mode
        return q, mse

    @staticmethod
    def backward(ctx, grad_q, grad_mse):
        x, q = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None, None
        return _x_grad(ctx.mode, grad_q, x, q, grad_mse), None, None, None


def _codebook_grad(grad_q, idx, num_codes):
    """gE[k] = sum of grad_q over the rows assigned to k.  Under torch.use_deterministic_algorithms(True): the ordered
    per-code sums of code_stats (one fp32 chain per (code, dim) in ascending rows, the order of CPU index_add_)
    instead of the atomic kernel."""
    if torch.are_deterministic_algorithms_enabled():
        return (_code_stats_impl if _fast() else code_stats)(grad_q, idx, num_codes, True)[1]
    return (_gather_bwd_codebook_impl if _fast() else gather_bwd_codebook)(grad_q, idx, num_codes)


class _EvalGather(torch.autograd.Function):
    """Eval forward: q = E[idx].  Like the reference's one_hot matmul (vq_img.py:169-170) the gradient
    goes to the codebook only."""

    @staticmethod
    def forward(ctx, codebook, x_like, idx, mode):
        q, _ = (_gather_ste_impl if _fast() else gather_ste)(x_like, codebook, idx, mode)
        ctx.save_for_backward(idx)
        ctx.num_codes = codebook.shape[0]
        return q

    @staticmethod
    def backward(ctx, grad_q):
        (idx,) = ctx.saved_tensors
        ge = _codebook_grad(grad_q, idx, ctx.num_codes) if ctx.needs_input_grad[0] else None
        return ge, None, None, None


class _FusedTrainForward(torch.autograd.Function):
    """Training forward in one host call: lookup + STE + commitment mse + usage.  Same gradients as
    _StraightThrough (identity to x, 2 (x - q) / numel from the mse; nothing to the codebook; the rotation
    trick with MODE_ROTATE)."""

    @staticmethod
    def forward(ctx, x, codebook, blob, mode, algo):
        q, idx, mse, usage = (_vq_forward_impl if _fast() else vq_forward)(x, codebook, blob, mode, algo)
        ctx.save_for_backward(x, q)
        ctx.mark_non_differentiable(idx, usage)
        ctx.mode = mode
        return q, idx, mse, usage

    @staticmethod
    def backward(ctx, grad_q, _gi, grad_mse, _gu):
        x, q = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None, None, None
        return _x_grad(ctx.mode, grad_q, x, q, grad_mse), None, None, None, None


class _FusedEvalForward(torch.autograd.Function):
    """Eval forward in one host call; like the reference's one-hot matmul the gradient goes to the codebook."""

    @staticmethod
    def forward(ctx, codebook, x, blob, mode, algo):
        q, idx, mse, usage = (_vq_forward_impl if _fast() else vq_forward)(x, codebook, blob, mode, algo)
        ctx.save_for_backward(idx)
        ctx.num_codes = codebook.shape[0]
        ctx.mark_non_differentiable(idx, usage, mse)
        return q, idx, mse, usage

    @staticmethod
    def backward(ctx, grad_q, _gi, _gm, _gu):
        (idx,) = ctx.saved_tensors
        ge = _codebook_grad(grad_q, idx, ctx.num_codes) if ctx.needs_input_grad[0] else None
        return ge, None, None, None, None


def autocast_code_dtype(amp_compat=True):
    """The dtype the reference's one-hot matmul (vq_img.py:169-170) rounds the gathered code through in this context:
    torch.float16 / torch.bfloat16 under CUDA autocast to that dtype, None (exact fp32 codes) without autocast or
    with amp_compat=False.  Indices are not affected: cdist is on autocast's fp32 list."""
    if not (amp_compat and torch.is_autocast_enabled()):
        return None
    dtype = torch.get_autocast_dtype('cuda')
    return dtype if dtype in (torch.float16, torch.bfloat16) else None


def gather_mode(training, amp=None, rotate=False):
    """The gather mode (MODE_*) that rounds the code through `amp`: None for exact fp32 codes, torch.float16 or
    torch.bfloat16 (autocast_code_dtype()); False / True stand for None / torch.float16.  rotate=True (training only)
    adds MODE_ROTATE: the rotation trick instead of the straight-through estimator."""
    if rotate and not training:
        raise ValueError("the rotation trick applies to training forwards only")
    rot = MODE_ROTATE if rotate else 0
    if amp is None or amp is False:
        return MODE_TRAIN | rot if training else MODE_EVAL
    if amp is True or amp == torch.float16:
        return MODE_TRAIN_AMP | rot if training else MODE_EVAL_AMP
    if amp == torch.bfloat16:
        return MODE_TRAIN_AMP_BF16 | rot if training else MODE_EVAL_AMP_BF16
    raise ValueError(f"the gathered code can be rounded through torch.float16 or torch.bfloat16, not {amp}")


def fused_forward(x, weight, blob, training, amp=None, algo=ALGO_AUTO, rotate=False):
    """(q, idx, mse, usage) with autograd attached when needed; `amp` and `rotate` as in gather_mode."""
    mode = gather_mode(training, amp, rotate)
    if training:
        if torch.is_grad_enabled() and x.requires_grad:
            return _FusedTrainForward.apply(x, weight.detach(), blob, mode, algo)
        return (_vq_forward_impl if _fast() else vq_forward)(x, weight, blob, mode, algo)
    if torch.is_grad_enabled() and weight.requires_grad:
        return _FusedEvalForward.apply(weight, x, blob, mode, algo)
    return (_vq_forward_impl if _fast() else vq_forward)(x, weight, blob, mode, algo)


def straight_through(x, codebook, idx, amp=None, rotate=False):
    return _StraightThrough.apply(x, codebook, idx, gather_mode(True, amp, rotate))


def eval_gather(codebook, x_like, idx, amp=None):
    return _EvalGather.apply(codebook, x_like, idx, gather_mode(False, amp))


def fast_assign(x, codebook, blob, algo=ALGO_AUTO, kblock=0, samples=None):
    return (_assign_impl if _fast() else assign)(x, codebook, blob, algo, kblock, samples)


def fast_code_usage(counts):
    return (_code_usage_impl if _fast() else code_usage)(counts)


def fast_refresh_codebook(blob, codebook, ip=False):
    return (_refresh_codebook_impl if _fast() else refresh_codebook)(blob, codebook, ip)


def fast_prepare_codebook(codebook, ip=False):
    return (_prepare_codebook_impl if _fast() else prepare_codebook)(codebook, ip)
