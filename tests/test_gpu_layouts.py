"""Every entry point that takes a strided (B, P, D) view, over the layout catalogue of tests/layouts.py (channels-last
maps, channel and batch slices, misaligned bases, CNHW views, 1 x 1 maps, expanded batches).  The kernels choose
their paths by layout, so each result is checked twice:
  (i)  bit-equal to the same call on the packed copy of the view (layout-specific indexing and dispatch);
  (ii) against a CPU or float64 reference of the same operation (bugs common to all layouts).
A forced algorithm may refuse a layout only with "not supported"; AUTO must take every valid view."""
import pytest
import torch
import torch.nn.functional as F
from torch import nn

import layouts
from oracle import vq_oracle as O

pytestmark = pytest.mark.gpu

EPS = torch.finfo(torch.float32).eps
CASES = layouts.cases()
WRITABLE_CASES = layouts.cases(layouts.WRITABLE)
ASSIGN_ALGOS = ("ALGO_EXACT", "ALGO_AUTO", "ALGO_TC_STREAM", "ALGO_TC_PAIR", "ALGO_TC_TMA", "ALGO_TC_STREAM_PAIR")
# classes of the segmentation-head tests: at most 32 (the per-pixel kernels' limit) and more than 25, so that CPU cdist
# takes the augmented GEMM form the kernels restate for every shape (with at most 25 rows and 25 classes it takes exact
# differences instead, and its fp32 error would not bound the cancellation of the augmented form)
K_SEG = 27


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


def setup(case, dev, seed=0):
    """(v, vg, e, eg): the case's (B, P, D) view on the CPU and on the GPU (same strides, same values) and a codebook
    of rows near feature rows"""
    layout, s = case
    shape, k = layouts.SHAPES[s]
    full, x = layouts.make(layout, shape, seed)
    fg, xg = layouts.make(layout, shape, seed, dev)
    v, vg = layouts.bpd(x, full, layout), layouts.bpd(xg, fg, layout)
    g = torch.Generator().manual_seed(seed + 1)
    rows = v.reshape(-1, shape[1])
    e = rows[torch.randint(0, rows.shape[0], (k,), generator=g)] + 0.05 * torch.randn(k, shape[1], generator=g)
    return v, vg, e, e.to(dev)


def rel_to_max(a, b):
    return (a.double() - b.double()).abs().max().item() / max(b.double().abs().max().item(), 1e-30)


def forced(fn, name):
    """fn() for a forced algorithm: None when it refuses the layout, which it may only do as 'not supported'"""
    try:
        return fn()
    except RuntimeError as ex:
        if name in ("ALGO_AUTO", "ALGO_EXACT") or "not supported" not in str(ex):
            raise
        return None


def euclid_tie_ok(v, e, idx, ref):
    """rows where idx and ref differ are within 2 ulp in the reference's own fp32 distances"""
    bad = (idx != ref).nonzero()
    if bad.numel() == 0:
        return True
    d = O.euclidean_dist(v, e)
    for b, p in bad.tolist():
        dg, dr = d[b, p, idx[b, p]], d[b, p, ref[b, p]]
        if not (dg - dr).abs() <= 2 * EPS * dr.abs():
            return False
    return True


def ip_tie_ok(v, e, idx):
    """idx is a float64 argmax of <x, e_k> up to two roundings at the magnitude of the fp32 dot products"""
    s = torch.einsum("bpd,kd->bpk", v.double(), e.double())
    mag = torch.einsum("bpd,kd->bpk", v.double().abs(), e.double().abs())
    best = s.argmax(-1)
    got, top = s.gather(-1, idx.unsqueeze(-1))[..., 0], s.gather(-1, best.unsqueeze(-1))[..., 0]
    return bool(((top - got) <= 2 * EPS * mag.gather(-1, best.unsqueeze(-1))[..., 0]).all())


# ---- assignment ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", ["euclidean", "ip"])
@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_assign_every_algorithm(dev, case, metric):
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    ip = metric == "ip"
    flag = ops.METRIC_IP if ip else 0
    blob = ops.prepare_codebook(eg, ip)
    pk = vg.contiguous()
    i_ex, c_ex = ops.assign(vg, eg, None, ops.ALGO_EXACT | flag)
    assert torch.equal(c_ex.cpu(), torch.bincount(i_ex.cpu().reshape(-1), minlength=e.shape[0]))
    if ip:
        assert ip_tie_ok(v, e, i_ex.cpu())
    else:
        assert euclid_tie_ok(v, e, i_ex.cpu(), O.assign_euclidean(v, e))
    bad = []
    runs = [(n, (lambda x, a=getattr(ops, n): ops.assign(x, eg, None if a == ops.ALGO_EXACT else blob, a | flag)))
            for n in ASSIGN_ALGOS]
    if not ip:
        runs.append(("prepared", lambda x: ops.assign(x, eg, blob, ops.ALGO_AUTO, 0, ops.prepare_samples(x))))
    for name, run in runs:
        got = forced(lambda: run(vg), name)
        if got is None:
            continue
        if not (torch.equal(got[0], i_ex) and torch.equal(got[1], c_ex)):
            bad.append((name, "exact scorer", (got[0] != i_ex).sum().item()))
        ref = forced(lambda: run(pk), name)
        if ref is not None and not (torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])):
            bad.append((name, "packed copy", (got[0] != ref[0]).sum().item()))
    assert not bad, bad


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_assign_keys_distances(dev, case):
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    blob = ops.prepare_codebook(eg)
    for algo, b in ((ops.ALGO_EXACT, None), (ops.ALGO_AUTO, blob)):
        i1, d1, c1 = ops.unpack_keys(ops.assign_keys(vg, eg, b, 5, algo), e.shape[0] + 5)
        i2, d2, c2 = ops.unpack_keys(ops.assign_keys(vg.contiguous(), eg, b, 5, algo), e.shape[0] + 5)
        assert torch.equal(i1, i2) and torch.equal(d1, d2) and torch.equal(c1, c2), algo
        assert torch.equal(i1 - 5, ops.assign(vg, eg, None, ops.ALGO_EXACT)[0])


# ---- forward: gather, straight-through estimator, loss, usage ------------------------------------------------------
def expected_q(vg, eg, idx, mode):
    from vq_seg_b200 import ops
    code = eg[idx]
    if mode in (ops.MODE_TRAIN_AMP, ops.MODE_EVAL_AMP):
        code = code.half().float()
    return vg + (code - vg) if mode in (ops.MODE_TRAIN, ops.MODE_TRAIN_AMP) else code


def check_loss(loss, q, v, train):
    if not train:
        assert loss.item() == 0.0
        return
    ref = (q.cpu().double() - v.double()).pow(2).mean().item()
    assert abs(loss.item() - ref) <= 1e-6 * ref, (loss.item(), ref)


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_vq_forward_all_modes(dev, case):
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    blob = ops.prepare_codebook(eg)
    i_ex = ops.assign(vg, eg, None, ops.ALGO_EXACT)[0]
    k = e.shape[0]
    for mode in (ops.MODE_EVAL, ops.MODE_TRAIN, ops.MODE_TRAIN_AMP, ops.MODE_EVAL_AMP):
        q, idx, loss, usage = ops.vq_forward(vg, eg, blob, mode)
        qp, idxp, _, usagep = ops.vq_forward(vg.contiguous(), eg, blob, mode)
        assert torch.equal(idx, i_ex) and torch.equal(idx, idxp), mode
        assert torch.equal(q, expected_q(vg, eg, idx, mode)) and torch.equal(q, qp), mode
        assert torch.equal(usage.cpu(), O.code_usage_from_counts(torch.bincount(idx.cpu().reshape(-1), minlength=k), k))
        assert torch.equal(usage, usagep)
        check_loss(loss, q, v, mode in (ops.MODE_TRAIN, ops.MODE_TRAIN_AMP))


@pytest.mark.parametrize("case", WRITABLE_CASES, ids=layouts.case_id)
def test_raw_gather_writes_q_in_the_layout_of_x(dev, case):
    """vqseg_gather_ste_f32 with q_out strided like x (the ops wrapper always allocates NCHW order): every element of
    the view written, nothing around it"""
    from vq_seg_b200 import _native, ops
    v, vg, e, eg = setup(case, dev)
    layout, s = case
    L = _native.lib()
    idx = ops.assign(vg, eg, None, ops.ALGO_EXACT)[0]
    b, p, d = vg.shape
    for mode in (ops.MODE_EVAL, ops.MODE_TRAIN, ops.MODE_TRAIN_AMP, ops.MODE_EVAL_AMP):
        qfull, qx = layouts.make(layout, layouts.SHAPES[s][0], 9, dev)
        qfull.fill_(float("nan"))
        q = layouts.bpd(qx, qfull, layout)
        loss = torch.zeros(1, device=dev)
        nws = L.vqseg_gather_workspace_bytes(b * p, d)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        _native.check(L.vqseg_gather_ste_f32(vg.data_ptr(), b, p, d, *vg.stride(), eg.data_ptr(), e.shape[0],
                                             idx.data_ptr(), q.data_ptr(), *q.stride(), loss.data_ptr(), mode,
                                             ws.data_ptr(), nws, torch.cuda.current_stream().cuda_stream), "gather_ste")
        assert torch.equal(q, expected_q(vg, eg, idx, mode)), mode
        assert qfull.isnan().sum().item() == qfull.numel() - q.numel(), "wrote outside the view"
        check_loss(loss, q, v, mode in (ops.MODE_TRAIN, ops.MODE_TRAIN_AMP))


def grad_like(shape, order, seed, dev):
    """a (B, P, D) gradient in NCHW order (pixel-contiguous) or channels-last order (packed rows)"""
    b, p, d = shape
    g = torch.randn(b, d, p, generator=torch.Generator().manual_seed(seed))
    g = g.permute(0, 2, 1) if order == "nchw" else g.permute(0, 2, 1).contiguous()
    return g.to(dev)


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_ste_backward(dev, case):
    """gx = g + coef * (x - q) as one fma: within 1 ulp of the float64 evaluation of g + coef * fl(x - q)"""
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    q = ops.vq_forward(vg, eg, ops.prepare_codebook(eg), ops.MODE_TRAIN)[0]
    gm = torch.tensor([1.7], device=dev)
    scale = 2.0 / vg.numel()
    coef = (torch.tensor(scale, dtype=torch.float32) * gm.cpu()).double()
    for order in ("nchw", "nhwc"):
        g = grad_like(vg.shape, order, 3, dev)
        gx = ops.ste_bwd(g, vg, q, gm, scale)
        assert torch.equal(gx, ops.ste_bwd(g, vg.contiguous(), q, gm, scale)), order
        ref = g.cpu().double() + coef * (v - q.cpu()).double()
        assert ((gx.cpu().double() - ref).abs() <= EPS * ref.abs()).all(), order
        assert torch.equal(ops.ste_bwd(g, vg, q, None, scale), g), order        # no loss term: the gradient itself


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_gather_backward_to_the_codebook(dev, case):
    """the case's view as the incoming gradient: gE[idx[n]] += g[n] against a float64 index_add_"""
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    k = e.shape[0]
    idx = torch.randint(0, k, vg.shape[:2], generator=torch.Generator().manual_seed(5))
    ge = ops.gather_bwd_codebook(vg, idx.to(dev), k)
    ref = torch.zeros(k, v.shape[2], dtype=torch.float64).index_add_(0, idx.reshape(-1), v.reshape(-1, v.shape[2]).double())
    assert rel_to_max(ge.cpu(), ref) <= 1e-6


# ---- k-means building blocks ---------------------------------------------------------------------------------------
def skewed_idx(shape, k, seed):
    """code ids with a few large clusters and many small ones"""
    g = torch.Generator().manual_seed(seed)
    big = torch.randint(0, 4, shape, generator=g)
    small = torch.randint(0, k, shape, generator=g)
    return torch.where(torch.rand(shape, generator=g) < 0.5, big, small)


def ordered_sums(v, idx, k):
    """the reference's sequential CPU scatter_add_ in row order (vq_img.py:47-51)"""
    rows = v.reshape(-1, v.shape[-1])
    i = idx.reshape(-1, 1).expand(-1, rows.shape[1]).contiguous()
    return torch.zeros(k, rows.shape[1]).scatter_add_(0, i, rows)


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_code_stats(dev, case):
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    k = e.shape[0]
    idx = skewed_idx(vg.shape[:2], k, 6)
    counts_ref = torch.bincount(idx.reshape(-1), minlength=k)
    c1, s1 = ops.code_stats(vg, idx.to(dev), k, True)
    assert torch.equal(c1.cpu(), counts_ref)
    assert torch.equal(s1.cpu(), ordered_sums(v, idx, k))
    c2, s2 = ops.code_stats(vg, idx.to(dev), k, False)
    assert torch.equal(c2.cpu(), counts_ref)
    ref64 = torch.zeros(k, v.shape[2], dtype=torch.float64).index_add_(0, idx.reshape(-1), v.reshape(-1, v.shape[2]).double())
    assert rel_to_max(s2.cpu(), ref64) <= 1e-5


def test_code_stats_sorted_windows_on_padded_rows(dev):
    """>= 2^18 channels-last rows padded to C + 8 floats: the unordered statistics take the counting sort and the
    sorted-window sums with a row pitch wider than D"""
    from vq_seg_b200 import ops
    shape, k = (3, 100, 400, 250), 300
    full, x = layouts.make("nhwc_ch_slice", shape, 11, dev)
    vg = layouts.bpd(x, full, "nhwc_ch_slice")
    idx = skewed_idx(vg.shape[:2], k, 12)
    c, s = ops.code_stats(vg, idx.to(dev), k, False)
    v = vg.cpu()
    assert torch.equal(c.cpu(), torch.bincount(idx.reshape(-1), minlength=k))
    ref64 = torch.zeros(k, 100, dtype=torch.float64).index_add_(0, idx.reshape(-1), v.reshape(-1, 100).double())
    assert rel_to_max(s.cpu(), ref64) <= 1e-5
    c1, s1 = ops.code_stats(vg, idx.to(dev), k, True)
    assert torch.equal(c1, c) and torch.equal(s1.cpu(), ordered_sums(v, idx, k))


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_gather_rows(dev, case):
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    n = v.shape[0] * v.shape[1]
    ids = torch.randint(0, n, (77,), generator=torch.Generator().manual_seed(7))
    assert torch.equal(ops.gather_rows(vg, ids.to(dev)).cpu(), v.reshape(n, -1)[ids])


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_l2norm_rows_is_cpu_normalize_of_the_same_layout(dev, case):
    """F.normalize's summation order follows the layout (tests/test_layout_rules.py): bit-equal, not just close"""
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    ref = F.normalize(v, p=2, dim=-1)
    out = ops.l2norm_rows(vg)
    bad = (out.cpu() != ref).any(-1).sum().item()
    assert bad == 0, f"{bad} of {v.shape[0] * v.shape[1]} rows differ from F.normalize on the CPU"


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_raw_l2norm_order_follows_x_not_out(dev, case):
    """vqseg_l2norm_f32 with an output laid out unlike x (NCHW order and packed rows)"""
    from vq_seg_b200 import _native
    v, vg, e, eg = setup(case, dev)
    L = _native.lib()
    ref = F.normalize(v, p=2, dim=-1)
    b, p, d = vg.shape
    for ostr in ((d * p, 1, p), (p * d, d, 1)):
        out = torch.full((b * p * d,), float("nan"), device=dev).as_strided((b, p, d), ostr)
        _native.check(L.vqseg_l2norm_f32(vg.data_ptr(), b, p, d, *vg.stride(), out.data_ptr(), *ostr,
                                         torch.cuda.current_stream().cuda_stream), "l2norm")
        assert torch.equal(out.cpu(), ref), ostr


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_kmeans_with_injected_init(dev, case):
    import vq_seg_b200 as V
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    n = v.shape[0] * v.shape[1]
    init = torch.randperm(n, generator=torch.Generator().manual_seed(8))[:16]
    m1, b1 = V.kmeans(vg, 16, 3, init_indices=init.to(dev))
    m2, b2 = V.kmeans(vg.contiguous(), 16, 3, init_indices=init.to(dev))
    assert torch.equal(m1, m2) and torch.equal(b1, b2)
    mc, bc = V.kmeans(ops.l2norm_rows(vg), 16, 3, use_cosine_sim=True, init_indices=init.to(dev))
    mo, bo = O.kmeans(O.l2norm(v), 16, 3, use_cosine_sim=True, init_indices=init)
    assert torch.equal(bc[0].cpu(), bo) and torch.equal(mc[0].cpu(), mo)


# ---- segmentation head ---------------------------------------------------------------------------------------------
def map_bwd64(v, e, g, dist, score=None):
    """(gx, gE, gx_bound, gE_bound): the float64 backward of the Euclidean map given its fp32 values (and the fp32
    class scores when `g` is the gradient w.r.t. them): w = g / d, gx = sum_k w (x - e_k), gE = sum_n w (e_k - x).
    The map is an input of the backward: next to a prototype the distance is cancellation noise of the augmented form
    (bit-equal to the exact scorer, checked above), and a reference that recomputed it would measure that noise.
    The bounds are a-priori fp32 error bounds of any summation order, (terms + 2 K + 8) eps times the magnitudes the
    kernels cancel (x sum_k w - sum_k w e_k, e_k sum_n w - sum_n w x, and the score chain's two differences):
    rounding stays far inside them, a wrong element or stride is far outside"""
    d, g = dist.double(), g.double()
    k = d.shape[-1]
    gm = g.abs()
    if score is not None:
        sc = score.double()
        gt = sc * (g - (g * sc).sum(-1, keepdim=True))
        gt_m = sc * (g.abs() + (g * sc).abs().sum(-1, keepdim=True))
        tot = d.sum(-1, keepdim=True)
        g = ((gt * d).sum(-1, keepdim=True) / tot - gt) / tot
        gm = ((gt_m * d).sum(-1, keepdim=True) / tot + gt_m) / tot
    w = torch.where(d == 0, torch.zeros_like(d), g / d)
    wm = torch.where(d == 0, torch.zeros_like(d), gm / d)
    x, ed = v.double(), e.double()
    t = w.unsqueeze(-1) * (x.unsqueeze(2) - ed)                      # (B, P, K, D)
    mag = wm.unsqueeze(-1) * (x.abs().unsqueeze(2) + ed.abs())
    n = x.shape[0] * x.shape[1]
    return (t.sum(2), -t.sum((0, 1)), (3 * k + 8) * EPS * mag.sum(2), (n + 2 * k + 8) * EPS * mag.sum((0, 1)))


@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_seghead_maps_and_gradients(dev, case):
    from test_gpu_seghead_wide import _grad_bar
    from vq_seg_b200 import _native, ops
    v, vg, e, eg = setup(case, dev)
    eg = eg[:K_SEG].contiguous()
    w = eg.clone()
    ops.l2norm_rows_(w)
    xn = ops.l2norm_rows(vg)
    i_ex = ops.assign(vg, eg, None, ops.ALGO_EXACT)[0]
    i_ip = ops.assign(xn, w, None, ops.ALGO_EXACT | ops.METRIC_IP)[0]
    b, p, d = vg.shape
    gout = torch.randn(b, p, K_SEG, generator=torch.Generator().manual_seed(9))
    cos64, cos32 = _grad_bar("cosine", v, w.cpu(), gout)
    L = _native.lib()
    for algo in (ops.SEGHEAD_PIXEL, ops.SEGHEAD_TILED):
        dm, sc, idx, cnt = ops.seghead_score_map(vg, eg, algo)
        packed = ops.seghead_score_map(vg.contiguous(), eg, algo)
        assert all(torch.equal(a, c) for a, c in zip((dm, sc, idx, cnt), packed)), algo
        assert torch.equal(idx, i_ex) and torch.equal(cnt, torch.bincount(i_ex.reshape(-1), minlength=K_SEG)), algo
        dm2, idx2, cnt2 = ops.seghead_map(vg, eg, False, algo)
        assert torch.equal(dm2, dm) and torch.equal(idx2, idx) and torch.equal(cnt2, cnt), algo
        for j in (0, K_SEG // 2, K_SEG - 1):
            _, dj, _ = ops.unpack_keys(ops.assign_keys(vg, eg[j:j + 1].contiguous(), None, 0, ops.ALGO_EXACT), 1)
            assert torch.equal(dm[:, :, j], dj), (algo, j)
        sim, sidx, scnt = ops.seghead_map(xn, w, True, algo)
        packed = ops.seghead_map(xn.contiguous(), w, True, algo)
        assert all(torch.equal(a, c) for a, c in zip((sim, sidx, scnt), packed)), algo
        assert torch.equal(sidx, i_ip), algo
        # the map written in (P*K, K, 1) order by a raw call
        alt = torch.empty(b * p * K_SEG, device=dev)
        ai, ac = torch.empty(b, p, dtype=torch.int64, device=dev), torch.empty(K_SEG, dtype=torch.int64, device=dev)
        _native.check(L.vqseg_seghead_map_f32(vg.data_ptr(), b, p, d, *vg.stride(), eg.data_ptr(), K_SEG, 0,
                                              alt.data_ptr(), p * K_SEG, K_SEG, 1, ai.data_ptr(), ac.data_ptr(), None,
                                              algo, torch.cuda.current_stream().cuda_stream), "seghead_map")
        assert torch.equal(alt.view(b, p, K_SEG), dm) and torch.equal(ai, idx) and torch.equal(ac, cnt), algo
        # Euclidean gradients: the float64 backward evaluated on the same fp32 map and scores, within fp32 error bounds
        for kind, s_ in (("dist", None), ("score", sc)):
            gx, ge = ops.seghead_map_bwd(gout.to(dev), dm, vg, eg, False, s_, algo)
            gx64, ge64, gx_b, ge_b = map_bwd64(v, e[:K_SEG], gout, dm.cpu(), None if s_ is None else s_.cpu())
            for ours, ref64, bound in ((gx, gx64, gx_b), (ge, ge64, ge_b)):
                err = (ours.cpu().double() - ref64).abs()
                assert (err <= bound).all(), (algo, kind, (err / bound).max().item())
        # cosine: against float64 of the whole mathematics, bar max(1e-5, 2 x the CPU fp32 error)
        gx, ge = ops.seghead_map_bwd(gout.to(dev), sim, vg, w, True, None, algo)
        for ours, ref32, ref64 in ((gx, cos32[0], cos64[0]), (ge, cos32[1], cos64[1])):
            bar = max(1e-5, 2 * rel_to_max(ref32, ref64))
            assert rel_to_max(ours.cpu(), ref64) <= bar, (algo, "cosine", rel_to_max(ours.cpu(), ref64), bar)


# ---- modules -------------------------------------------------------------------------------------------------------
MODULE_CASES = [("nhwc", "odd"), ("nchw_ch_slice_odd", "odd"), ("nhwc_batch_step", "odd"), ("cnhw", "odd"),
                ("map_1x1", "px1")]


def module_input(case, dev):
    layout, s = case
    shape, k = layouts.SHAPES[s]
    full, x = layouts.make(layout, shape, 21)
    fg, xg = layouts.make(layout, shape, 21, dev)
    g = torch.Generator().manual_seed(22)
    rows = layouts.bpd(x).reshape(-1, shape[1])
    e = rows[torch.randint(0, rows.shape[0], (k,), generator=g)] + 0.05 * torch.randn(k, shape[1], generator=g)
    return x, xg, e


def nchw_grad(shape, order, seed, dev):
    g = torch.randn(shape, generator=torch.Generator().manual_seed(seed))
    return (g if order == "nchw" else g.contiguous(memory_format=torch.channels_last)).to(dev)


@pytest.mark.parametrize("amp", [False, True], ids=["fp32", "autocast_fp16"])
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("case", MODULE_CASES, ids=layouts.case_id)
def test_vector_quantizer_module(dev, case, distance, train, amp):
    import vq_seg_b200 as V
    x, xg, e = module_input(case, dev)
    b, c, h, wd = x.shape
    k = e.shape[0]
    eu = O.l2norm(e) if distance == "cosine" else e
    ref = O.vq_forward(x, eu, training=train, distance=distance)
    for order in ("nchw", "nhwc"):
        m = V.VectorQuantizer(dim=c, num_embeddings=k, distance=distance).to(dev)   # (renormalising twice is not idempotent)
        m.codebook.embedding.weight.data.copy_(e)
        m.train(train)
        xin = xg.detach().requires_grad_(train)                  # the layout view itself is the leaf
        with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
            q, idx, loss, usage = m(xin)
        assert torch.equal(idx.cpu(), ref["embed_index"]), order
        assert torch.equal(usage.cpu(), ref["code_usage"])
        if distance == "cosine":
            assert torch.equal(m.codebook.embedding.weight.detach().cpu(), eu)
        xv = layouts.bpd(x)
        code = eu[ref["embed_index"].reshape(b, -1)]
        if amp:
            code = code.half().float()
        qv = xv + (code - xv) if train else code
        want = qv.permute(0, 2, 1).reshape(b, c, h, wd)
        assert torch.equal(q.detach().cpu(), want), order
        if not train:
            assert loss.item() == 0.0
            break
        ref_loss = (qv.double() - xv.double()).pow(2).mean().item()
        assert abs(loss.item() - ref_loss) <= 1e-6 * ref_loss
        gq = nchw_grad(q.shape, order, 23, dev)
        ((q * gq).sum() + loss.sum()).backward()
        gref = O.vq_backward(x, want, gq.cpu(), torch.tensor(1.0), 1.0)
        # the oracle rounds coef * (x - q) and then the sum; the kernel rounds once (fma)
        t = (gref - gq.cpu()).abs().double()
        err = (xin.grad.cpu().double() - gref.double()).abs()
        assert (err <= EPS * (gref.double().abs() + t)).all(), order


@pytest.mark.parametrize("variant", ["softmax2d", "sigmoid", "cosine"])
@pytest.mark.parametrize("case", MODULE_CASES, ids=layouts.case_id)
def test_segmentation_head_module(dev, case, variant):
    import vq_seg_b200 as V
    from oracle.seghead_oracle import OracleVQSegmentationHead
    from test_gpu_seghead_wide import _head64
    x, xg, e = module_input(case, dev)
    b, c, h, wd = x.shape
    e = e[:K_SEG].contiguous()
    kw = dict(dim=c, num_embeddings=K_SEG)
    if variant == "sigmoid":
        kw["activation"] = nn.Sigmoid
    if variant == "cosine":
        kw["distance"] = "cosine"
    for order in ("nchw", "nhwc"):
        m = V.VQSegmentationHead(**kw).to(dev)
        o = OracleVQSegmentationHead(**kw)
        m.codebook.embedding.weight.data.copy_(e.to(dev))
        o.embedding.weight.data.copy_(e)
        m.train(); o.train()
        xin = xg.detach().requires_grad_(True)
        xc = x.detach().requires_grad_(True)
        a, r = m(xin), o(xc)
        assert torch.equal(a[2].cpu(), r[2]) and torch.equal(a[0].detach().cpu(), r[0].detach()), order
        assert a[4].item() == r[4].item()
        assert rel_to_max(a[1].detach().cpu(), r[1].detach()) <= 1e-5
        gs = nchw_grad(r[1].shape, order, 24, dev)
        gq = nchw_grad(r[0].shape, order, 25, dev)
        ((a[1] * gs).sum() + (a[0] * gq).sum() + a[3].sum()).backward()
        x64 = x.double().requires_grad_(True)
        w64 = o.embedding.weight.detach().double().requires_grad_(True)
        q64, s64, l64 = _head64(x64, w64, variant, r[2])
        assert abs(a[3].item() - l64.item()) <= 1e-6 * l64.item()
        ((s64 * gs.cpu().double()).sum() + (q64 * gq.cpu().double()).sum() + l64.sum()).backward()
        ((r[1] * gs.cpu()).sum() + (r[0] * gq.cpu()).sum() + r[3].sum()).backward()
        for ours, ref32, ref64 in ((xin.grad, xc.grad, x64.grad), (m.codebook.embedding.weight.grad, o.embedding.weight.grad, w64.grad)):
            bar = max(1e-5, 2 * rel_to_max(ref32, ref64))
            assert rel_to_max(ours.cpu(), ref64) <= bar, (order, rel_to_max(ours.cpu(), ref64), bar)
    m.eval(); o.eval()
    with torch.no_grad():
        a, r = m(xg), o(x)
    assert torch.equal(a[2].cpu(), r[2])
    assert rel_to_max(a[1].cpu(), r[1]) <= 1e-5
