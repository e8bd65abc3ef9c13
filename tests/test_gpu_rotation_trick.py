"""The rotation trick on the B200 (opt-in extension, no reference counterpart): vqseg_rotate_bwd_f32 bit-equal to the
float32 restatement of tests/rotation_oracle.py on every layout path, the VQSEG_MODE_ROTATE forward (quantize = the
code the eval gather writes, the loss mean((c - x)^2)), and VectorQuantizer.rotation_trick end to end: Euclidean and
cosine, with and without autocast, with the EMA update, under CUDA-graph capture and deterministic algorithms."""
import pytest
import torch

import layouts
from rotation_oracle import F32, lam_of, rotate_grad
from test_gpu_layouts import setup

pytestmark = pytest.mark.gpu

CASES = layouts.cases()
WRITABLE_CASES = layouts.cases(layouts.WRITABLE)
AMPS = {"fp32": None, "fp16": torch.float16, "bf16": torch.bfloat16}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


def raw_rotate(g, x, q, gm, scale, gx):
    """vqseg_rotate_bwd_f32 writing gx (any strides)"""
    from vq_seg_b200 import _native
    L = _native.lib()
    b, p, d = x.shape
    gp = (g.data_ptr(), *g.stride()) if g is not None else (None, 0, 0, 0)
    _native.check(L.vqseg_rotate_bwd_f32(*gp, x.data_ptr(), *x.stride(), q.data_ptr(), *q.stride(),
                                         gm.data_ptr() if gm is not None else None, scale, gx.data_ptr(), *gx.stride(),
                                         b, p, d, torch.cuda.current_stream().cuda_stream), "rotate_bwd")
    return gx


def in_layout(values, layout, shape, seed, dev):
    """a (B, P, D) view in `layout` holding `values`"""
    full, xm = layouts.make(layout, shape, seed, dev)
    v = layouts.bpd(xm, full, layout)
    v.copy_(values)
    return v


def placed(values, kind, dev):
    """a (B, P, D) tensor holding `values`, laid out for one kernel path: "nchw" pixel-contiguous (sP == 1), "nhwc"
    packed rows (sD == 1), "strided" neither (sP = 2D, sD = 2: one thread per row)"""
    b, p, d = values.shape
    if kind == "nchw":
        t = torch.empty(b, d, p, device=dev).permute(0, 2, 1)
    elif kind == "nhwc":
        t = torch.empty(b, p, d, device=dev)
    else:
        t = torch.empty(b, p, d, 2, device=dev)[..., 0]
    t.copy_(values)
    return t


def edge_rows(x, c):
    """zero x rows, zero c rows and c = -2x rows at the front of (B, P, D) tensors x, c (in place)"""
    xr, cr = x[0], c[0]
    xr[0:2] = 0
    cr[2:4] = 0
    cr[4:6] = -2 * xr[4:6]


# ---- the kernel ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_rotate_bwd_every_layout(dev, case):
    """x, c and g in the case's layout and in others: bit-equal to the restatement, whatever the path"""
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    layout, s = case
    shape = layouts.SHAPES[s][0]
    idx = ops.assign(vg, eg, None, ops.ALGO_EXACT)[0]
    c = eg[idx]
    gm = torch.tensor([1.7], device=dev)
    scale = 2.0 / vg.numel()
    want = rotate_grad(vg, c, layouts.bpd(layouts.make("nchw", shape, 3, dev)[1]), lam_of(scale, 1.7))
    cl = in_layout(c, layout, shape, 11, dev) if layout != "expand" else c
    for order in ("nchw", "nhwc"):
        g = layouts.bpd(layouts.make("nchw", shape, 3, dev)[1])
        if order == "nhwc":
            g = g.contiguous()
        for q in (c, cl):
            gx = ops.rotate_bwd(g, vg, q, gm, scale)
            assert torch.equal(gx.cpu(), want), (order, q.stride())
        assert torch.equal(ops.rotate_bwd(g, vg.contiguous(), c, gm, scale).cpu(), want), order


@pytest.mark.parametrize("case", WRITABLE_CASES, ids=layouts.case_id)
def test_rotate_bwd_writes_gx_in_any_layout(dev, case):
    v, vg, e, eg = setup(case, dev)
    layout, s = case
    shape = layouts.SHAPES[s][0]
    from vq_seg_b200 import ops
    c = eg[ops.assign(vg, eg, None, ops.ALGO_EXACT)[0]]
    g = layouts.bpd(layouts.make(layout, shape, 4, dev)[1])
    gm = torch.tensor([0.5], device=dev)
    scale = 2.0 / vg.numel()
    full, gxm = layouts.make(layout, shape, 9, dev)
    full.fill_(float("nan"))
    gx = raw_rotate(g, vg, c, gm, scale, layouts.bpd(gxm, full, layout))
    assert torch.equal(gx.cpu(), rotate_grad(vg, c, g, lam_of(scale, 0.5)))
    assert full.isnan().sum().item() == full.numel() - gx.numel(), "wrote outside the view"


@pytest.mark.parametrize("d", [1, 3, 7, 64, 200, 256, 300, 512, 2048])
def test_rotate_bwd_widths(dev, d):
    """the three paths (pixel tiles, 8 lanes per row, a thread per row) at odd P, with the degenerate rows, with g null
    and with coef_dev null; x, c and g laid out alike and mixed"""
    from vq_seg_b200 import ops
    shape = (2, d, 5, 9)
    gen = torch.Generator().manual_seed(d)
    x = layouts.bpd(torch.randn(shape, generator=gen))
    c = (x * 0.7 + 0.5 * torch.randn(x.shape, generator=gen)).contiguous()
    if d > 1:
        edge_rows(x, c)
    g = torch.randn(x.shape, generator=gen)
    scale = 2.0 / x.numel()
    gm = torch.tensor([1.3], device=dev)
    kinds = ("nchw", "nhwc", "strided")
    for xk, ck, gk in [(k, k, k) for k in kinds] + [("nchw", "nhwc", "strided"), ("strided", "nchw", "nhwc")]:
        layout = (xk, ck, gk)
        xg, qg, gg = placed(x, xk, dev), placed(c, ck, dev), placed(g, gk, dev)
        for gi, gmi, lam in ((gg, gm, lam_of(scale, 1.3)), (None, gm, lam_of(scale, 1.3)), (gg, None, F32(0)),
                             (None, None, F32(0))):
            got = ops.rotate_bwd(gi, xg, qg, gmi, scale).cpu()
            want = rotate_grad(x, c, None if gi is None else g, lam)
            assert torch.isfinite(got).all()
            assert torch.equal(got, want), (layout, gi is None, gmi is None)


def test_rotate_bwd_large_map(dev):
    """more than 10^5 rows (pixel tiles over many blocks, a grid-stride loop)"""
    from vq_seg_b200 import ops
    shape = (2, 24, 250, 201)
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(shape, generator=gen)
    c = x * 0.8 + 0.4 * torch.randn(shape, generator=gen)
    g = torch.randn(shape, generator=gen)
    xv, cv, gv = (layouts.bpd(t) for t in (x, c, g))
    assert xv.shape[0] * xv.shape[1] > 10 ** 5
    gm = torch.tensor([1.0], device=dev)
    scale = 2.0 / xv.numel()
    want = rotate_grad(xv, cv, gv, lam_of(scale, 1.0))
    for order in ("nchw", "nhwc"):
        mk = (lambda t: t.to(dev)) if order == "nchw" else (lambda t: t.to(dev).contiguous(memory_format=torch.channels_last))
        got = ops.rotate_bwd(layouts.bpd(mk(g)), layouts.bpd(mk(x)), layouts.bpd(mk(c)), gm, scale)
        assert torch.equal(got.cpu(), want), order


def test_opcheck(dev):
    from vq_seg_b200 import ops
    x = torch.randn(2, 16, 50, device=dev).permute(0, 2, 1)
    e = torch.randn(24, 16, device=dev)
    idx, _ = ops.assign(x, e, None, ops.ALGO_EXACT)
    blob = ops.prepare_codebook(e)
    q = e[idx]
    g = torch.randn_like(q)
    gm = torch.tensor([1.0], device=dev)
    utils = ("test_schema", "test_faketensor")
    torch.library.opcheck(torch.ops.vqseg.rotate_bwd, (g, x, q, gm, 0.01), test_utils=utils)
    torch.library.opcheck(torch.ops.vqseg.rotate_bwd, (None, x, q, None, 0.01), test_utils=utils)
    for base in (ops.MODE_TRAIN, ops.MODE_TRAIN_AMP, ops.MODE_TRAIN_AMP_BF16):
        mode = base | ops.MODE_ROTATE
        torch.library.opcheck(torch.ops.vqseg.gather_ste, (x, e, idx, mode), test_utils=utils)
        torch.library.opcheck(torch.ops.vqseg.vq_forward, (x, e, blob, mode), test_utils=utils)


def test_rotate_flag_needs_a_train_mode(dev):
    """EVAL | ROTATE and unknown bits are refused by both gather entry points"""
    from vq_seg_b200 import _native, ops
    x = torch.randn(1, 40, 8, device=dev)
    e = torch.randn(16, 8, device=dev)
    idx, _ = ops.assign(x, e, None, ops.ALGO_EXACT)
    blob = ops.prepare_codebook(e)
    L = _native.lib()
    q = torch.empty_like(x)
    loss = torch.zeros(1, device=dev)
    nws = L.vqseg_gather_workspace_bytes(40, 8)
    ws = torch.empty(nws, dtype=torch.uint8, device=dev)
    bad = [ops.MODE_ROTATE | m for m in (ops.MODE_EVAL, ops.MODE_EVAL_AMP, ops.MODE_EVAL_AMP_BF16)] + [0x20 | ops.MODE_TRAIN,
                                                                                                       0x30 | ops.MODE_TRAIN]
    for mode in bad:
        rc = L.vqseg_gather_ste_f32(x.data_ptr(), 1, 40, 8, *x.stride(), e.data_ptr(), 16, idx.data_ptr(), q.data_ptr(),
                                    *q.stride(), loss.data_ptr(), mode, ws.data_ptr(), nws,
                                    torch.cuda.current_stream().cuda_stream)
        assert rc == -1, mode
        with pytest.raises(RuntimeError, match="failed \\(-1\\)"):
            ops.vq_forward(x, e, blob, mode)
    torch.cuda.synchronize()


# ---- the forward -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=layouts.case_id)
def test_rotate_forward_every_layout(dev, case):
    """both gather entry points: q = the eval gather's output, indices and usage as without the flag, the loss the mse
    of c against x"""
    from vq_seg_b200 import ops
    v, vg, e, eg = setup(case, dev)
    blob = ops.prepare_codebook(eg)
    for amp in AMPS.values():
        mode = ops.gather_mode(True, amp, True)
        qe, ie, _, ue = ops.vq_forward(vg, eg, blob, ops.gather_mode(False, amp))
        _, i0, _, u0 = ops.vq_forward(vg, eg, blob, ops.gather_mode(True, amp))
        q, idx, loss, usage = ops.vq_forward(vg, eg, blob, mode)
        assert torch.equal(q, qe) and torch.equal(idx, ie) and torch.equal(idx, i0), amp
        assert torch.equal(usage, ue) and torch.equal(usage, u0), amp
        ref = (qe.cpu().double() - v.double()).pow(2).mean().item()
        assert abs(loss.item() - ref) <= 1e-6 * ref, (amp, loss.item(), ref)
        q2, loss2 = ops.gather_ste(vg, eg, idx, mode)
        assert torch.equal(q2, qe), amp
        assert abs(loss2.item() - ref) <= 1e-6 * ref, amp


# ---- the module ------------------------------------------------------------------------------------------------------
def module_input(dev, seed=0, shape=(2, 48, 9, 11), k=40):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=gen)
    rows = layouts.bpd(x).reshape(-1, shape[1])
    e = rows[torch.randint(0, rows.shape[0], (k,), generator=gen)] * 0.9 + 0.3 * torch.randn(k, shape[1], generator=gen)
    gq = torch.randn(shape, generator=gen)
    return x, e, gq


def run_module(dev, x, e, gq, distance, amp, weight, rotate, channels_last=False, ema=False):
    import vq_seg_b200 as V
    m = V.VectorQuantizer(dim=x.shape[1], num_embeddings=e.shape[0], distance=distance, commitment_weight=weight).to(dev)
    m.codebook.embedding.weight.data.copy_(e)
    m.train()
    m.rotation_trick = rotate
    if ema:
        m.enable_ema()
    xin = x.to(dev)
    if channels_last:
        xin = xin.contiguous(memory_format=torch.channels_last)
    xin.requires_grad_(True)
    with torch.autocast("cuda", dtype=amp or torch.float16, enabled=amp is not None):
        q, idx, loss, usage = m(xin)
    ((q * gq.to(dev)).sum() + loss.sum()).backward()
    return m, xin, q.detach(), idx, loss.detach(), usage


@pytest.mark.parametrize("weight", [1, 0.25])
@pytest.mark.parametrize("amp", list(AMPS), ids=list(AMPS))
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_module_training_step(dev, distance, amp, weight):
    from vq_seg_b200 import ops
    x, e, gq = module_input(dev)
    dtype = AMPS[amp]
    for channels_last in (False, True):
        m, xin, q, idx, loss, usage = run_module(dev, x, e, gq, distance, dtype, weight, True, channels_last)
        _, _, q0, idx0, _, usage0 = run_module(dev, x, e, gq, distance, dtype, weight, False, channels_last)
        assert torch.equal(idx, idx0) and torch.equal(usage, usage0)
        w = m.codebook.embedding.weight.detach()
        xv = layouts.bpd(xin.detach())
        b = x.shape[0]
        ce = ops.gather_ste(xv, w, idx.reshape(b, -1), ops.gather_mode(False, dtype))[0]     # the eval gather
        assert torch.equal(layouts.bpd(q), ce)
        assert not torch.equal(q, q0)
        ref = (ce.double() - xv.double()).pow(2).mean().item()
        assert abs(loss.item() / weight - ref) <= 1e-6 * ref
        scale = 2.0 / xv.numel()
        want = rotate_grad(xv, ce, layouts.bpd(gq), lam_of(scale, weight))
        assert torch.equal(layouts.bpd(xin.grad).cpu(), want), channels_last


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_module_with_ema_uses_the_codes_before_the_update(dev, distance):
    """the EMA update rewrites the codebook inside the training forward; the backward reads the saved quantize, i.e.
    the codes before the update (those of the same step without EMA)"""
    x, e, gq = module_input(dev, 4)
    m, xin, q, idx, loss, usage = run_module(dev, x, e, gq, distance, None, 1, True, ema=True)
    m0, _, q0, idx0, _, _ = run_module(dev, x, e, gq, distance, None, 1, True)
    assert torch.equal(idx, idx0) and torch.equal(q, q0)
    assert not torch.equal(m.codebook.embedding.weight, m0.codebook.embedding.weight)     # the update moved the codes
    if distance == "euclidean":
        assert torch.equal(layouts.bpd(q).cpu(), e[idx.cpu().reshape(x.shape[0], -1)])
    xv = layouts.bpd(x)
    want = rotate_grad(xv, layouts.bpd(q0), layouts.bpd(gq), lam_of(2.0 / xv.numel(), 1))
    assert torch.equal(layouts.bpd(xin.grad).cpu(), want)


def test_graphed_training_step_equals_eager(dev):
    import vq_seg_b200 as V
    torch.manual_seed(12)
    m = V.VectorQuantizer(dim=96, num_embeddings=64).to(dev).train()
    m.codebook.embedding.weight.data.normal_()
    m.rotation_trick = True
    x = torch.randn(2, 96, 24, 24, device=dev).requires_grad_(True)
    gy = torch.randn(2, 96, 24, 24, device=dev)
    one = torch.ones(1, device=dev)

    def step(fn):
        q, idx, loss, usage = fn(x)
        torch.autograd.backward((q, loss), (gy, one))
        g = x.grad.clone()
        x.grad = None
        return q.detach().clone(), idx.clone(), loss.detach().clone(), usage.clone(), g

    eager = step(m)
    gm = torch.cuda.make_graphed_callables(m, (x.detach().clone().requires_grad_(True),), allow_unused_input=True)
    for _ in range(2):
        graphed = step(gm)
        for a, b in zip(eager, graphed):
            assert torch.equal(a, b)
    xv = layouts.bpd(x.detach())
    want = rotate_grad(xv, layouts.bpd(eager[0]), layouts.bpd(gy), lam_of(2.0 / xv.numel(), 1.0))
    assert torch.equal(layouts.bpd(eager[4]).cpu(), want)


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_repeatable_and_deterministic(dev, distance):
    x, e, gq = module_input(dev, 7, (4, 256, 16, 16), 128)
    runs = [run_module(dev, x, e, gq, distance, None, 1, True)[1].grad for _ in range(2)]
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        runs.append(run_module(dev, x, e, gq, distance, None, 1, True)[1].grad)
    finally:
        torch.use_deterministic_algorithms(was)
    for r in runs[1:]:
        assert torch.equal(runs[0], r)
