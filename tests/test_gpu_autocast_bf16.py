"""bf16 autocast on the B200: the gathered code is rounded through bf16 like the reference's autocast one-hot matmul
(vq_img.py:169-170; the rule is pinned on the CPU in tests/test_autocast_bf16_rule.py).  Everything here is bit-equal
to that rule: x + (float(bf16(E[idx])) - x) in training, float(bf16(E[idx])) in eval, with the fp32 indices."""
import pytest
import torch

import layouts
from oracle import vq_oracle as O
from test_gpu_layouts import MODULE_CASES, check_loss, module_input, nchw_grad
from test_gpu_layouts import setup as layout_case

pytestmark = pytest.mark.gpu

EPS = torch.finfo(torch.float32).eps
BF16_MODES = ("MODE_TRAIN_AMP_BF16", "MODE_EVAL_AMP_BF16")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


def rounded(code, dtype):
    return code if dtype is None else code.to(dtype).float()


def rule(xv, code, dtype, train):
    """the (B, P, D) output for fp32 x and E[idx] under autocast to `dtype` (None: no autocast)"""
    code = rounded(code, dtype)
    return xv + (code - xv) if train else code


def to_map(v, shape):
    b, c, h, w = shape
    return v.permute(0, 2, 1).reshape(b, c, h, w)


# ---- ops -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", layouts.cases(), ids=layouts.case_id)
def test_gather_ste_and_vq_forward_bf16_modes(dev, case):
    """both entry points (vqseg_gather_ste_f32 and the fused forward's ticket gather) on every layout: q bit-equal to
    the rule, the packed copy gives the same bits, the loss is the mse of the rounded q"""
    from vq_seg_b200 import ops
    v, vg, e, eg = layout_case(case, dev)
    blob = ops.prepare_codebook(eg)
    i_ex = ops.assign(vg, eg, None, ops.ALGO_EXACT)[0]
    for name in BF16_MODES:
        mode = getattr(ops, name)
        train = mode == ops.MODE_TRAIN_AMP_BF16
        want = rule(vg, eg[i_ex], torch.bfloat16, train)
        q, idx, loss, usage = ops.vq_forward(vg, eg, blob, mode)
        qp, idxp, _, _ = ops.vq_forward(vg.contiguous(), eg, blob, mode)
        assert torch.equal(idx, i_ex) and torch.equal(idxp, i_ex), name
        assert torch.equal(q, want) and torch.equal(qp, q), name
        assert torch.equal(usage, ops.vq_forward(vg, eg, blob, ops.MODE_EVAL)[3]), name
        check_loss(loss, q, v, train)
        q2, loss2 = ops.gather_ste(vg, eg, i_ex, mode)
        assert torch.equal(q2, want), name
        check_loss(loss2, q2, v, train)


def raw_gather(xv, e, idx, mode, q):
    """vqseg_gather_ste_f32 writing q (any strides): the pixel-tile kernel when x and q are pixel-contiguous, the
    generic one otherwise"""
    from vq_seg_b200 import _native
    L = _native.lib()
    b, p, d = xv.shape
    loss = torch.zeros(1, device=xv.device)
    nws = L.vqseg_gather_workspace_bytes(b * p, d)
    ws = torch.empty(nws, dtype=torch.uint8, device=xv.device)
    _native.check(L.vqseg_gather_ste_f32(xv.data_ptr(), b, p, d, *xv.stride(), e.data_ptr(), e.shape[0], idx.data_ptr(),
                                         q.data_ptr(), *q.stride(), loss.data_ptr(), mode, ws.data_ptr(), nws,
                                         torch.cuda.current_stream().cuda_stream), "gather_ste")
    return q


def test_bf16_modes_on_special_values(dev):
    """signed zeros, infinities, NaN, fp32 values beyond the bf16 range, subnormals and exact rounding ties go through
    the conversion as torch's .bfloat16() takes them (NaN stays NaN, of either sign), on both gather kernels; the fp16
    modes on the same codes as the behaviour the bf16 modes follow"""
    from vq_seg_b200 import ops
    big = torch.finfo(torch.float32).max
    tie = torch.tensor([0x3F808000, 0x3F818000, -0x407F8000], dtype=torch.int32).view(torch.float32).tolist()
    special = [0.0, -0.0, float("inf"), float("-inf"), float("nan"), big, -big, 3.3961e38, 1e-40, -1e-40,
               70000.0, 6e-8] + tie
    k, d = 4, 40
    g = torch.Generator().manual_seed(3)
    e = torch.randn(k, d, generator=g)
    e[0, :len(special)] = torch.tensor(special)
    e[1, :len(special)] = torch.tensor(special[::-1])
    x = torch.randn(2, d, 6, 10, generator=g)
    x[0, :, 0, 0] = -0.0
    idx = torch.randint(0, k, (2, 60), generator=g)
    idx[0, :8] = torch.tensor([0, 1, 0, 1, 0, 1, 0, 1])
    eg, ig = e.to(dev), idx.to(dev)
    xvc = layouts.bpd(x)
    for layout in ("nchw", "nhwc"):
        xg = x.to(dev) if layout == "nchw" else x.to(dev).contiguous(memory_format=torch.channels_last)
        xv = layouts.bpd(xg)
        for suffix, dtype in (("_BF16", torch.bfloat16), ("", torch.float16)):
            for train in (True, False):
                mode = getattr(ops, ("MODE_TRAIN_AMP" if train else "MODE_EVAL_AMP") + suffix)
                want = rule(xvc, e[idx], dtype, train)
                for q in (ops.gather_ste(xv, eg, ig, mode)[0], raw_gather(xv, eg, ig, mode, layouts.bpd(torch.empty_like(xg)))):
                    torch.testing.assert_close(q.cpu(), want, rtol=0, atol=0, equal_nan=True,
                                               msg=f"{layout} mode {mode}")
                    # the sign of a NaN means nothing: the device writes the positive canonical NaN, torch's
                    # vectorised CPU conversion to bf16 a negative one (0xffff)
                    num = ~want.isnan()
                    assert torch.equal(q.cpu().signbit()[num], want.signbit()[num]), (layout, mode)


def test_opcheck_bf16_modes(dev):
    from vq_seg_b200 import ops
    x = torch.randn(2, 16, 50, device=dev).permute(0, 2, 1)
    e = torch.randn(24, 16, device=dev)
    idx, _ = ops.assign(x, e, None, ops.ALGO_EXACT)
    blob = ops.prepare_codebook(e)
    for mode in (ops.MODE_TRAIN_AMP_BF16, ops.MODE_EVAL_AMP_BF16):
        torch.library.opcheck(torch.ops.vqseg.gather_ste, (x, e, idx, mode), test_utils=("test_schema", "test_faketensor"))
        torch.library.opcheck(torch.ops.vqseg.vq_forward, (x, e, blob, mode), test_utils=("test_schema", "test_faketensor"))


# ---- VectorQuantizer -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("case", [("nchw", "aligned"), ("nchw", "odd")] + MODULE_CASES, ids=layouts.case_id)
def test_vector_quantizer_bf16(dev, case, distance, train):
    """outputs on NCHW, channels-last and the other layouts of tests/layouts.py; in training the input gradient (laid
    out either way) is the straight-through gradient with the mse term on the rounded q"""
    import vq_seg_b200 as V
    x, xg, e = module_input(case, dev)
    b, c, h, wd = x.shape
    k = e.shape[0]
    eu = O.l2norm(e) if distance == "cosine" else e
    ref = O.vq_forward(x, eu, training=train, distance=distance)
    xv = layouts.bpd(x)
    qv = rule(xv, eu[ref["embed_index"].reshape(b, -1)], torch.bfloat16, train)
    want = to_map(qv, x.shape)
    assert not torch.equal(want, ref["quantize"])
    for order in ("nchw", "nhwc"):
        m = V.VectorQuantizer(dim=c, num_embeddings=k, distance=distance).to(dev)
        m.codebook.embedding.weight.data.copy_(e)
        m.train(train)
        xin = xg.detach().requires_grad_(train)                  # the layout view itself is the leaf
        with torch.autocast("cuda", dtype=torch.bfloat16):
            q, idx, loss, usage = m(xin)
        assert q.dtype == torch.float32 and loss.dtype == torch.float32
        assert torch.equal(idx.cpu(), ref["embed_index"]), order
        assert torch.equal(usage.cpu(), ref["code_usage"]), order
        assert torch.equal(q.detach().cpu(), want), order
        if not train:
            assert loss.item() == 0.0
            continue
        ref_loss = (qv.double() - xv.double()).pow(2).mean().item()
        assert abs(loss.item() - ref_loss) <= 1e-6 * ref_loss, order
        gq = nchw_grad(q.shape, order, 23, dev)
        ((q * gq).sum() + loss.sum()).backward()
        gref = O.vq_backward(x, want, gq.cpu(), torch.tensor(1.0), 1.0)
        t = (gref - gq.cpu()).abs().double()                 # the kernel rounds g + coef * (x - q) once (fma)
        err = (xin.grad.cpu().double() - gref.double()).abs()
        assert (err <= EPS * (gref.double().abs() + t)).all(), order


def test_amp_compat_off_and_fp16_unchanged(dev):
    """amp_compat = False keeps exact fp32 codes under bf16 autocast; fp16 autocast still rounds through fp16"""
    import vq_seg_b200 as V
    x, xg, e = module_input(MODULE_CASES[0], dev)
    b, c = x.shape[:2]
    ref = O.vq_forward(x, e, training=True)
    xv = layouts.bpd(x)
    m = V.VectorQuantizer(dim=c, num_embeddings=e.shape[0]).to(dev).train()
    m.codebook.embedding.weight.data.copy_(e)
    for dtype, compat, want_dtype in ((torch.bfloat16, False, None), (torch.float16, True, torch.float16),
                                      (torch.bfloat16, True, torch.bfloat16)):
        m.amp_compat = compat
        with torch.autocast("cuda", dtype=dtype):
            q, idx, _, _ = m(xg)
        want = to_map(rule(xv, e[ref["embed_index"].reshape(b, -1)], want_dtype, True), x.shape)
        assert torch.equal(idx.cpu(), ref["embed_index"]) and torch.equal(q.cpu(), want), (dtype, compat)


def test_cuda_graph_cache_keeps_fp16_and_bf16_apart(dev):
    """enable_cuda_graphs(): fp16, bf16 and no-autocast calls alternating on ONE input buffer each replay their own
    graph and return their own rounding"""
    import vq_seg_b200 as V
    x, xg, e = module_input(MODULE_CASES[0], dev)
    b, c = x.shape[:2]
    ref = O.vq_forward(x, e, training=False)
    code = e[ref["embed_index"].reshape(b, -1)]
    m = V.VectorQuantizer(dim=c, num_embeddings=e.shape[0]).to(dev).eval().enable_cuda_graphs()
    m.codebook.embedding.weight.data.copy_(e)
    seq = (torch.float16, torch.bfloat16, None, torch.bfloat16, torch.float16, None, torch.bfloat16)
    with torch.no_grad():
        for dtype in seq:
            with torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
                q, idx, _, _ = m(xg)
            assert torch.equal(idx.cpu(), ref["embed_index"]), dtype
            assert torch.equal(q.cpu(), to_map(rounded(code, dtype), x.shape)), dtype
    assert len(m._graphs) == 3


def test_graphed_training_step_bf16_equals_eager(dev):
    """torch.cuda.make_graphed_callables under bf16 autocast: outputs and the input gradient bit-equal to eager, and
    eager is the bf16 rule"""
    import vq_seg_b200 as V
    torch.manual_seed(12)
    m = V.VectorQuantizer(dim=96, num_embeddings=64).to(dev).train()
    m.codebook.embedding.weight.data.normal_()
    x = torch.randn(2, 96, 24, 24, device=dev).requires_grad_(True)
    gy = torch.randn(2, 96, 24, 24, device=dev)
    one = torch.ones(1, device=dev)

    def step(fn):
        q, idx, loss, usage = fn(x)
        torch.autograd.backward((q, loss), (gy, one))
        g = x.grad.clone()
        x.grad = None
        return q.detach().clone(), idx.clone(), loss.detach().clone(), usage.clone(), g

    # autocast's weight cache must be off while graphs are captured and replayed (make_graphed_callables' contract)
    with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
        eager = step(m)
        gm = torch.cuda.make_graphed_callables(m, (x.detach().clone().requires_grad_(True),), allow_unused_input=True)
        for _ in range(2):
            graphed = step(gm)
            for a, b in zip(eager, graphed):
                assert torch.equal(a, b)
    e = m.codebook.embedding.weight.detach()
    xv = layouts.bpd(x.detach())
    want = to_map(rule(xv, e[eager[1].reshape(2, -1)], torch.bfloat16, True), x.shape)
    assert torch.equal(eager[0], want)
    with torch.no_grad():
        _, idx32, _, _ = m(x)
    assert torch.equal(eager[1], idx32)


# ---- VQSegmentationHead --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("variant", ["softmax2d", "cosine"])
def test_segmentation_head_quantize_bf16(dev, variant, train):
    """the fused Euclidean + Softmax2d path and the cosine path: quantize is the bf16 rule, indices and scores are
    those of the same head without autocast"""
    import vq_seg_b200 as V
    x, xg, e = module_input(MODULE_CASES[0], dev)
    b, c, h, wd = x.shape
    k = 27
    e = e[:k].contiguous()
    kw = dict(dim=c, num_embeddings=k, **({"distance": "cosine"} if variant == "cosine" else {}))
    outs = {}
    for dtype in (None, torch.bfloat16):
        m = V.VQSegmentationHead(**kw).to(dev).train(train)   # a fresh head each: the cosine one renormalises in place
        m.codebook.embedding.weight.data.copy_(e)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=dtype is not None):
            outs[dtype] = [t.detach() for t in m(xg)] + [m.codebook.embedding.weight.detach().clone()]
    (q32, s32, i32, _, u32, w32), (q, s, idx, loss, u, w) = outs[None], outs[torch.bfloat16]
    assert torch.equal(idx, i32) and torch.equal(s, s32) and torch.equal(u, u32) and torch.equal(w, w32)
    xv = layouts.bpd(x)
    qv = rule(xv, w.cpu()[idx.cpu().reshape(b, -1)], torch.bfloat16, train)
    assert q.dtype == torch.float32 and torch.equal(q.cpu(), to_map(qv, x.shape))
    assert not torch.equal(q, q32)
    if train:
        ref_loss = (qv.double() - xv.double()).pow(2).mean().item()
        assert abs(loss.item() - ref_loss) <= 1e-6 * ref_loss
    else:
        assert loss.item() == 0.0
