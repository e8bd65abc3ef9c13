"""ResidualVectorQuantizer on the B200 (opt-in extension, no reference counterpart): Q = 1 bit-equal to VectorQuantizer,
Q > 1 against the CPU restatement of tests/rvq_oracle.py on shapes that send the stage lookups through every filter and
the exact scorer, train / eval / decode agreement, a chain of VectorQuantizer modules, every input layout, the k-means
init and the EMA update per layer, CUDA graphs, deterministic algorithms and edge cases."""
import pytest
import torch

import layouts
import rvq_oracle as R
from ema_expire_oracle import ema_expire
from oracle import vq_oracle as O

pytestmark = pytest.mark.gpu

AMPS = {"fp32": None, "fp16": torch.float16, "bf16": torch.bfloat16}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from vq_seg_b200 import _native
    _native.lib()
    return torch.device("cuda:0")


def codebooks(x, k, q, seed):
    """Q codebooks: layer 0 near rows of x, later layers at halving scales (what the residuals shrink to)"""
    g = torch.Generator().manual_seed(seed)
    b, c = x.shape[:2]
    rows = x.reshape(b, c, -1).permute(0, 2, 1).reshape(-1, c)
    e0 = rows[torch.randint(0, rows.shape[0], (k,), generator=g)] + 0.05 * torch.randn(k, c, generator=g)
    return [e0] + [torch.randn(k, c, generator=g) * 0.5 ** l for l in range(1, q)]


def module(cbs, dev, distance="euclidean", w=1.0, algo=None, **kw):
    import vq_seg_b200 as V
    k, d = cbs[0].shape
    m = V.ResidualVectorQuantizer(d, k, len(cbs), distance=distance, commitment_weight=w, **kw).to(dev)
    for layer, e in zip(m.layers, cbs):
        layer.codebook.embedding.weight.data.copy_(e)
        if algo is not None:
            layer.codebook.algo = algo
    return m


def flat_idx(ei):
    """(B, H, W, Q) -> (Q, B, P)"""
    b, h, w, q = ei.shape
    return ei.permute(3, 0, 1, 2).reshape(q, b, h * w)


def run_train(m, x, g, gl):
    """training forward + backward of (quantize * g).sum() + loss * gl: (outputs on the CPU, gx)"""
    xg = x.detach().requires_grad_(True)                  # (a leaf with x's strides)
    q, ei, loss, usage = m(xg)
    torch.autograd.backward((q, loss), (g, torch.full_like(loss, gl)))
    return [t.detach().cpu() for t in (q, ei, loss, usage)], xg.grad.cpu()


# ---- 1. Q = 1 is VectorQuantizer ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("amp", list(AMPS))
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("training", [True, False])
def test_q1_bit_equal_to_vector_quantizer(dev, amp, distance, training):
    import vq_seg_b200 as V
    x = torch.randn(2, 64, 16, 16, generator=torch.Generator().manual_seed(1))
    cbs = codebooks(x, 128, 1, 2)
    w = 0.7
    m = module(cbs, dev, distance, w).train(training)
    v = V.VectorQuantizer(64, 128, distance=distance, commitment_weight=w).to(dev).train(training)
    v.codebook.embedding.weight.data.copy_(cbs[0])
    xd = x.to(dev)
    g = torch.randn(xd.shape, generator=torch.Generator().manual_seed(3)).to(dev)
    ctx = torch.autocast("cuda", dtype=AMPS[amp]) if AMPS[amp] else torch.autocast("cuda", enabled=False)
    outs = []
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)          # the eval codebook gradient in its ordered form (no fp32 atomics)
    for mod in (m, v):
        with ctx:
            if training:
                xg = xd.clone().requires_grad_(True)
                q, ei, loss, usage = mod(xg)
                torch.autograd.backward((q, loss), (g, torch.full_like(loss, 1.3)))
                grad = xg.grad
            else:
                wt = (mod.layers[0] if mod is m else mod).codebook.embedding.weight
                q, ei, loss, usage = mod(xd)
                q.backward(g)
                grad = wt.grad
        outs.append([q.detach(), ei.reshape(2, 16, 16), loss.detach(), usage, grad])
        assert loss.requires_grad == training
    torch.use_deterministic_algorithms(was)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# ---- 2. Q > 1 against the restatement ------------------------------------------------------------------------------------
SHAPES = {
    "c2": ((8, 256, 64, 64), 512, (3,)),            # the config-2 map: the codebook-resident TMA filter
    "k1024": ((2, 512, 32, 32), 1024, (2,)),        # K = 1024 at D = 512: a streamed codebook
    "splitd": ((2, 2048, 16, 16), 512, (2,)),       # few rows, many dims: the split-D filter
    "odd": ((3, 96, 7, 9), 300, (2, 3, 8)),         # P = 63: not TMA-loadable
    "small": ((2, 64, 16, 16), 128, (2, 3, 8)),
}
CASES = [(s, q) for s, (_, _, qs) in SHAPES.items() for q in qs] + [("exact", 3)]


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-q{c[1]}")
def test_against_oracle(dev, case, distance):
    from vq_seg_b200 import ops
    name, nq = case
    shape, k, _ = SHAPES["odd" if name == "exact" else name]
    x = torch.randn(shape, generator=torch.Generator().manual_seed(nq))
    cbs = codebooks(x, k, nq, 5)
    algo = ops.ALGO_EXACT if name == "exact" else None
    w, gl = 0.8, 1.3
    g = torch.randn(shape, generator=torch.Generator().manual_seed(9))
    # eval
    with torch.no_grad():
        q, ei, loss, usage = module(cbs, dev, distance, w, algo).eval()(x.to(dev))
    want = R.rvq_forward(x, cbs, False, w, distance)
    assert torch.equal(flat_idx(ei).cpu(), want["idx"])
    assert torch.equal(q.cpu(), want["quantize"])
    assert torch.equal(usage.cpu(), want["usage"]) and float(loss) == 0.0
    # training: outputs and gx
    (q, ei, loss, usage), gx = run_train(module(cbs, dev, distance, w, algo).train(), x.to(dev), g.to(dev), gl)
    want = R.rvq_forward(x, cbs, True, w, distance)
    assert torch.equal(flat_idx(ei), want["idx"])
    assert torch.equal(q, want["quantize"])
    assert torch.equal(usage, want["usage"])
    torch.testing.assert_close(loss, want["loss"], rtol=1e-5, atol=0)
    gq = g.reshape(shape[0], shape[1], -1).permute(0, 2, 1)
    wgx = R.rvq_backward(want["A"], gq, torch.tensor([gl]), w)
    assert torch.equal(gx.reshape(shape[0], shape[1], -1).permute(0, 2, 1), wgx)
    # the per-layer statistics
    m = module(cbs, dev, distance, w, algo).train()
    with torch.no_grad():
        _, _, lloss, lusage = m(x.to(dev), return_layer_stats=True)
    assert torch.equal(lusage.cpu(), want["layer_usage"])
    torch.testing.assert_close(lloss.cpu(), want["layer_mse"] * w, rtol=1e-5, atol=0)


# ---- 3. train / eval / decode ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("amp", list(AMPS))
def test_train_eval_decode_agree(dev, amp):
    x = torch.randn(2, 96, 12, 12, generator=torch.Generator().manual_seed(4)).to(dev)
    cbs = codebooks(x.cpu(), 200, 4, 6)
    m = module(cbs, dev)
    ctx = torch.autocast("cuda", dtype=AMPS[amp]) if AMPS[amp] else torch.autocast("cuda", enabled=False)
    with ctx, torch.no_grad():
        qe, ie, _, _ = m.eval()(x)
        dec = m.get_output_from_indices(ie)
        qt, it, _, _ = m.train()(x)
    assert torch.equal(ie, it)
    assert torch.equal(dec, qe)
    assert torch.equal(qt, x + (qe - x))


# ---- 4. a chain of VectorQuantizer modules ----------------------------------------------------------------------------------
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_eval_equals_a_chain_of_vector_quantizers(dev, distance):
    import vq_seg_b200 as V
    x = torch.randn(4, 128, 16, 16, generator=torch.Generator().manual_seed(7)).to(dev)
    cbs = codebooks(x.cpu(), 256, 3, 8)
    m = module(cbs, dev, distance).eval()
    chain = []
    for e in cbs:
        v = V.VectorQuantizer(128, 256, distance=distance).to(dev).eval()
        v.codebook.embedding.weight.data.copy_(e)
        chain.append(v)
    with torch.no_grad():
        q, ei, _, _ = m(x)
        r, s, idxs = x, None, []
        for v in chain:
            ql, il, _, _ = v(r)
            s = ql if s is None else s + ql
            r = r - ql
            idxs.append(il)
    assert torch.equal(ei, torch.stack(idxs, -1))
    assert torch.equal(q, s)


# ---- 5. layouts -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", layouts.cases(shapes=("odd", "aligned", "px1")), ids=layouts.case_id)
def test_every_layout_equals_the_packed_copy(dev, case):
    layout, s = case
    shape, k = layouts.SHAPES[s]
    full, x = layouts.make(layout, shape, 3, dev)
    cbs = codebooks(x.cpu().contiguous(), k, 3, 4)
    g = torch.randn(shape, generator=torch.Generator().manual_seed(2)).to(dev)
    res = []
    for inp in (x, x.contiguous()):
        with torch.no_grad():
            qe, ie, _, ue = module(cbs, dev).eval()(inp)
        (qt, it, lt, ut), gx = run_train(module(cbs, dev, w=0.5).train(), inp, g, 1.0)
        res.append((qe.cpu(), ie.cpu(), ue.cpu(), qt, it, ut, gx, lt))
    for a, b in zip(res[0][:-1], res[1][:-1]):
        assert torch.equal(a, b)
    torch.testing.assert_close(res[0][-1], res[1][-1], rtol=1e-6, atol=0)


# ---- 6. k-means init and EMA per layer ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_kmeans_init_per_layer(dev, distance):
    nq, k, iters = 3, 64, 4
    cosine = distance == "cosine"
    x = torch.randn(2, 32, 16, 16, generator=torch.Generator().manual_seed(12))
    import vq_seg_b200 as V
    m = V.ResidualVectorQuantizer(32, k, nq, kmeans_init=True, kmeans_iters=iters, distance=distance).to(dev).train()
    gen = torch.Generator().manual_seed(13)
    ids = [O.sample_indices(512, k, gen) for _ in range(nq)]
    for layer, i in zip(m.layers, ids):
        layer.codebook.kmeans_init_indices = i.to(dev)
    with torch.no_grad():
        m(x.to(dev))
    xv = x.reshape(2, 32, -1).permute(0, 2, 1)
    r, means = xv, []
    for l in range(nq):
        src = O.l2norm(r) if cosine else r
        e, _ = O.kmeans(src, k, iters, use_cosine_sim=cosine, init_indices=ids[l])
        e = O.l2norm(e) if cosine else e                   # the lookup renormalises the weights in place
        means.append(e)
        idx = O.assign_cosine(r, e) if cosine else O.assign_euclidean(r, e)
        r = R.nchw(r - e[idx])
    for layer, e in zip(m.layers, means):
        assert layer.codebook.initted
        assert torch.equal(layer.codebook.embedding.weight.detach().cpu(), e)


@pytest.mark.parametrize("distance", ["euclidean", "cosine"])
def test_ema_with_expiry_per_layer(dev, distance):
    nq, k, d, decay, thr = 3, 128, 32, 0.8, 1.0
    cosine = distance == "cosine"
    x = torch.randn(2, d, 16, 16, generator=torch.Generator().manual_seed(21))
    m = module(codebooks(x, k, nq, 22), dev, distance, decay=decay).train()
    m.enable_ema(deterministic=True, threshold_ema_dead_code=thr)
    n = 2 * 256
    for step in range(3):
        gen = torch.Generator().manual_seed(100 + step)
        ids = [O.sample_indices(n, k, gen) for _ in range(nq)]
        before = []
        for layer, i in zip(m.layers, ids):
            cb = layer.codebook
            cb.expire_indices = i.to(dev)
            before.append((cb.embedding.weight.detach().cpu().clone(), cb.cluster_size.cpu().clone(),
                           cb.embed_avg.cpu().clone()))
        with torch.no_grad():
            _, ei, _, _ = m(x.to(dev))
        want = R.rvq_forward(x, [b[0] for b in before], True, 1.0, distance)
        assert torch.equal(flat_idx(ei).cpu(), want["idx"])
        for l, (layer, (w0, cs0, ea0)) in enumerate(zip(m.layers, before)):
            cb = layer.codebook
            src = want["residuals"][l]
            src = (O.l2norm(src) if cosine else src).reshape(-1, d)
            flat = want["idx"][l].reshape(-1)
            counts = torch.bincount(flat, minlength=k)
            sums = torch.zeros(k, d).index_add_(0, flat, src)
            cs1, ea1, w1 = O.ema_update(counts, sums, cs0, ea0, torch.tensor(decay), 1e-5)
            want_cs, want_ea, want_w, _ = ema_expire(cs1, ea1, w1, src[ids[l]], thr)
            assert torch.equal(cb.cluster_size.cpu(), want_cs), (step, l)
            assert torch.allclose(cb.embedding.weight.detach().cpu(), want_w, rtol=1e-4, atol=1e-5), (step, l)
            assert torch.allclose(cb.embed_avg.cpu(), want_ea, rtol=1e-4, atol=1e-5), (step, l)


# ---- 7. graphs and determinism --------------------------------------------------------------------------------------------------
def test_graph_replay_equals_eager(dev):
    x = torch.randn(2, 96, 16, 16, generator=torch.Generator().manual_seed(31)).to(dev)
    cbs = codebooks(x.cpu(), 200, 3, 32)
    eager, graphed = module(cbs, dev).eval(), module(cbs, dev).eval().enable_cuda_graphs()
    with torch.no_grad():
        for step in range(3):
            a, b = eager(x), graphed(x)
            for u, v in zip(a, b):
                assert torch.equal(u, v), step
            for m in (eager, graphed):                      # the graph follows weight updates
                m.layers[1].codebook.embedding.weight.data.mul_(0.7)
        assert len(graphed._graphs) == 1


def test_make_graphed_callables_training(dev):
    x = torch.randn(2, 96, 24, 24, generator=torch.Generator().manual_seed(41)).to(dev).requires_grad_(True)
    cbs = codebooks(x.detach().cpu(), 64, 3, 42)
    m = module(cbs, dev, w=0.6).train()
    gy = torch.randn(x.shape, generator=torch.Generator().manual_seed(43)).to(dev)
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
        for a, b in zip(eager, step(gm)):
            assert torch.equal(a, b)
    m.layers[0].codebook.embedding.weight.data.mul_(0.5)
    e2, g2 = step(m), step(gm)
    assert not torch.equal(e2[0], eager[0])
    for a, b in zip(e2, g2):
        assert torch.equal(a, b)


def test_deterministic_runs_are_identical(dev):
    x = torch.randn(2, 64, 16, 16, generator=torch.Generator().manual_seed(51)).to(dev)
    cbs = codebooks(x.cpu(), 128, 3, 52)
    g = torch.randn(x.shape, generator=torch.Generator().manual_seed(53)).to(dev)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        runs = []
        for _ in range(2):
            outs, gx = run_train(module(cbs, dev).train(), x, g, 1.0)
            m = module(cbs, dev).eval()
            m(x)[0].backward(g)
            runs.append(outs + [gx] + [layer.codebook.embedding.weight.grad.cpu() for layer in m.layers])
        for a, b in zip(*runs):
            assert torch.equal(a, b)
    finally:
        torch.use_deterministic_algorithms(was)


# ---- 8. edge cases ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1, 64, 8, 8), (6, 64, 1, 1), (0, 64, 4, 4)], ids=["b1", "map1x1", "empty"])
@pytest.mark.parametrize("training", [True, False])
def test_edge_shapes_like_vector_quantizer(dev, shape, training):
    import vq_seg_b200 as V
    x = torch.randn(shape, generator=torch.Generator().manual_seed(61)).to(dev)
    cbs = codebooks(torch.randn(2, 64, 4, 4), 32, 1, 62)
    v = V.VectorQuantizer(64, 32).to(dev).train(training)
    v.codebook.embedding.weight.data.copy_(cbs[0])
    outs = []
    for mod in (module(cbs, dev).train(training), v):
        xg = x.clone().requires_grad_(training)
        q, ei, loss, usage = mod(xg)
        if training and shape[0]:
            torch.autograd.backward((q, loss), (torch.ones_like(q), torch.ones_like(loss)))
        outs.append([q.detach(), ei.reshape(shape[0], shape[2], shape[3]), loss.detach(), usage] +
                    ([xg.grad] if training and shape[0] else []))
    for a, b in zip(*outs):
        assert a.shape == b.shape and torch.equal(a, b)
    m3 = module(codebooks(torch.randn(2, 64, 4, 4), 32, 3, 63), dev).train(training)
    q, ei, loss, usage = m3(x)
    assert q.shape == x.shape and ei.shape == (shape[0], shape[2], shape[3], 3)
    if shape[0] == 0:
        assert float(usage) == 100.0 and float(loss) == 0.0
