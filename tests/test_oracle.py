"""Pins the restated CPU oracle: (1) against the committed golden vectors produced by the live
reference, (2) against the live reference itself when VQSEG_REF names a checkout of it."""
import pytest
import torch

import cases
from oracle import vq_oracle as O


@pytest.fixture
def golden_threads(golden, golden_seghead):
    """ATen splits a float reduction (the mse loss, softmax's sum, ...) over its intra-op threads, so the last bits of
    a CPU result depend on the thread count: the oracle runs with the count the goldens were recorded with."""
    threads = {golden["meta"]["threads"], golden_seghead["meta"]["threads"]}
    assert len(threads) == 1
    n = torch.get_num_threads()
    torch.set_num_threads(threads.pop())
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", list(cases.FORWARD_CASES))
def test_oracle_matches_golden_forward(golden, golden_threads, name):
    rec = golden["forward"][name]
    x, e = cases.FORWARD_CASES[name]()
    assert cases.sha(x) == rec["x_sha"] and cases.sha(e) == rec["e_sha"], "seeded inputs drifted"
    ev = O.vq_forward(x, e, training=False)
    assert torch.equal(ev["embed_index"].to(torch.int32), rec["idx"])       # bit-exact indices
    assert torch.equal(ev["counts"], rec["counts"])                         # bit-exact code counts
    assert torch.equal(ev["code_usage"], rec["usage"])
    assert cases.sha(ev["quantize"]) == rec["q_eval_sha"]
    assert torch.equal(ev["loss"], rec["loss_eval"]) and ev["loss"].shape == (1,)
    tr = O.vq_forward(x, e, training=True, commitment_weight=1)
    assert cases.sha(tr["quantize"]) == rec["q_train_sha"]
    assert torch.equal(tr["loss"], rec["loss_train"])
    gx = O.vq_backward(x, tr["quantize"], None, torch.tensor(1.5), 1)
    step = max(1, gx.numel() // 4096)
    torch.testing.assert_close(gx.reshape(-1)[::step], rec["gx_l_sample"], rtol=1e-6, atol=1e-12)
    assert rec["gx_q_is_gq"]


@pytest.mark.parametrize("name", cases.KMEANS_CASES)
def test_oracle_matches_golden_kmeans(golden, golden_threads, name):
    rec = golden["kmeans"][name]
    x, k, iters, init_idx, use_cos = cases.kmeans_case(name)
    assert cases.sha(x) == rec["x_sha"]
    b, c, h, w = x.shape
    flat = x.reshape(b, c, h * w).permute(0, 2, 1)
    if use_cos:
        flat = O.l2norm(flat)
    means, bins = O.kmeans(flat, k, iters, use_cosine_sim=use_cos, init_indices=init_idx)
    assert torch.equal(bins, rec["bins"])
    assert torch.equal(means, rec["means"])


def test_euclidean_dist_restatement_is_cdist():
    g = torch.Generator().manual_seed(3)
    for (n, k, d) in [(300, 77, 48), (4096, 512, 256), (16, 20, 16), (26, 3, 8), (2, 600, 1024), (25, 25, 8), (25, 26, 8), (1000, 512, 2048), (777, 130, 512)]:
        x = torch.randn(2, n, d, generator=g)
        e = torch.randn(k, d, generator=g)
        assert torch.equal(O.euclidean_dist(x, e), torch.cdist(x, e, p=2)), (n, k, d)


def test_live_reference_forward_backward(ref_vq):
    if ref_vq is None:
        pytest.skip("no reference checkout (VQSEG_REF): golden vectors are the pin")
    torch.manual_seed(5)
    for (b, c, h, w, k, wgt) in [(2, 64, 16, 16, 128, 1), (1, 256, 8, 8, 512, 0.25), (2, 512, 12, 12, 64, 0)]:
        ref = ref_vq.VectorQuantizer(dim=c, num_embeddings=k, commitment_weight=wgt)
        ref.codebook.embedding.weight.data.normal_()
        port = O.OracleVectorQuantizer(dim=c, num_embeddings=k, commitment_weight=wgt)
        port.load_state_dict(ref.state_dict())                      # same state_dict keys
        for training in (True, False):
            ref.train(training); port.train(training)
            x1 = torch.randn(b, c, h, w, requires_grad=True)
            x2 = x1.detach().clone().requires_grad_(True)
            r = ref(x1); p = port(x2)
            for a, bb in zip(r, p):
                assert torch.equal(a, bb)
            assert r[2].requires_grad == p[2].requires_grad == training
            if training:
                gq = torch.randn_like(r[0])
                ((r[0] * gq).sum() + 2 * r[2].sum()).backward()
                ((p[0] * gq).sum() + 2 * p[2].sum()).backward()
                assert torch.equal(x1.grad, x2.grad)
                assert ref.codebook.embedding.weight.grad is None
                assert port.codebook.embedding.weight.grad is None
                torch.testing.assert_close(
                    x1.grad, O.vq_backward(x1.detach(), r[0].detach(), gq, torch.tensor(2.0), wgt),
                    rtol=1e-6, atol=1e-9)


def test_live_reference_kmeans_same_rng(ref_vq):
    if ref_vq is None:
        pytest.skip("no reference checkout (VQSEG_REF)")
    x = torch.relu(torch.randn(2, 200, 32))
    torch.manual_seed(11); m1, b1 = ref_vq.kmeans(x, 16, 5)
    torch.manual_seed(11); m2, b2 = O.kmeans(x, 16, 5)
    assert torch.equal(m1[0], m2) and torch.equal(b1[0], b2)


def test_live_reference_kmeans_init_module(ref_vq):
    if ref_vq is None:
        pytest.skip("no reference checkout (VQSEG_REF)")
    ref = ref_vq.VectorQuantizer(dim=32, num_embeddings=20, kmeans_init=True)
    port = O.OracleVectorQuantizer(dim=32, num_embeddings=20, kmeans_init=True)
    x = torch.relu(torch.randn(2, 32, 12, 12))
    ref.train(); port.train()
    torch.manual_seed(21); r = ref(x)
    torch.manual_seed(21); p = port(x)
    for a, bb in zip(r, p):
        assert torch.equal(a, bb)
    assert torch.equal(ref.codebook.embedding.weight, port.codebook.embedding.weight)
    assert ref.codebook.initted and port.codebook.initted


def test_live_reference_cosine(golden, golden_threads):
    for name, build in cases.COSINE_CASES.items():
        x, e = build()
        port = O.OracleVectorQuantizer(dim=x.shape[1], num_embeddings=e.shape[0], distance="cosine")
        port.codebook.embedding.weight.data.copy_(e)
        port.train()
        q, idx, loss, usage = port(x)
        rec = golden["cosine"][name]
        assert torch.equal(idx.to(torch.int32), rec["idx"])
        assert cases.sha(q) == rec["q_train_sha"]
        assert torch.equal(loss.detach(), rec["loss_train"])
        assert cases.sha(port.codebook.embedding.weight.data) == rec["weight_after_sha"]


def test_make_vq_module_port():
    ml = O.oracle_make_vq_module({"num_embeddings": [0, 0, 8, 8, 8], "distance": "euclidean", "kmeans_init": True},
                                 [3, 64, 256, 512, 1024, 2048], 5)
    assert [type(m).__name__ for m in ml] == ["OracleIdentity"] * 2 + ["OracleVectorQuantizer"] * 3
    assert ml[2].codebook.embedding.weight.shape == (8, 512)
    with pytest.raises(ValueError):
        O.oracle_make_vq_module({"num_embeddings": [-1]}, [3, 64], 1)
    with pytest.raises(TypeError):
        O.oracle_make_vq_module({"num_embeddings": 1.5}, [3, 64], 1)


@pytest.mark.parametrize("name", list(cases.SEGHEAD_CASES))
def test_seghead_oracle_matches_golden(golden_seghead, golden_threads, name):
    """The restated segmentation head (oracle/seghead_oracle.py) against the live reference's outputs and
    gradients: same torch build -> bit-equal."""
    from oracle.seghead_oracle import OracleVQSegmentationHead
    build, distance = cases.SEGHEAD_CASES[name]
    x, e = build()
    rec = golden_seghead["seghead"][name]
    assert cases.sha(x) == rec["x_sha"] and cases.sha(e) == rec["e_sha"]
    m = OracleVQSegmentationHead(dim=x.shape[1], num_embeddings=e.shape[0], distance=distance)
    m.embedding.weight.data.copy_(e)
    m.train()
    xg = x.clone().requires_grad_(True)
    quantize, score, idx, loss, usage = m(xg)
    g = torch.Generator().manual_seed(4242)
    gs = torch.randn(score.shape, generator=g)
    gq = torch.randn(quantize.shape, generator=g)
    ((score * gs).sum() + (quantize * gq).sum() + 1.5 * loss.sum()).backward()
    assert torch.equal(idx.to(torch.int32), rec["idx"])
    assert torch.equal(quantize.detach(), rec["quantize"]) and torch.equal(score.detach(), rec["score"])
    assert torch.equal(loss.detach(), rec["loss"]) and torch.equal(usage, rec["usage"])
    assert torch.equal(xg.grad, rec["gx"]) and torch.equal(m.embedding.weight.grad, rec["gw"])
    assert torch.isfinite(rec["gx"]).all() and torch.isfinite(rec["gw"]).all()
    m.eval()
    with torch.no_grad():
        q2, s2, i2, l2, u2 = m(x)
    assert torch.equal(q2, rec["quantize_eval"]) and torch.equal(s2, rec["score_eval"]) and l2.item() == 0.0


def test_live_reference_seghead_kmeans_init():
    """First training forward with kmeans_init=True: the oracle and the live reference draw the same start rows
    from the same RNG state and must agree bit for bit afterwards."""
    from oracle.ref_loader import load_reference_seghead
    from oracle.seghead_oracle import OracleVQSegmentationHead
    R = load_reference_seghead()
    if R is None:
        pytest.skip("no reference checkout (VQSEG_REF): golden vectors are the pin")
    x, _ = cases.SEGHEAD_CASES["sh_c3_d32"][0]()
    for distance in ("euclidean", "cosine"):
        torch.manual_seed(5)
        ref = R.VQSegmentationHead(dim=32, num_embeddings=3, kmeans_init=True, kmeans_iters=4, distance=distance)
        torch.manual_seed(5)
        ora = OracleVQSegmentationHead(dim=32, num_embeddings=3, kmeans_init=True, kmeans_iters=4, distance=distance)
        ora.embedding.weight.data.copy_(ref.codebook.embedding.weight.data)
        torch.manual_seed(6); ref.train(); a = ref(x)
        torch.manual_seed(6); ora.train(); b = ora(x)
        assert torch.equal(ref.codebook.embedding.weight, ora.embedding.weight)
        for u, v in zip(a, b):
            assert torch.equal(u, v)


def test_cpu_sqrt_is_not_correctly_rounded():
    """DESIGN.md 2.4: ATen's CPU sqrt (MKL VML in this build) is 1 ulp off on a fraction of a percent of inputs, so
    distances can only be pinned to 1 ulp; the kernels use the IEEE sqrt."""
    g = torch.Generator().manual_seed(0)
    c = torch.rand(200_000, generator=g) * 60 + 1
    exact = c.double().sqrt().float()
    live = c.sqrt()
    frac = (live != exact).float().mean().item()
    assert frac < 0.02                                             # a correctly rounded build gives 0: also fine
    assert ((live - exact).abs() <= torch.finfo(torch.float32).eps * exact).all()


def test_single_image_batch_takes_the_strided_norm_order():
    """DESIGN.md 2.4: with B == 1 cdist works on the permuted NCHW view itself and sums |x|^2 over the strided dim in
    another order than for B >= 2 (where it copies first).  The oracle and the kernels use the B >= 2 arithmetic for
    every B: distances within a few ulp, same indices on these inputs."""
    g = torch.Generator().manual_seed(1)
    for (b, c, h, w, k) in [(1, 256, 32, 32, 512), (1, 64, 16, 16, 100), (2, 40, 9, 9, 33)]:
        x = torch.randn(b, c, h, w, generator=g)
        e = torch.randn(k, c, generator=g)
        xv = x.reshape(b, c, h * w).permute(0, 2, 1)
        live = torch.cdist(xv, e, p=2)
        ours = O.euclidean_dist(xv, e)
        assert torch.equal(ours, torch.cdist(xv.contiguous(), e, p=2))
        if b >= 2:
            assert torch.equal(live, ours)
        assert ((live - ours).abs() <= 4 * torch.finfo(torch.float32).eps * ours.abs().clamp_min(1e-3)).all()
        assert torch.equal(live.argmin(-1), ours.argmin(-1))
