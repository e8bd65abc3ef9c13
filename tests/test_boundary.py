"""Host-side mirror of the reference interface (CPU): constructor surface, config keys, state_dict keys,
factory behaviour and error behaviour (reference: vq_img.py:193-226, vector_quantizer/__init__.py:5-32)."""
import inspect
import json
import os

import pytest
import torch

import vq_seg_b200 as V
from oracle.ref_loader import reference_root
from oracle.vq_oracle import OracleVectorQuantizer

REF_CFG = os.path.join(reference_root() or "", "config")


def test_constructor_signature_matches_reference(ref_vq):
    ours = inspect.signature(V.VectorQuantizer.__init__)
    expect = ["self", "dim", "num_embeddings", "embedding_dim", "decay", "eps", "kmeans_init", "kmeans_iters",
              "distance", "commitment_weight", "num_codebook"]
    assert list(ours.parameters) == expect
    d = {k: p.default for k, p in ours.parameters.items()}
    assert (d["embedding_dim"], d["decay"], d["eps"], d["kmeans_init"], d["kmeans_iters"], d["distance"],
            d["commitment_weight"], d["num_codebook"]) == (None, 0.8, 1e-5, False, 10, "euclidean", 1, 1)
    if ref_vq is not None:
        ref = inspect.signature(ref_vq.VectorQuantizer.__init__)
        assert list(ref.parameters) == expect
        assert {k: p.default for k, p in ref.parameters.items()} == d


def test_state_dict_and_attributes(ref_vq):
    m = V.VectorQuantizer(dim=32, num_embeddings=16, kmeans_init=True, kmeans_iters=7, decay=0.5)
    assert list(m.state_dict().keys()) == ["codebook.embedding.weight"]
    assert m.state_dict()["codebook.embedding.weight"].shape == (16, 32)
    assert len(list(m.buffers())) == 0 and len(list(m.parameters())) == 1
    cb = m.codebook
    assert (cb.kmeans_init, cb.kmeans_iters, cb.initted, cb.num_codebook, cb.decay, cb.num_embeddings,
            cb.embedding_dim) == (True, 7, False, 1, 0.5, 16, 32)
    assert (m.num_embeddings, m.eps, m.commitment_weight) == (16, 1e-5, 1)
    m2 = V.VectorQuantizer(dim=32, num_embeddings=16)           # kmeans_init=False -> uniform(-1/K, 1/K), initted
    assert m2.codebook.initted and m2.codebook.embedding.weight.abs().max() <= 1 / 16
    if ref_vq is not None:                                        # checkpoints are interchangeable
        ref = ref_vq.VectorQuantizer(dim=32, num_embeddings=16)
        m2.load_state_dict(ref.state_dict())
        ref.load_state_dict(m2.state_dict())
    OracleVectorQuantizer(dim=32, num_embeddings=16).load_state_dict(m2.state_dict())


def test_errors_match_reference():
    with pytest.raises(KeyError):
        V.VectorQuantizer(dim=8, num_embeddings=4, distance="manhattan")
    with pytest.raises(TypeError):
        V.VectorQuantizer(dim=8, num_embeddings=4, not_a_key=1)
    with pytest.raises(ValueError):
        V.VectorQuantizer(dim=8, num_embeddings=4)(torch.randn(8, 4, 4))      # non-4-D input


def test_make_vq_module():
    chans = [3, 64, 256, 512, 1024, 2048]
    ml = V.make_vq_module({"num_embeddings": [0, 0, 512, 512, 512], "distance": "euclidean", "kmeans_init": True}, chans, 5)
    assert [type(m).__name__ for m in ml] == ["Identity", "Identity"] + ["VectorQuantizer"] * 3
    assert [m.codebook.embedding.weight.shape for m in ml[2:]] == [(512, 512), (512, 1024), (512, 2048)]
    x = torch.randn(1, 4, 2, 2)
    out = ml[0](x)
    assert out[0] is x and out[1:] == (None, None, None)
    ml2 = V.make_vq_module({"num_embeddings": 32, "distance": "cosine", "kmeans_init": False}, chans, 5)
    assert len(ml2) == 5 and ml2[4].codebook.embedding.weight.shape == (32, 2048)
    assert type(ml2[0].codebook).__name__ == "CosinesimCodebook"
    with pytest.raises(ValueError):
        V.make_vq_module({"num_embeddings": [-3]}, chans, 1)
    with pytest.raises(TypeError):
        V.make_vq_module({"num_embeddings": "512"}, chans, 1)
    with pytest.raises(AssertionError):
        V.make_vq_module({"num_embeddings": [0, 512]}, chans, 5)


@pytest.mark.skipif(reference_root() is None, reason="needs a reference checkout (VQSEG_REF) for its config/*.json")
def test_every_reference_vq_cfg_constructs():
    n = 0
    for dirpath, _, files in os.walk(REF_CFG):
        for f in files:
            if not f.endswith(".json"):
                continue
            cfg = json.load(open(os.path.join(dirpath, f)))
            vq_cfg = cfg.get("model", {}).get("params", {}).get("vq_cfg")
            if not vq_cfg:
                continue
            depth = cfg["model"]["params"].get("depth", 5)
            ne = vq_cfg["num_embeddings"]
            depth = len(ne) if isinstance(ne, list) else depth
            V.make_vq_module(vq_cfg, [3, 64, 256, 512, 1024, 2048][:depth + 1], depth)
            n += 1
    assert n >= 30


def test_install_patches_imported_reference_modules():
    import sys
    import types
    fake = types.ModuleType("vector_quantizer")
    fake.VectorQuantizer = object
    sys.modules["vector_quantizer"] = fake
    try:
        assert "vector_quantizer" in V.install()
        assert fake.VectorQuantizer is V.VectorQuantizer
    finally:
        del sys.modules["vector_quantizer"]


def test_custom_ops_registered_with_fake_impls():
    for name in ["assign", "gather_ste", "ste_bwd", "code_stats", "prepare_codebook", "code_usage", "assign_keys"]:
        assert hasattr(torch.ops.vqseg, name)
    x = torch.empty(2, 9, 16, device="meta")
    e = torch.empty(8, 16, device="meta")
    idx, counts = torch.ops.vqseg.assign(x, e, None, 0, 0)
    assert idx.shape == (2, 9) and idx.dtype == torch.int64 and counts.shape == (8,)
    q, mse = torch.ops.vqseg.gather_ste(x, e, idx, 1)
    assert q.shape == (2, 9, 16) and q.stride() == (144, 1, 9) and mse.shape == (1,)


def test_seghead_module_surface():
    """VQSegmentationHead: reference kwargs / defaults / state_dict key, KeyError on an unknown distance, loud
    error (no CPU fallback) on a CPU tensor."""
    import inspect
    import torch
    import vq_seg_b200 as V
    sig = inspect.signature(V.VQSegmentationHead.__init__)
    assert list(sig.parameters)[1:] == ["dim", "num_embeddings", "embedding_dim", "decay", "eps", "kmeans_init",
                                        "kmeans_iters", "distance", "commitment_weight", "num_codebook", "activation"]
    m = V.VQSegmentationHead(dim=16, num_embeddings=3)
    assert list(m.state_dict()) == ["codebook.embedding.weight"] and m.codebook.initted
    assert m.codebook.embedding.weight.abs().max().item() <= 1 / 3
    assert not V.VQSegmentationHead(dim=16, num_embeddings=3, kmeans_init=True).codebook.initted
    with pytest.raises(KeyError):
        V.VQSegmentationHead(dim=16, num_embeddings=3, distance="manhattan")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 16, 4, 4))


def test_ema_extension_surface_and_oracle():
    """enable_ema() keeps the reference's state_dict keys (moving averages are non-persistent buffers); the restated
    rule reduces to the smoothed batch means when decay == 0."""
    from oracle import vq_oracle as O
    m = V.VectorQuantizer(dim=8, num_embeddings=5, decay=0.7, eps=1e-4)
    assert not m.codebook.ema_enabled
    m.enable_ema()
    assert m.codebook.ema_enabled and list(m.state_dict()) == ["codebook.embedding.weight"]
    assert m.codebook.decay == 0.7 and m.codebook.ema_eps == 1e-4 and m.codebook.cluster_size.shape == (5,)
    counts = torch.tensor([4, 0, 2, 1, 3]); sums = torch.randn(5, 8) * counts.unsqueeze(1)
    cs, ea, w = O.ema_update(counts, sums, torch.zeros(5), torch.zeros(5, 8), 0.0, 0.0)
    assert torch.equal(cs, counts.float()) and torch.equal(ea, sums)
    nz = counts > 0
    assert torch.allclose(w[nz], sums[nz] / counts[nz].unsqueeze(1).float())
    assert V.stack_code_usage([torch.tensor(1.0), None, torch.tensor(3.0)]).tolist() == [1.0, 3.0]
