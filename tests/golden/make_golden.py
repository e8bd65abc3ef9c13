"""Generates tests/golden/*.pt from the LIVE reference (run in the authoring container only).

    python tests/golden/make_golden.py

Imports /root/reference/vector_quantizer/vq_img.py by file path (oracle/ref_loader.py), runs the
unmodified reference VectorQuantizer / kmeans on CPU on the seeded inputs of cases.py and stores
the small outputs (indices as int32, counts, loss, usage) plus SHA-256 digests of the big ones
(quantize, inputs).  /root/reference does not exist on the GPU box, so these files are the pin
the GPU parity tests compare against there.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
from oracle.ref_loader import load_reference_vq_img  # noqa: E402
import cases  # noqa: E402


def main():
    R = load_reference_vq_img()
    assert R is not None, "reference not found: set VQSEG_REF to a checkout of the original repository"
    torch.set_num_threads(os.cpu_count())
    out = {"meta": {"torch": torch.__version__, "threads": torch.get_num_threads()}}

    fwd = {}
    for name, build in cases.FORWARD_CASES.items():
        x, e = build()
        b, c, h, w = x.shape
        k = e.shape[0]
        m = R.VectorQuantizer(dim=c, num_embeddings=k, kmeans_init=False)
        m.codebook.embedding.weight.data.copy_(e)
        rec = {"x_sha": cases.sha(x), "e_sha": cases.sha(e), "shape": (b, c, h, w), "k": k}
        m.eval()
        with torch.no_grad():
            q, idx, loss, usage = m(x)
        rec["idx"] = idx.to(torch.int32)
        rec["counts"] = torch.bincount(idx.reshape(-1), minlength=k)
        rec["usage"] = usage.clone()
        rec["q_eval_sha"] = cases.sha(q)
        rec["loss_eval"] = loss.clone()
        m.train()
        xg = x.clone().requires_grad_(True)
        q, idx2, loss, usage2 = m(xg)
        assert torch.equal(idx2.to(torch.int32), rec["idx"])
        g = torch.Generator().manual_seed(999)
        gq = torch.randn(q.shape, generator=g)
        (q * gq).sum().backward(retain_graph=True)
        gx_q = xg.grad.clone(); xg.grad = None
        (loss * 1.5).sum().backward()
        gx_l = xg.grad.clone()
        rec["q_train_sha"] = cases.sha(q)
        rec["q_train_sample"] = q.detach().reshape(-1)[:: max(1, q.numel() // 4096)].clone()
        rec["loss_train"] = loss.detach().clone()
        rec["gx_q_is_gq"] = bool(torch.equal(gx_q, gq))
        rec["gx_l_sample"] = gx_l.reshape(-1)[:: max(1, gx_l.numel() // 4096)].clone()
        rec["gx_l_absmax"] = gx_l.abs().max().clone()
        assert m.codebook.embedding.weight.grad is None
        fwd[name] = rec
        print(f"{name:16s} N={b*h*w:6d} D={c:5d} K={k:5d} usage={usage.item():7.3f} loss={loss.item():.6f}")
    out["forward"] = fwd

    km = {}
    for name in cases.KMEANS_CASES:
        x, k, iters, init_idx, use_cos = cases.kmeans_case(name)
        b, c, h, w = x.shape
        flat = x.reshape(b, c, h * w).permute(0, 2, 1)            # the (B,HW,C) view the codebook sees
        if use_cos:
            flat = R.l2norm(flat)
        orig = R.sample_vectors
        R.sample_vectors = lambda sample, num, _i=init_idx: sample[_i]   # inject the init rows
        try:
            means, bins = R.kmeans(flat, k, iters, use_cosine_sim=use_cos)
        finally:
            R.sample_vectors = orig
        km[name] = {"x_sha": cases.sha(x), "means": means[0].clone(), "bins": bins[0].clone(),
                    "k": k, "iters": iters, "cosine": use_cos}
        print(f"{name:16s} kmeans K={k} iters={iters} empty={(bins[0]==0).sum().item()}")
    out["kmeans"] = km

    cos = {}
    for name, build in cases.COSINE_CASES.items():
        x, e = build()
        b, c, h, w = x.shape
        k = e.shape[0]
        m = R.VectorQuantizer(dim=c, num_embeddings=k, kmeans_init=False, distance="cosine")
        m.codebook.embedding.weight.data.copy_(e)
        m.train()
        q, idx, loss, usage = m(x)
        cos[name] = {"x_sha": cases.sha(x), "idx": idx.to(torch.int32), "usage": usage.clone(),
                     "loss_train": loss.detach().clone(), "q_train_sha": cases.sha(q),
                     "weight_after_sha": cases.sha(m.codebook.embedding.weight.data)}
        print(f"{name:16s} cosine usage={usage.item():.3f} loss={loss.item():.6f}")
    out["cosine"] = cos

    path = os.path.join(HERE, "golden_v1.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
