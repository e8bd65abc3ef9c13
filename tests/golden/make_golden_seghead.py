"""Generates tests/golden/golden_seghead_v1.pt from the LIVE reference VQSegmentationHead (authoring container only).

    python tests/golden/make_golden_seghead.py

Imports /root/reference/models/modules/vq_segmentation_head.py by file path, runs the unmodified class on CPU in
training mode on the seeded inputs of cases.SEGHEAD_CASES and stores outputs and gradients
(loss + sum(score * g) backpropagated to the features and to the prototypes).
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
from oracle.ref_loader import load_reference_seghead  # noqa: E402
import cases  # noqa: E402


def run_case(cls, build, distance):
    x, e = build()
    b, c, h, w = x.shape
    k = e.shape[0]
    m = cls(dim=c, num_embeddings=k, kmeans_init=False, distance=distance)
    emb = m.codebook.embedding if hasattr(m, "codebook") else m.embedding
    emb.weight.data.copy_(e)
    m.train()
    xg = x.clone().requires_grad_(True)
    quantize, score, idx, loss, usage = m(xg)
    g = torch.Generator().manual_seed(4242)
    gs = torch.randn(score.shape, generator=g)
    gq = torch.randn(quantize.shape, generator=g)
    ((score * gs).sum() + (quantize * gq).sum() + 1.5 * loss.sum()).backward()
    rec = {"x_sha": cases.sha(x), "e_sha": cases.sha(e), "shape": (b, c, h, w), "k": k, "distance": distance,
           "quantize": quantize.detach().clone(), "score": score.detach().clone(), "idx": idx.to(torch.int32),
           "loss": loss.detach().clone(), "usage": usage.detach().clone(),
           "gx": xg.grad.clone(), "gw": emb.weight.grad.clone(), "w_after": emb.weight.detach().clone()}
    m.eval()
    with torch.no_grad():
        q2, s2, i2, l2, u2 = m(x)
    rec["quantize_eval"] = q2.clone(); rec["score_eval"] = s2.clone(); rec["loss_eval"] = l2.clone()
    assert torch.equal(i2.to(torch.int32), rec["idx"])
    return rec


def main():
    R = load_reference_seghead()
    assert R is not None, "reference not found: set VQSEG_REF to a checkout of the original repository"
    torch.set_num_threads(os.cpu_count())
    out = {"meta": {"torch": torch.__version__, "threads": torch.get_num_threads()}, "seghead": {}}
    for name, (build, distance) in cases.SEGHEAD_CASES.items():
        out["seghead"][name] = run_case(R.VQSegmentationHead, build, distance)
        print(name, "usage", out["seghead"][name]["usage"].item(), "loss", out["seghead"][name]["loss"].item())
    path = os.path.join(HERE, "golden_seghead_v1.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
