"""Generates tests/golden/golden_cosine_v2.pt from the LIVE reference (run in the authoring container only).

    python tests/golden/make_golden_cosine.py

The unmodified reference VectorQuantizer(distance='cosine') (vq_img.py:65-130, 193-244) on CPU, on the seeded inputs
cases.COSINE2_CASES: one TRAINING forward (indices, quantize, loss, usage, the in-place renormalised weights), then an
EVAL forward of the same module (the weights are renormalised a second time), and the intermediate
l2norm(x) of the strided 'b c h w -> b (h w) c' view.  Indices are stored, big tensors as SHA-256 digests.
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
    out = {"meta": {"torch": torch.__version__, "threads": torch.get_num_threads(),
                    "cpu_capability": torch.backends.cpu.get_cpu_capability()}}
    cos = {}
    for name, build in cases.COSINE2_CASES.items():
        x, e = build()
        b, c, h, w = x.shape
        k = e.shape[0]
        m = R.VectorQuantizer(dim=c, num_embeddings=k, kmeans_init=False, distance="cosine")
        m.codebook.embedding.weight.data.copy_(e)
        xv = x.reshape(b, c, h * w).permute(0, 2, 1)
        rec = {"x_sha": cases.sha(x), "e_sha": cases.sha(e), "xn_sha": cases.sha(R.l2norm(xv)),
               "w1_sha": cases.sha(R.l2norm(e))}
        m.train()
        q, idx, loss, usage = m(x)
        rec.update({"idx_train": idx.to(torch.int32), "usage_train": usage.clone(), "loss_train": loss.detach().clone(),
                    "q_train_sha": cases.sha(q), "w_after_train_sha": cases.sha(m.codebook.embedding.weight.data)})
        m.eval()
        with torch.no_grad():
            q, idx, loss, usage = m(x)
        rec.update({"idx_eval": idx.to(torch.int32), "usage_eval": usage.clone(), "q_eval_sha": cases.sha(q),
                    "w_after_eval_sha": cases.sha(m.codebook.embedding.weight.data),
                    "counts_eval": torch.bincount(idx.reshape(-1), minlength=k)})
        cos[name] = rec
        print(f"{name:12s} usage={usage.item():.3f} loss_train={rec['loss_train'].item():.6f} "
              f"train==eval idx: {bool(torch.equal(rec['idx_train'], rec['idx_eval']))}")
    out["cosine2"] = cos
    # F.normalize itself, where ATen's summation order shows: contiguous rows of every tail length D % 8 (the
    # vectorised last-dim reduction: 8 lanes, then 4 unfused + <= 3 fused tail terms) and strided (B, HW, C) views with
    # pixel counts that are not multiples of 32 (one sequential chain per pixel)
    norm = {}
    g = torch.Generator().manual_seed(4242)
    for d in cases.L2NORM_LASTDIM_DIMS:
        e = torch.randn(200, d, generator=g)
        norm[f"rows_d{d}"] = {"in_sha": cases.sha(e), "out_sha": cases.sha(R.l2norm(e))}
    for (b, c, p) in cases.L2NORM_VIEW_SHAPES:
        x = torch.randn(b, c, p, generator=g)
        norm[f"view_{b}x{c}x{p}"] = {"in_sha": cases.sha(x), "out_sha": cases.sha(R.l2norm(x.permute(0, 2, 1)))}
    out["l2norm"] = norm
    path = os.path.join(HERE, "golden_cosine_v2.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
