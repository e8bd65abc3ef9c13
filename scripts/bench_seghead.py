"""Times the VQ segmentation head (Euclidean + Softmax2d) on one GPU and prints one JSON line.

Per shape: the module's eval forward (no_grad) and train forward + backward, the map kernel and its backward alone
(replayed from a CUDA graph, with the FLOP rate of the 2NKD contraction each one runs), the backward again with
VQSEG_SEGHEAD_DETERMINISTIC (what the head runs under torch.use_deterministic_algorithms), and the same head written
with torch ops on the same GPU (cdist, normalisation, Softmax2d, autograd).  The fp32 rate denominator is a cuBLAS SGEMM (8192^3, TF32 off) timed in
the same call; the device name and power limit are read in the same call too.  CUDA events over --iters iterations
after warm-up; the inputs are cycled through enough buffers to exceed the 126 MB L2.

    python scripts/bench_seghead.py [--iters 100] [--warmup 10]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vq_seg_b200 as V  # noqa: E402
from vq_seg_b200 import ops  # noqa: E402

SHAPES = [(4, 32, 256, 256, 3), (4, 64, 256, 256, 150), (4, 256, 128, 128, 150), (2, 512, 64, 64, 150)]
L2_BYTES = 126 << 20


def timed(fn, inputs, iters, warmup):
    """mean ms per call of fn(inputs[i % len(inputs)])"""
    for i in range(warmup):
        fn(inputs[i % len(inputs)])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(inputs[i % len(inputs)])
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def graphed(fn, inputs, iters, warmup):
    """mean us per call of fn over the inputs, replayed from one CUDA graph that holds a call per input (the kernels
    without the host's launch latency)"""
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        for v in inputs:
            fn(v)
    torch.cuda.current_stream().wait_stream(st)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for v in inputs:
            fn(v)
    reps = max(1, iters // len(inputs))
    return 1e3 * timed(lambda _: gr.replay(), [None], reps, max(1, warmup // len(inputs))) / len(inputs)


def torch_head(x, w):
    """the reference head's Euclidean + Softmax2d score path in torch ops"""
    b, c, h, wd = x.shape
    xv = x.reshape(b, c, h * wd).permute(0, 2, 1)
    dist = torch.cdist(xv, w, p=2)
    idx = dist.argmin(-1)
    score = dist.permute(0, 2, 1).reshape(b, -1, h, wd)
    score = nn.functional.softmax(1 - score / score.sum(1, keepdim=True), dim=1)
    return score, idx, torch.bincount(idx.reshape(-1), minlength=w.shape[0])


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        out = f"unavailable ({exc})"
    return name, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_seghead.py needs a CUDA device")
    dev = torch.device("cuda:0")
    name, power = device_info()
    torch.backends.cuda.matmul.allow_tf32 = False
    n = 8192
    ga, gb = torch.randn(n, n, device=dev), torch.randn(n, n, device=dev)
    sgemm_ms = timed(lambda _: torch.mm(ga, gb), [None], 20, 3)
    sgemm_tflops = 2 * n ** 3 / sgemm_ms / 1e9
    del ga, gb
    rows = []
    gen = torch.Generator(device="cuda").manual_seed(0)
    for (b, c, h, w, k) in SHAPES:
        nbuf = max(2, -(-2 * L2_BYTES // (b * c * h * w * 4)))
        xs = [torch.relu(torch.randn(b, c, h, w, generator=gen, device=dev)) for _ in range(nbuf)]
        e = xs[0].permute(0, 2, 3, 1).reshape(-1, c)[:k].clone() + 0.05
        m = V.VQSegmentationHead(dim=c, num_embeddings=k).to(dev)
        m.codebook.embedding.weight.data.copy_(e)
        wt = e.clone().requires_grad_(True)
        flop = 2.0 * b * h * w * k * c
        r = {"shape": [b, c, h, w], "K": k, "N": b * h * w, "gflop_fwd": flop / 1e9}

        m.eval()
        with torch.no_grad():
            r["module_eval_fwd_us"] = 1e3 * timed(lambda x: m(x), xs, args.iters, args.warmup)
            r["torch_eval_fwd_us"] = 1e3 * timed(lambda x: torch_head(x, e), xs, args.iters, args.warmup)
        m.train()
        gs = torch.randn(b, k, h, w, generator=gen, device=dev)

        def step(x):
            xg = x.requires_grad_(True)
            q, s, _, loss, _ = m(xg)
            ((s * gs).sum() + loss.sum()).backward()
            x.requires_grad_(False)

        def tstep(x):
            xg = x.requires_grad_(True)
            s, _, _ = torch_head(xg, wt)
            (s * gs).sum().backward()
            x.requires_grad_(False)

        r["module_train_fwd_bwd_us"] = 1e3 * timed(step, xs, args.iters, args.warmup)
        r["torch_train_fwd_bwd_us"] = 1e3 * timed(tstep, xs, args.iters, args.warmup)

        # the kernels alone (AUTO: per-pixel for the 3-class head, tiled otherwise)
        views = [x.reshape(b, c, h * w).permute(0, 2, 1) for x in xs]
        r["map_us"] = graphed(lambda v: ops._seghead_score_map_impl(v, e), views, args.iters, args.warmup)
        dm, sc, _, _ = ops._seghead_score_map_impl(views[0], e)
        g = torch.randn_like(sc)
        r["bwd_us"] = graphed(lambda v: ops._seghead_map_bwd_impl(g, dm, v, e, False, sc), views, args.iters, args.warmup)
        det = ops.SEGHEAD_AUTO | ops.SEGHEAD_DETERMINISTIC
        r["bwd_det_us"] = graphed(lambda v: ops._seghead_map_bwd_impl(g, dm, v, e, False, sc, det), views, args.iters,
                                  args.warmup)
        r["map_tflops"] = flop / r["map_us"] / 1e6
        r["bwd_tflops"] = 2 * flop / r["bwd_us"] / 1e6          # gx and gE: two contractions of 2NKD each
        r["map_frac_of_sgemm"] = r["map_tflops"] / sgemm_tflops
        r["bwd_frac_of_sgemm"] = r["bwd_tflops"] / sgemm_tflops
        r["eval_speedup_vs_torch"] = r["torch_eval_fwd_us"] / r["module_eval_fwd_us"]
        r["train_speedup_vs_torch"] = r["torch_train_fwd_bwd_us"] / r["module_train_fwd_bwd_us"]
        rows.append({kk: (round(v, 4) if isinstance(v, float) else v) for kk, v in r.items()})
        del xs, views, dm, sc, g, gs, m
        torch.cuda.empty_cache()
    print(json.dumps({"device": name, "power_limit": power, "sgemm_fp32_tflops": round(sgemm_tflops, 2),
                      "iters": args.iters, "rows": rows}))


if __name__ == "__main__":
    main()
