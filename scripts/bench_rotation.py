"""Cost of the rotation trick on one GPU: prints one JSON line.

Kernel alone: vqseg_ste_bwd_f32 against vqseg_rotate_bwd_f32 on NCHW maps (g, x, q and gx pixel-contiguous, as in the
module's backward): the config-2 map (8 x 256 x 64 x 64) and the three config-1 latent layers (2 x 512 x 64^2,
2 x 1024 x 32^2, 2 x 2048 x 16^2).  Each arm is --launches launches captured in one CUDA graph (no host time in the
window), cycling through enough input sets to exceed the 126 MB L2, timed with CUDA events over --rounds alternating
rounds.  Algorithmic bytes: 16 N D for both (read g, x, q; write gx).  A torch.profiler pass of its own gives the per
kernel average of the same launches.

Module: a training forward + backward of VectorQuantizer (K = 512) through the public module, straight-through
against rotation_trick = True, on identically initialised modules, alternating in rounds as above.
The device name and power limit are read in the same call.

    python scripts/bench_rotation.py [--launches 200] [--iters 200] [--rounds 4] [--warmup 10]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vq_seg_b200 as V  # noqa: E402
from vq_seg_b200 import _native  # noqa: E402

SHAPES = {"c2": (8, 256, 64, 64), "c1_l3": (2, 512, 64, 64), "c1_l4": (2, 1024, 32, 32), "c1_l5": (2, 2048, 16, 16)}
K = 512
L2_BYTES = 126 << 20
HBM_PEAK = 6542e9            # measured HBM copy bandwidth of a B200, for the share of peak


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        out = f"unavailable ({exc})"
    return name, out


def bpd(t):
    b, c, h, w = t.shape
    return t.reshape(b, c, h * w).permute(0, 2, 1)


def launch(fn, g, x, q, gm, gx, scale):
    b, p, d = x.shape
    _native.check(fn(g.data_ptr(), *g.stride(), x.data_ptr(), *x.stride(), q.data_ptr(), *q.stride(), gm.data_ptr(), scale,
                     gx.data_ptr(), *gx.stride(), b, p, d, torch.cuda.current_stream().cuda_stream))


def kernel_arms(shape, dev, launches, rounds):
    L = _native.lib()
    fns = {"ste_bwd": L.vqseg_ste_bwd_f32, "rotate_bwd": L.vqseg_rotate_bwd_f32}
    b, c, h, w = shape
    n_el = b * c * h * w
    nset = max(2, -(-2 * L2_BYTES // (16 * n_el)))
    gen = torch.Generator(device=dev).manual_seed(3)
    sets = [[bpd(torch.randn(shape, generator=gen, device=dev)) for _ in range(4)] for _ in range(nset)]
    gm = torch.ones(1, device=dev)
    scale = 2.0 / n_el
    graphs = {}
    for name, fn in fns.items():
        for i in range(nset):                                 # warm-up (module load, shared-memory attributes)
            launch(fn, *sets[i][:3], gm, sets[i][3], scale)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for i in range(launches):
                s = sets[i % nset]
                launch(fn, s[0], s[1], s[2], gm, s[3], scale)
        graphs[name] = gr
    ms = {name: 0.0 for name in fns}
    for _ in range(rounds):
        for name, gr in graphs.items():
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            gr.replay()
            e.record()
            torch.cuda.synchronize()
            ms[name] += a.elapsed_time(e)
    out = {"shape": list(shape), "input_sets": nset, "launches_per_arm": launches * rounds}
    for name in fns:
        us = ms[name] * 1e3 / (launches * rounds)
        out[f"{name}_us"] = round(us, 2)
        out[f"{name}_share_of_hbm_peak"] = round(16 * n_el / (us * 1e-6) / HBM_PEAK, 3)
    out["rotate_over_ste"] = round(out["rotate_bwd_us"] / out["ste_bwd_us"], 3)
    # torch.profiler pass of its own: per-kernel averages of the same launches
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for gr in graphs.values():
            gr.replay()
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if "rotate_bwd" in ev.key or "ste_bwd" in ev.key:
            kern[ev.key.split("(")[0].replace("vqseg::", "")] = round(ev.device_time_total / max(ev.count, 1), 2)
    out["profiler_avg_us"] = kern
    return out


def module_arms(shape, dev, iters, rounds, warmup):
    b, c, h, w = shape
    gen = torch.Generator(device=dev).manual_seed(42)
    init = torch.randn(K, c, generator=gen, device=dev)
    nbuf = max(2, -(-2 * L2_BYTES // (b * c * h * w * 4)))
    xs = [torch.randn(shape, generator=gen, device=dev).requires_grad_(True) for _ in range(nbuf)]
    gq = torch.randn(shape, generator=gen, device=dev)
    one = torch.ones(1, device=dev)
    mods = {}
    for arm, rot in (("ste", False), ("rotation", True)):
        m = V.VectorQuantizer(dim=c, num_embeddings=K).to(dev).train()
        m.codebook.embedding.weight.data.copy_(init)
        m.rotation_trick = rot
        mods[arm] = m

    def steps(m, n, start):
        for i in range(n):
            x = xs[(start + i) % nbuf]
            q, idx, loss, usage = m(x)
            torch.autograd.backward((q, loss), (gq, one))
            x.grad = None

    for m in mods.values():
        steps(m, warmup, 0)
    torch.cuda.synchronize()
    per_round = max(1, iters // rounds)
    ms = {arm: 0.0 for arm in mods}
    for r in range(rounds):
        for arm, m in mods.items():
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            steps(m, per_round, r * per_round)
            e.record()
            torch.cuda.synchronize()
            ms[arm] += a.elapsed_time(e)
    us = {arm: ms[arm] * 1e3 / (per_round * rounds) for arm in mods}
    return {"input_buffers": nbuf, "steps_per_arm": per_round * rounds, "ste_step_us": round(us["ste"], 2),
            "rotation_step_us": round(us["rotation"], 2), "rotation_added_us": round(us["rotation"] - us["ste"], 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rotation.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    name, power = device_info()
    result = {"device": name, "power_limit": power, "kernel": {}, "module": {}}
    for sname, shape in SHAPES.items():
        result["kernel"][sname] = kernel_arms(shape, dev, args.launches, args.rounds)
    for sname, shape in SHAPES.items():
        result["module"][sname] = module_arms(shape, dev, args.iters, args.rounds, args.warmup)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
