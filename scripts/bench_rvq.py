"""Residual VQ on the B200: ResidualVectorQuantizer against the torch chain of Q VectorQuantizer modules it replaces
(r = r - q; S = S + q), and against VectorQuantizer itself at Q = 1.  One JSON line on stdout.

    python scripts/bench_rvq.py [--rounds 5] [--reps 20] [--quick]

- eval: the no-grad forward of each arm captured as one CUDA graph per input buffer and replayed, with the inputs cycled
  over a ring larger than the 126 MB L2 (every replay reads its input from HBM);
- train: forward + backward of (quantize, loss), eager and under torch.cuda.make_graphed_callables;
- arms alternate within every round; the median over rounds and the spread (max - min) / median are reported;
- a separate torch.profiler pass gives the stage kernel's mean time per stage position at Q = 4 and its rate from the
  algorithmic bytes (a middle stage moves 16 N D bytes in eval -- r, S in, r_next, S out -- and 24 N D in training, with
  A in and out), as a share of the 6.54 TB/s the repository measured on this GPU (DESIGN.md).
The device name and power limit are read in the same call."""
import argparse
import json
import os
import re
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MEASURED_TBS = 6.54
MAPS = {"c2": (8, 256, 64, 64), "c1_l3": (2, 512, 64, 64)}
K = 512


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except Exception as e:                                   # noqa: BLE001
        name, power = torch.cuda.get_device_name(), f"unknown ({e})"
    return name, power


def ring_of(shape, dev, gen):
    n = max(3, -(-(160 << 20) // (4 * torch.Size(shape).numel())))       # > 126 MB of inputs
    return [torch.randn(shape, generator=gen).to(dev) for _ in range(n)]


def make_arms(shape, nq, dev):
    import vq_seg_b200 as V
    b, c, h, w = shape
    torch.manual_seed(nq)
    rvq = V.ResidualVectorQuantizer(c, K, nq).to(dev)
    for l, layer in enumerate(rvq.layers):
        layer.codebook.embedding.weight.data.normal_().mul_(0.5 ** l)
    chain = []
    for layer in rvq.layers:
        v = V.VectorQuantizer(c, K).to(dev)
        v.codebook.embedding.weight.data.copy_(layer.codebook.embedding.weight)
        chain.append(v)

    def run_chain(x):
        r, s, idx, loss = x, None, [], None
        for v in chain:
            q, i, l_, _ = v(r)
            s = q if s is None else s + q
            loss = l_ if loss is None else loss + l_
            r = r - q
            idx.append(i)
        return s, idx, loss

    arms = {"rvq": rvq, "chain": run_chain}
    if nq == 1:
        arms["vq"] = chain[0]
    return arms, rvq, chain


def graphs_for(fn, ring):
    gs = []
    for x in ring:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn(x)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn(x)
        gs.append((g, out))
    return gs


def timed(call, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        call(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / n                            # us per call


def summary(vals):
    vals = sorted(vals)
    med = vals[len(vals) // 2]
    return {"median_us": round(med, 2), "spread": round((vals[-1] - vals[0]) / med, 3) if med else None}


def bench_shape(name, shape, nq, dev, rounds, reps, gen):
    arms, rvq, chain = make_arms(shape, nq, dev)
    ring = ring_of(shape, dev, gen)
    res = {"map": name, "shape": list(shape), "K": K, "Q": nq}
    # eval, graph replays
    for m in [rvq] + chain:
        m.eval()
    with torch.no_grad():
        graphs = {k: graphs_for(lambda x, f=f: f(x), ring) for k, f in arms.items()}
        times = {k: [] for k in arms}
        for _ in range(rounds):
            for k, gs in graphs.items():
                times[k].append(timed(lambda i, gs=gs: gs[i % len(gs)][0].replay(), reps))
    res["eval_graph"] = {k: summary(v) for k, v in times.items()}
    del graphs
    # train: forward + backward, eager and make_graphed_callables
    for m in [rvq] + chain:
        m.train()
    gy = torch.randn(shape, generator=gen).to(dev)
    one = torch.ones(1, device=dev)
    xs = [x.detach().clone().requires_grad_(True) for x in ring[:4]]

    def step(fn, x):
        out = fn(x)
        torch.autograd.backward((out[0], out[2]), (gy, one))
        x.grad = None

    train_arms = {"rvq": rvq, "chain": arms["chain"]}
    if nq == 1:
        train_arms["vq"] = chain[0]
    graphed = {"rvq": torch.cuda.make_graphed_callables(rvq, (xs[0].detach().clone().requires_grad_(True),),
                                                        allow_unused_input=True)}
    if nq == 1:
        graphed["vq"] = torch.cuda.make_graphed_callables(chain[0], (xs[0].detach().clone().requires_grad_(True),),
                                                          allow_unused_input=True)
    t_eager = {k: [] for k in train_arms}
    t_graph = {k: [] for k in graphed}
    for k, f in list(train_arms.items()) + [("g_" + k, f) for k, f in graphed.items()]:
        for i in range(3):
            step(f, xs[i % len(xs)])
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, f in train_arms.items():
            t_eager[k].append(timed(lambda i, f=f: step(f, xs[i % len(xs)]), reps))
        for k, f in graphed.items():
            t_graph[k].append(timed(lambda i, f=f: step(f, xs[i % len(xs)]), reps))
    res["train_eager"] = {k: summary(v) for k, v in t_eager.items()}
    res["train_graphed"] = {k: summary(v) for k, v in t_graph.items()}
    return res, rvq, ring


STAGE = re.compile(r"gather_ste_(pxc_kernel<\d+, (true|false), true>|generic_kernel<\d+, true>)")


def profile_stages(rvq, ring, nq, shape, dev, iters=10):
    """mean stage-kernel time per stage position (a separate, traced pass)"""
    from torch.profiler import ProfilerActivity, profile
    b, c, h, w = shape
    nd = b * h * w * c
    out = {}
    for mode in ("eval", "train"):
        rvq.train(mode == "train")
        with torch.no_grad():
            for x in ring[:2]:
                rvq(x)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(iters):
                    if mode == "train":
                        xg = ring[i % len(ring)].detach().requires_grad_(True)
                        with torch.enable_grad():
                            rvq(xg)
                    else:
                        rvq(ring[i % len(ring)])
                torch.cuda.synchronize()
        kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and STAGE.search(e.name)]
        per = [[] for _ in range(nq)]
        for j, e in enumerate(kern):
            per[j % nq].append(e.device_time if hasattr(e, "device_time") else e.cuda_time)
        mid = 16 if mode == "eval" else 24
        pos = []
        for l, ts in enumerate(per):
            us = sum(ts) / max(len(ts), 1)
            entry = {"stage": l, "mean_us": round(us, 2), "n": len(ts)}
            if 0 < l < nq - 1 and us > 0:
                tbs = mid * nd / (us * 1e-6) / 1e12
                entry.update(bytes=mid * nd, tb_s=round(tbs, 3), share_of_measured=round(tbs / MEASURED_TBS, 3))
            pos.append(entry)
        out[mode] = pos
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="Q in {1, 2} on c1_l3 only")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_rvq.py needs a CUDA device")
    name, power = device_info()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(0)
    maps = {"c1_l3": MAPS["c1_l3"]} if args.quick else MAPS
    qs = (1, 2) if args.quick else (1, 2, 4, 8)
    results, stages = [], None
    for mname, shape in maps.items():
        for nq in qs:
            res, rvq, ring = bench_shape(mname, shape, nq, dev, args.rounds, args.reps, gen)
            results.append(res)
            if mname == "c2" and nq == 4 or (args.quick and nq == 2):
                stages = {"map": mname, "Q": nq, "positions": profile_stages(rvq, ring, nq, shape, dev)}
            del rvq, ring
            torch.cuda.empty_cache()
    print(json.dumps({"device": name, "power_limit": power, "results": results, "stage_kernel": stages}))


if __name__ == "__main__":
    main()
