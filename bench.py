#!/usr/bin/env python
"""bench.py -- VQ lookup throughput on B200 (BASELINE.json metric: "VQ lookup vectors/sec at K=512, D=256").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): N = 8 x 64 x 64 latent vectors, D = 256, K = 512 codebook, fp32, per GPU.
One "step" = one eval-mode lookup of the whole batch: nearest-code assignment (tcgen05 filter + exact
rescoring, indices + per-code counts) + codebook gather (quantized NCHW tensor) + code usage -- i.e.
everything VectorQuantizer.forward returns (vq_img.py:228-244).  Inputs are synthetic (seeded randn).
  value : whole-job vectors/s with inputs resident in HBM; a ring of input/output batches larger than
          L2 is cycled so no step finds its input in cache.
  e2e   : the same metric through the public nn.Module API with HOST (pinned) input, host->device copy
          and device->host read of indices + usage inside the timed region.
  roofline : the dominant kernel (assign_tc_kernel): 2*N*K*D flops / its CUDA-event duration vs the
          measured dense bf16/fp16 tensor peak of MEASURED_PEAKS.json.
  cpu_baseline : the oracle port of the reference's CPU path on the box's host cores (rank 0, N=1).
With --impl reference the reference's CPU path itself is timed (oracle port, or the original module when
VQSEG_REF points to a checkout of it) on the same workload.
--dump-outputs DIR writes what the last timed step returned (quantize, embed_index, loss, code_usage; rank 0's
with several GPUs) as DIR/<name>.npy, floats as float32 and integers as float64.  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.  The GPU arm's last step reads ring slot
(steps - 1) % ring; slot 0 is the seed-0 batch and codebook, which tests/golden pins as case "c2_randn".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B, C, H, W, K = 8, 256, 64, 64, 512
N_VEC = B * H * W
METRIC = "vq_lookup_vectors_per_sec"
WORKLOAD = "VQ codebook lookup microbench: N=8x64x64 latent vectors, D=256, K=512, fp32 (BASELINE.json configs[1])"


def make_inputs(seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=g)
    e = torch.randn(K, C, generator=g)
    return x.to(device), e.to(device)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower() == "active":
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_reference_step(model, x):
    with torch.no_grad():
        return model(x)


def dump_outputs(out_dir, outputs):
    """(quantize, embed_index, loss, code_usage) of one forward -> out_dir/<name>.npy: floating outputs as float32,
    integer ones as float64 (exact for any index).  The C2 batch comes to 32 MiB of quantize + 256 KiB of indices."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(("quantize", "embed_index", "loss", "code_usage"), outputs):
        t = t.detach().cpu()
        t = t.to(torch.float32 if t.is_floating_point() else torch.float64)
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def build_cpu_model(e):
    """The reference's CPU path: the original module if VQSEG_REF points to a checkout of it, else the oracle port."""
    from oracle.ref_loader import load_reference_vq_img
    ref = load_reference_vq_img()
    if ref is not None:
        m, kind = ref.VectorQuantizer(dim=C, num_embeddings=K), "reference"
    else:
        from oracle.vq_oracle import OracleVectorQuantizer
        m, kind = OracleVectorQuantizer(dim=C, num_embeddings=K), "port"
        m.faithful_ops = True          # the reference's literal op sequence: cdist -> argmin -> one_hot -> matmul -> bincount
    m.codebook.embedding.weight.data.copy_(e)
    m.eval()
    return m, kind


def run_reference(args, rank, world):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count())
    x, e = make_inputs(0)
    model, kind = build_cpu_model(e)
    for _ in range(max(1, min(args.warmup, 3))):
        cpu_reference_step(model, x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = cpu_reference_step(model, x)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    val = N_VEC * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "vectors/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "device": "host CPU, torch eager"},
            "cpu_baseline": {"value": val, "unit": "vectors/s", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": f"{args.steps} full eval-mode forwards of the C2 batch ({N_VEC} vectors each)"},
            "e2e": {"value": val, "unit": "vectors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# =====================================================================================================================
# extras: the other BASELINE.json configs, measured in the same run (the headline keys above stay config 2)
# =====================================================================================================================
def _ev_time(fn, iters, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def extras_c1(dev):
    """configs[0] on the GPU: VectorQuantizer train-mode forward + backward at the three resnet50 latent shapes of a
    2x3x512x512 batch (models/encoders/resnet.py:150-162), K=512, through the public module."""
    import vq_seg_b200 as V
    out = {}
    for name, (b, c, h, w) in {"l3": (2, 512, 64, 64), "l4": (2, 1024, 32, 32), "l5": (2, 2048, 16, 16)}.items():
        g = torch.Generator(device=dev).manual_seed(42)
        m = V.VectorQuantizer(dim=c, num_embeddings=512).to(dev).train()
        m.codebook.embedding.weight.data.normal_(generator=g)
        x = torch.randn(b, c, h, w, generator=g, device=dev, requires_grad=True)
        gq = torch.randn(b, c, h, w, generator=g, device=dev)
        one = torch.ones(1, device=dev)

        def step():
            q, idx, loss, usage = m(x)
            torch.autograd.backward((q, loss), (gq, one))
            x.grad = None
        us = _ev_time(step, 30, 5) * 1e3
        # the same training forward + backward captured by torch.cuda.make_graphed_callables (the codebook gets no
        # gradient in training, hence allow_unused_input): GPU time instead of host time, results bit-equal to eager
        us_train_graph = None
        try:
            xs = x.detach().clone().requires_grad_(True)
            gm = torch.cuda.make_graphed_callables(m, (xs,), allow_unused_input=True)

            def gstep():
                q, idx, loss, usage = gm(x)
                torch.autograd.backward((q, loss), (gq, one))
                x.grad = None
            us_train_graph = _ev_time(gstep, 50, 5) * 1e3
        except Exception as exc:  # noqa: BLE001 -- an extra, never fatal to the bench line
            us_train_graph = "failed: %s" % (str(exc)[:120],)
        with torch.no_grad():
            m.eval()
            us_eval = _ev_time(lambda: m(x), 30, 5) * 1e3
            m.enable_cuda_graphs()                 # the same call replayed as one CUDA graph: GPU time, not host time
            xd = x.detach()
            us_graph = _ev_time(lambda: m(xd), 50, 5) * 1e3
        n = b * h * w
        out[name] = {"shape": [b, c, h, w], "train_fwd_bwd_us": us, "train_fwd_bwd_cuda_graph_us": us_train_graph, "eval_fwd_us": us_eval, "eval_fwd_cuda_graph_us": us_graph,
                     "train_vectors_per_s": n / (us * 1e-6)}
    return out


def extras_c4(dev, rank, world, n_total=10_000_000, d=512, k=1024, iters=3):
    """configs[3]: k-means codebook init (vq_img.py:29-63), N = 10 M latent vectors, K=1024, D=512, rows sharded over
    the ranks; every iteration = assign (tcgen05 filter + rescoring) + per-code counts and sums + ONE all-reduce of
    counts and sums (inside the timed region) + finalize."""
    import torch.distributed as dist
    from vq_seg_b200 import ops, distributed as D
    n = n_total // world
    # synthetic latents WITH cluster structure (a mixture of K Gaussians: centres randn, sigma 0.5) -- k-means on pure
    # iid noise has no structure to find, and its near-zero centroids make every code a near-tie for every row
    gc = torch.Generator(device=dev).manual_seed(99)
    centres = torch.randn(k, d, generator=gc, device=dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.empty(1, n, d, device=dev)
    for i in range(0, n, 1 << 20):
        m = min(1 << 20, n - i)
        x[0, i:i + m].normal_(generator=g).mul_(0.5)
        x[0, i:i + m] += centres[torch.randint(0, k, (m,), generator=g, device=dev)]
    means = x[0, :k].clone()                                  # sample_vectors (vq_img.py:10-17): K rows of the data
    if world > 1:
        dist.broadcast(means, src=0)
    # the product's kmeans() converts a large sample set ONCE to the filter's fp16 operand (prepare_samples) and every
    # Lloyd iteration streams it: timed separately, amortised over the reference's 10 iterations in `iter_ms_amortised`
    samples = ops.prepare_samples(x)                          # (first call: allocation of the 10 GB blob, module load)
    del samples
    prep_ms = _ev_time(lambda: ops.prepare_samples(x), 1, 0)
    samples = ops.prepare_samples(x)
    rescored = []
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    t_assign, t_stats, t_ar, t_iter, t_filter, t_rescore = [], [], [], [], [], []
    from vq_seg_b200 import _native
    prof = _native.ProfileEvents()                            # the filter / rescoring kernels' own times (events in the C ABI)
    for it in range(iters + 1):
        ev[0].record()
        blob = ops.prepare_codebook(means)
        ops.set_profile_events(prof)
        buckets, _ = ops.assign(x, means, blob, ops.ALGO_AUTO, 0, samples)
        ops.set_profile_events(None)
        ev[1].record()
        ws = ops._last_assign_ws
        bins, sums = ops.code_stats(x, buckets, k, False)
        ev[2].record()
        D.allreduce_code_stats(bins, sums)
        ev[3].record()
        ops.kmeans_finalize(sums, bins, means, False)
        ev[4].record()
        torch.cuda.synchronize()
        if it > 0:                                            # first iteration = warm-up
            rescored.append(ws[:4].view(torch.int32).item() / n)
            t_assign.append(ev[0].elapsed_time(ev[1])); t_stats.append(ev[1].elapsed_time(ev[2]))
            t_ar.append(ev[2].elapsed_time(ev[3])); t_iter.append(ev[0].elapsed_time(ev[4]))
            t_filter.append(prof.filter_ms()); t_rescore.append(prof.rescore_ms())
    # the bit-exact ordered statistics (the reference's scatter_add_ order), once
    det_ms = _ev_time(lambda: ops.code_stats(x, buckets, k, True), 1, 1)
    vals = torch.tensor([statistics.median(t_assign), statistics.median(t_stats), statistics.median(t_ar),
                         statistics.median(t_iter), det_ms, statistics.median(t_filter), statistics.median(t_rescore), prep_ms], device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    a_ms, s_ms, ar_ms, it_ms, det_ms, f_ms, r_ms, prep_ms = [float(v) for v in vals.tolist()]
    total = int(bins.sum().item())
    return {"rows_total": n * world, "rows_per_gpu": n, "D": d, "K": k, "iter_ms": it_ms, "assign_ms": a_ms, "stats_atomic_ms": s_ms,
            "allreduce_ms": ar_ms, "allreduce_bytes": k * 8 + k * d * 4, "stats_ordered_ms": det_ms,
            "vector_iters_per_s": n * world / (it_ms * 1e-3), "assign_tflops_per_gpu": 2.0 * n * k * d / (a_ms * 1e-3) / 1e12,
            "samples_prepare_ms_once": prep_ms, "iter_ms_amortised_over_10_iterations": it_ms + prep_ms / 10.0,
            "filter_kernel_ms": f_ms, "rescoring_kernels_ms": r_ms,
            "filter_kernel_tflops_per_gpu": 2.0 * n * k * d / (f_ms * 1e-3) / 1e12 if f_ms > 0 else None,
            "assign_is": "codebook preparation + tcgen05 filter (assign_tc4_kernel on the prepared fp16 samples) + exact rescoring of the undecided rows",
            "stats_atomic_GBps_per_gpu": (4.0 * n * d + 8.0 * n) / (s_ms * 1e-3) / 1e9,
            "counts_sum_equals_rows": total == n * world, "rows_rescored_frac": max(rescored),
            "data": "mixture of K Gaussians (centres randn, sigma 0.5), rank-seeded; start = K rows of rank 0", "collective": "all_reduce(SUM) of counts[K] int64 + sums[K,D] fp32, inside the timed iteration",
            "scaling": "strong (10 M rows split over the ranks)"}


def extras_c5(dev, rank, world, n=4 << 20, d=256, k=65536):
    """configs[4]: large-codebook assignment, N = 4 Mi rows, K = 65536, D = 256.  (a) codebook-sharded: every rank
    scores ALL rows against K / world codes and the ranks MIN-all-reduce 8-byte (distance, index) keys (inside the
    timed region); (b) row-sharded: every rank scores N / world rows against the whole codebook, no exchange."""
    import torch.distributed as dist
    from vq_seg_b200 import ops, distributed as D
    g = torch.Generator(device=dev).manual_seed(77)           # same rows and codebook on every rank
    x = torch.empty(1, n, d, device=dev)
    for i in range(0, n, 1 << 20):
        x[0, i:i + (1 << 20)].normal_(generator=g)
    e = torch.randn(k, d, generator=g, device=dev)
    kl = k // world
    shard = e[rank * kl:(rank + 1) * kl].contiguous()
    blob_s = ops.prepare_codebook(shard)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    t_local, t_ar = [], []
    idx = None
    for it in range(2):
        ev[0].record()
        keys = ops.assign_keys(x, shard, blob_s, rank * kl, ops.ALGO_AUTO)
        ev[1].record()
        if world > 1:
            dist.all_reduce(keys, op=dist.ReduceOp.MIN)
        idx, dd, counts = ops.unpack_keys(keys, k)
        ev[2].record()
        torch.cuda.synchronize()
        if it > 0 or world == 1:
            t_local.append(ev[0].elapsed_time(ev[1])); t_ar.append(ev[1].elapsed_time(ev[2]))
    # (b) row-sharded over the whole codebook
    nl = n // world
    xs = x[:, rank * nl:(rank + 1) * nl]
    blob = ops.prepare_codebook(e)
    t_rows = _ev_time(lambda: ops.assign(xs, e, blob, ops.ALGO_AUTO), 1, 0 if world == 1 else 1)
    idx_rows, _ = ops.assign(xs, e, blob, ops.ALGO_AUTO)
    same = bool(torch.equal(idx_rows, idx[:, rank * nl:(rank + 1) * nl]))
    vals = torch.tensor([min(t_local), min(t_ar), t_rows], device=dev)
    flag = torch.tensor([int(same)], device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    l_ms, ar_ms, r_ms = [float(v) for v in vals.tolist()]
    return {"rows": n, "D": d, "K": k, "codes_per_gpu": kl,
            "sharded_local_assign_ms": l_ms, "sharded_min_allreduce_plus_unpack_ms": ar_ms, "allreduce_bytes": 8 * n,
            "sharded_vectors_per_s": n / ((l_ms + ar_ms) * 1e-3), "sharded_assign_tflops_per_gpu": 2.0 * n * kl * d / (l_ms * 1e-3) / 1e12,
            "row_split_ms": r_ms, "row_split_vectors_per_s": n / (r_ms * 1e-3),
            "row_split_assign_tflops_per_gpu": 2.0 * nl * k * d / (r_ms * 1e-3) / 1e12,
            "sharded_equals_row_split": bool(flag.item() == 1),
            "collective": "all_reduce(MIN) of (float_bits(dist) << 32 | index) int64 keys, inside the timed region"}


def extras_cpu_port(budget_s=25.0):
    """The reference's CPU path (oracle port, or the original module when VQSEG_REF is set) beside the extras, at the
    largest sizes that finish in seconds: it cannot hold configs 4 and 5 at full size (BASELINE.md 2)."""
    from oracle import vq_oracle as O
    torch.set_num_threads(os.cpu_count())
    out = {"cores": torch.get_num_threads(), "kind": "port"}
    t_start = time.perf_counter()
    g = torch.Generator().manual_seed(42)
    for name, (b, c, h, w) in {"l3": (2, 512, 64, 64), "l4": (2, 1024, 32, 32), "l5": (2, 2048, 16, 16)}.items():
        m = O.OracleVectorQuantizer(dim=c, num_embeddings=512)
        m.faithful_ops = True
        m.train()
        x = torch.randn(b, c, h, w, generator=g, requires_grad=True)
        gq = torch.randn(b, c, h, w, generator=g)
        best = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            q, idx, loss, usage = m(x)
            torch.autograd.backward((q, loss), (gq, torch.ones(1)))
            x.grad = None
            best = min(best, time.perf_counter() - t0)
        out["c1_" + name + "_train_fwd_bwd_ms"] = best * 1e3
    if time.perf_counter() - t_start < budget_s:
        n, d, k = 100_000, 512, 1024
        xs = torch.randn(1, n, d, generator=g)
        t0 = time.perf_counter()
        O.kmeans(xs, k, 1, init_indices=torch.arange(k))
        dt = time.perf_counter() - t0
        out["c4_sample"] = f"N={n}, K={k}, D={d}, 1 Lloyd iteration (the reference needs ~100 GB of temporaries at N=1e7)"
        out["c4_vector_iters_per_s"] = n / dt
    if time.perf_counter() - t_start < budget_s:
        n, d, k = 2048, 256, 65536
        xs, e = torch.randn(1, n, d, generator=g), torch.randn(k, d, generator=g)
        t0 = time.perf_counter()
        O.assign_euclidean(xs, e)
        dt = time.perf_counter() - t0
        out["c5_sample"] = f"N={n} rows against K={k}, D={d} (the full N x K distance matrix would be 1.1 TB)"
        out["c5_vectors_per_s"] = n / dt
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ring", type=int, default=8, help="input batches cycled so the working set exceeds L2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-extras", action="store_true", help="skip the extras (configs 1, 4, 5, multi-GPU parity)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    import vq_seg_b200 as V
    from vq_seg_b200 import ops, _native
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200 GPU (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line.  NCCL_DEBUG=VERSION (set in the GPU image) does nothing but print
        # "NCCL version ..." to stdout ahead of it: drop that level; WARN / INFO requests are left alone
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)
    lib = _native.lib()
    args.warmup = max(args.warmup, 3)

    # ---- inputs: ring of batches (each rank its own data: data-parallel over latent pixels, weak scaling)
    xs, e = [], None
    for r in range(args.ring):
        x, e0 = make_inputs(1000 * rank + r)
        xs.append(x.to(dev))
        if e is None:
            _, e = make_inputs(0)
    e = e.to(dev)
    model = V.VectorQuantizer(dim=C, num_embeddings=K).to(dev)
    model.codebook.embedding.weight.data.copy_(e)
    model.codebook.invalidate()
    model.eval()
    views = [x.reshape(B, C, H * W).permute(0, 2, 1) for x in xs]
    # One step = the PUBLIC module call, model(x): VectorQuantizer.forward in eval mode under no_grad.  With
    # enable_cuda_graphs() (the module's own opt-in) each input buffer of the ring gets one captured graph of the
    # forward's four launches (prologue, tcgen05 filter, exact rescoring, gather) and a call is one graph replay;
    # --no-graph times the same call enqueueing its kernels from Python.
    if not args.no_graph:
        model.enable_cuda_graphs(max_entries=args.ring + 4)

    def step(i):
        with torch.no_grad():
            return model(xs[i % args.ring])        # (quantize, embed_index, loss, code_usage)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(25 * args.ring):     # every ring slot before anything is timed: with the module's CUDA graphs this is
        step(i)                         # where each slot's forward gets captured; 25 rounds (~10 ms) let clocks and caches settle
    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        out = step(i)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)    # before any further call overwrites the captured graph's outputs
    # ---- dominant kernel duration: CUDA events recorded by the C ABI on the launching stream around the filter
    # (which=0) and rescoring (which=1) kernels.  Captured into a second set of graphs so the kernels are timed
    # under the same launch conditions as the timed region (graph replay, ring of cold inputs).
    kt, rt = [], []
    prof = _native.ProfileEvents()
    ops.set_profile_events(prof)
    if not args.no_graph:
        model.enable_cuda_graphs(max_entries=args.ring + 4)      # fresh cache: the forwards are re-captured WITH the events
    for i in range(64 + args.ring):
        step(i)
        torch.cuda.synchronize()
        if i >= args.ring:
            kt.append(prof.filter_ms())
            rt.append(prof.rescore_ms())
    kt = [v for v in kt if v > 0]
    ops.set_profile_events(None)
    if not args.no_graph:
        model.enable_cuda_graphs(max_entries=args.ring + 4)      # and again without them for the e2e section
    sampler.stop_flag = True
    sampler.join(timeout=2)
    global_usage = None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        gc = model.codebook.lookup(views[0])[1].clone()
        torch.cuda.synchronize()
        dist.all_reduce(gc)
        global_usage = float(ops.code_usage(gc).item())
    value = N_VEC * world * args.steps / (ms * 1e-3)

    # ---- e2e: public module API, pinned host input, H2D + D2H inside the timed region
    host_x = [x.cpu().pin_memory() for x in xs[:min(4, args.ring)]]
    host_q = [torch.empty(B, C, H, W, dtype=torch.float32).pin_memory() for _ in range(2)]
    host_idx = [torch.empty(B, H, W, dtype=torch.int64).pin_memory() for _ in range(2)]
    host_usage = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    dev_in = [torch.empty(B, C, H, W, device=dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    out_stream = torch.cuda.Stream()                    # device -> host copies: PCIe is full duplex, they overlap the next H2D
    ev_in = [torch.cuda.Event() for _ in range(2)]      # H2D of slot done
    ev_free = [torch.cuda.Event() for _ in range(2)]    # compute on slot done (slot reusable)
    ev_done = [torch.cuda.Event() for _ in range(2)]    # forward on slot done (its outputs can be copied out)
    ev_out = [torch.cuda.Event() for _ in range(2)]     # D2H of slot's outputs done (the graph may overwrite them)
    e2e_steps = max(5, min(args.steps, 100))
    main = torch.cuda.current_stream()

    def issue_h2d(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[s])
            dev_in[s].copy_(host_x[i % len(host_x)], non_blocking=True)
            ev_in[s].record(copy_stream)

    def e2e_run(n):
        # every step: pinned host -> device copy of ITS input (copy stream, overlapping the previous step's
        # kernels, as a pinned-memory data loader does), the public nn.Module forward, and a device -> host read
        # of EVERYTHING it returns: the quantized map, the indices and the usage.  One host sync at the end.
        for s in range(2):
            ev_free[s].record(main)
            ev_out[s].record(out_stream)
        issue_h2d(0)
        for i in range(n):
            s = i % 2
            if i + 1 < n:
                issue_h2d(i + 1)
            main.wait_event(ev_in[s])
            main.wait_event(ev_out[s])                 # the slot's previous outputs have left the device
            with torch.no_grad():
                q, idx, loss, usage = model(dev_in[s])
            ev_free[s].record(main)
            ev_done[s].record(main)
            with torch.cuda.stream(out_stream):
                out_stream.wait_event(ev_done[s])
                for t_ in (q, idx, usage):
                    t_.record_stream(out_stream)       # (eager mode: fresh tensors of the main stream's allocator)
                host_q[s].copy_(q, non_blocking=True)
                host_idx[s].copy_(idx, non_blocking=True)
                host_usage[s].copy_(usage, non_blocking=True)
                ev_out[s].record(out_stream)
        main.synchronize()
        copy_stream.synchronize()
        out_stream.synchronize()

    e2e_run(4)
    e2e_passes = []
    for _ in range(5):                 # five passes: the PCIe link of a shared host is noisy (+-15 %); median reported,
        barrier()                      # best alongside
        t0 = time.perf_counter()
        e2e_run(e2e_steps)
        barrier()
        e2e_passes.append(time.perf_counter() - t0)
    if world > 1:
        t = torch.tensor(e2e_passes, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_passes = t.tolist()
    sampler.stop_flag = True          # clocks sampled from the first timed step to the end of the e2e passes (same workload)
    sampler.join(timeout=2)
    e2e_s = statistics.median(e2e_passes)
    e2e_val = N_VEC * world * e2e_steps / e2e_s
    e2e_best = N_VEC * world * e2e_steps / min(e2e_passes)

    # ---- extras: the other BASELINE configs (and, for N > 1, the multi-GPU parity check), same run
    extras = None
    if not args.no_extras:
        extras = {}
        try:
            if world == 1:
                extras["c1_vqreptunet_layers_train_fwd_bwd"] = extras_c1(dev)
            torch.cuda.empty_cache()
            extras["c4_kmeans_10M_K1024_D512"] = extras_c4(dev, rank, world)
            torch.cuda.empty_cache()
            extras["c5_K65536_D256_N4Mi"] = extras_c5(dev, rank, world)
            torch.cuda.empty_cache()
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            if world > 1:
                from multi_gpu_parity import run_parity
                extras["parity"] = run_parity(rank, world, dev)
            torch.cuda.empty_cache()
            from train_step_c3 import run_c3                  # BASELINE configs[2]: the training step, "train img/s"
            extras["c3_train_step"] = run_c3(dev, rank, world, steps=6, warmup=5)
            torch.cuda.empty_cache()
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                extras["cpu_port"] = extras_cpu_port()
        except Exception as exc:                            # the headline line must still print
            extras["error"] = f"{type(exc).__name__}: {exc}"
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops", 1590.0)
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops, burst; fp16 runs at the same rate)" if peaks else "fallback 1.59 PFLOP/s"
        k_ms = statistics.median(kt) if kt else None
        flops = 2.0 * N_VEC * K * C
        roof = None
        if k_ms:
            ach = flops / (k_ms * 1e-3) / 1e12
            traffic, traffic_src = None, "no profiles/kernel_traffic.json"
            try:                                    # dram bytes per launch of that kernel, written from an ncu --set full
                kt_json = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))       # capture by
                rec = kt_json["kernels"]["assign_tc3_kernel"]                                          # scripts/summarize_ncu.py
                traffic = rec["dram_bytes_read"] + rec["dram_bytes_write"]
                traffic_src = f"bytes/launch, dram read+write, {kt_json.get('source', 'ncu --set full')}; algorithmic {N_VEC * C * 4 + K * C * 2 + N_VEC * 8:.4g}"
            except Exception:
                pass
            roof = {"bound": "tensor", "kernel": "assign_tc3_kernel (TMA-fed tcgen05 cta_group::2 filter)", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": ach / peak_tf, "traffic": traffic, "traffic_unit": traffic_src,
                    "peak_source": peak_src, "kernel_ms": k_ms,
                    "algorithmic_flops_per_launch": flops, "rescore_kernel_ms": (statistics.median([v for v in rt if v > 0]) if any(v > 0 for v in rt) else None)}
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            torch.set_num_threads(os.cpu_count())
            xc, ec = make_inputs(0)
            cm, kind = build_cpu_model(ec)
            cpu_reference_step(cm, xc)
            reps, t0 = 0, time.perf_counter()
            while reps < 20 and (time.perf_counter() - t0 < 10.0 or reps < 3):
                cpu_reference_step(cm, xc); reps += 1
            dt = time.perf_counter() - t0
            cpu = {"value": N_VEC * reps / dt, "unit": "vectors/s", "cores": torch.get_num_threads(), "kind": kind,
                   "sample": f"{reps} full eval-mode forwards of the C2 batch ({N_VEC} vectors each), {dt:.1f} s"}
        line = {"metric": METRIC, "value": value, "unit": "vectors/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 (fp16 tensor-core filter, exact fp32 rescoring)", "data": "synthetic",
                "config": {"workload": WORKLOAD, "per_gpu_vectors": N_VEC, "l2": f"ring of {args.ring} input batches "
                           f"({args.ring * N_VEC * C * 4 / 2**20:.0f} MiB) cycled, larger than L2",
                           "codebook_prepared": "once (weights static)",
                           "settle": f"{25 * args.ring} untimed calls (graph capture of every ring slot, clock ramp) before the warm-up steps", "parallelism": f"dp{world} over latent pixels",
                           "launch": ("model(x), kernels enqueued from Python" if args.no_graph else
                                      "model(x) with VectorQuantizer.enable_cuda_graphs(): one graph replay per call"),
                           "collectives_in_timed_region": 0, "global_code_usage_pct": global_usage},
                "roofline": roof, "cpu_baseline": cpu,
                "e2e": {"value": e2e_val, "unit": "vectors/s", "h2d_bytes_per_step": N_VEC * C * 4,
                        "d2h_bytes_per_step": N_VEC * C * 4 + N_VEC * 8 + 4, "steps": e2e_steps, "best_of_passes": e2e_best,
                        "how": "model(x) (eval, no_grad, module CUDA graphs) per step on pinned host input; H2D of step i+1 on a copy "
                               "stream overlaps step i; quantize + indices + usage copied back to pinned host memory every step on a third "
                               "stream (full-duplex PCIe); median of 5 passes (best alongside)"},
                "gpu_launches": 5 * args.steps,   # per step: prologue / codebook guard, tcgen05 filter, rescoring, overflow rows, gather
                 "clocks": sampler.summary(), "extras": extras}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
