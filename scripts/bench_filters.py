"""Each tensor-core filter forced on seeded inputs: its kernel time, the rows it leaves to the rescoring pass, and a hash
of the indices and counts.  Prints one JSON line.

Two builds of libvqseg.so that make the same short-list decisions print the same `flagged` counts and hashes (split-D
mode adds partial scores with float atomics in a varying order, so there only the hashes have to agree).  Run the
script once per build, in separate processes, alternating the builds, to compare their times against the spread of
one build.

Cases: the config-2 map (8 x 256 x 64 x 64, K = 512) through each filter that takes it, config-4 rows (262144 x 512,
K = 1024) plain and as prepared samples, K = 16384 on the config-2 map, and a split-D layer (2 x 2048 x 16 x 16,
K = 512).  Each case runs against a randn codebook (the benchmark's) and against codes drawn from the inputs plus
small noise, whose near-ties fill the short-lists.  Inputs are cycled through enough buffers to exceed the 126 MB L2.
The filter time is the median over --reps calls of the CUDA events the C ABI records around the filter kernel.  The
device name and power limit are read in the same call.

    python scripts/bench_filters.py [--lib path/to/libvqseg.so] [--reps 30] [--warmup 5]
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vq_seg_b200 import _native  # noqa: E402

L2_BYTES = 126 << 20
C2 = (8, 256, 64, 64)
C4_ROWS = (262144, 512)
SPLIT_D = (2, 2048, 16, 16)
# name -> (input: ("map", B, C, H, W) or ("rows", N, D), K, algo name, prepared samples)
CASES = {
    "tc3_c2": (("map",) + C2, 512, "ALGO_TC_TMA", False),
    "tc2_c2": (("map",) + C2, 512, "ALGO_TC_PAIR", False),
    "tc_c2": (("map",) + C2, 512, "ALGO_TC_STREAM", False),
    "tc4_c2": (("map",) + C2, 512, "ALGO_TC_STREAM_PAIR", False),
    "tc4_c4_rows": (("rows",) + C4_ROWS, 1024, "ALGO_TC_STREAM_PAIR", False),
    "tc4_c4_prepared": (("rows",) + C4_ROWS, 1024, "ALGO_AUTO", True),
    "tc_c4_rows": (("rows",) + C4_ROWS, 1024, "ALGO_TC_STREAM", False),
    "tc4_c2_k16384": (("map",) + C2, 16384, "ALGO_AUTO", False),
    "splitd_2x2048x16x16": (("map",) + SPLIT_D, 512, "ALGO_AUTO", False),
}


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        out = f"unavailable ({exc})"
    return name, out


def make_inputs(spec, g, dev):
    """A ring of (B, P, D) views, together larger than twice the L2."""
    if spec[0] == "map":
        b, c, h, w = spec[1:]
        nbuf = max(1, -(-2 * L2_BYTES // (b * c * h * w * 4)))
        return [torch.randn(b, c, h, w, generator=g, device=dev).reshape(b, c, h * w).permute(0, 2, 1)
                for _ in range(nbuf)]
    n, d = spec[1:]
    nbuf = max(1, -(-2 * L2_BYTES // (n * d * 4)))
    return [torch.randn(1, n, d, generator=g, device=dev) for _ in range(nbuf)]


def run_case(ops, spec, k, algo, prepared, kind, reps, warmup, dev):
    g = torch.Generator(device=dev).manual_seed(1234)
    xs = make_inputs(spec, g, dev)
    d = xs[0].shape[2]
    if kind == "randn":
        cb = torch.randn(k, d, generator=g, device=dev)
    else:                                             # codes near the data: many near-ties within the error bound
        rows = xs[0].reshape(-1, d)
        pick = torch.randint(0, rows.shape[0], (k,), generator=g, device=dev)
        cb = rows[pick] + 1e-3 * torch.randn(k, d, generator=g, device=dev)
    blob = ops.prepare_codebook(cb)
    samples = [ops.prepare_samples(x) for x in xs] if prepared else [None] * len(xs)
    a = getattr(ops, algo)
    prof = _native.ProfileEvents()
    times = []
    for i in range(warmup + reps):
        j = i % len(xs)
        ops.set_profile_events(prof)
        ops.assign(xs[j], cb, blob, a, 0, samples[j])
        ops.set_profile_events(None)
        torch.cuda.synchronize()
        if i >= warmup:
            times.append(prof.filter_ms() * 1e3)
    idx, counts = ops.assign(xs[0], cb, blob, a, 0, samples[0])
    flagged = int(ops._last_assign_ws[:4].view(torch.int32)[0].item())
    h = hashlib.sha256(idx.cpu().numpy().tobytes() + counts.cpu().numpy().tobytes()).hexdigest()[:16]
    return {"filter_us": round(statistics.median(times), 2), "filter_us_min": round(min(times), 2),
            "flagged": flagged, "hash": h}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="libvqseg.so to load instead of the in-tree build")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--cases", default=",".join(CASES))
    args = ap.parse_args()
    if args.lib:
        _native.LIB_PATH = os.path.abspath(args.lib)  # before the first call loads the library
    if not torch.cuda.is_available():
        raise SystemExit("bench_filters.py measures on a GPU; none is visible")
    from vq_seg_b200 import ops
    dev = torch.device("cuda:0")
    name, power = device_info()
    result = {"device": name, "power_limit": power, "lib": _native.LIB_PATH, "cases": {}}
    for cname in args.cases.split(","):
        spec, k, algo, prepared = CASES[cname]
        for kind in ("randn", "data"):
            result["cases"][f"{cname}/{kind}"] = run_case(ops, spec, k, algo, prepared, kind, args.reps, args.warmup, dev)
            torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
