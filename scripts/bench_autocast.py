"""Cost of emulating the reference's autocast gather on one GPU: prints one JSON line.

Workload: a training forward + backward of VectorQuantizer (K = 512) through the public module on the config-2 map
(8 x 256 x 64 x 64).  Arms, on identically initialised modules: no autocast (exact fp32 codes), fp16 autocast (the
code rounded through fp16) and bf16 autocast (rounded through bf16).  The rounding is one conversion per gathered
element inside the gather kernel, so the arms should cost the same.  They alternate in rounds within one process so
that drift on a shared machine hits all three alike; each round times --iters / --rounds steps per arm with CUDA events
after --warmup steps, and the inputs are cycled through enough buffers to exceed the 126 MB L2.  The device name and
power limit are read in the same call.

    python scripts/bench_autocast.py [--iters 400] [--rounds 8] [--warmup 20]
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

SHAPE = (8, 256, 64, 64)
K = 512
L2_BYTES = 126 << 20
ARMS = {"fp32": None, "autocast_fp16": torch.float16, "autocast_bf16": torch.bfloat16}


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
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_autocast.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    name, power = device_info()
    per_round = max(1, args.iters // args.rounds)
    b, c, h, w = SHAPE
    g = torch.Generator(device=dev).manual_seed(42)
    init = torch.randn(K, c, generator=g, device=dev)
    nbuf = max(2, -(-2 * L2_BYTES // (b * c * h * w * 4)))
    xs = [torch.randn(b, c, h, w, generator=g, device=dev).requires_grad_(True) for _ in range(nbuf)]
    gq = torch.randn(b, c, h, w, generator=g, device=dev)
    one = torch.ones(1, device=dev)
    mods = {}
    for arm in ARMS:
        m = V.VectorQuantizer(dim=c, num_embeddings=K).to(dev).train()
        m.codebook.embedding.weight.data.copy_(init)
        mods[arm] = m

    def steps(arm, n, start):
        dtype = ARMS[arm]
        for i in range(n):
            x = xs[(start + i) % nbuf]
            with torch.autocast("cuda", dtype=dtype or torch.float16, enabled=dtype is not None):
                q, idx, loss, usage = mods[arm](x)
            torch.autograd.backward((q, loss), (gq, one))
            x.grad = None

    for arm in ARMS:
        steps(arm, args.warmup, 0)
    torch.cuda.synchronize()
    rounds = {arm: [] for arm in ARMS}
    names = list(ARMS)
    for r in range(args.rounds):
        for arm in names[r % 3:] + names[:r % 3]:           # the arms take turns at going first
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            steps(arm, per_round, r * per_round)
            e.record()
            torch.cuda.synchronize()
            rounds[arm].append(a.elapsed_time(e) * 1e3 / per_round)
    us = {arm: sum(v) / len(v) for arm, v in rounds.items()}
    result = {"device": name, "power_limit": power, "shape": list(SHAPE), "K": K, "input_buffers": nbuf,
              "iters_per_arm": per_round * args.rounds,
              **{f"{arm}_us": round(v, 2) for arm, v in us.items()},
              **{f"{arm}_round_us_min_max": [round(min(v), 2), round(max(v), 2)] for arm, v in rounds.items()},
              "bf16_minus_fp32_us": round(us["autocast_bf16"] - us["fp32"], 2),
              "bf16_minus_fp16_us": round(us["autocast_bf16"] - us["autocast_fp16"], 2)}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
