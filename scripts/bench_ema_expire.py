"""Cost of the EMA dead-code expiry on one GPU: prints one JSON line.

Workload: a training forward + backward of VectorQuantizer (K = 512) through the public module, on the config-2 map
(8 x 256 x 64 x 64) and the three config-1 latent layers (2 x 512 x 64^2, 2 x 1024 x 32^2, 2 x 2048 x 16^2).  Arms, on
identically initialised modules: no EMA, EMA, and EMA + expiry at threshold_ema_dead_code = 1.0.  The arms alternate in
rounds within one process so that drift on a shared machine hits all three alike; each round times --iters / --rounds
steps per arm with CUDA events after --warmup steps, and the inputs are cycled through enough buffers to exceed the
126 MB L2.  The device name and power limit are read in the same call.

    python scripts/bench_ema_expire.py [--iters 200] [--rounds 4] [--warmup 10]
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

SHAPES = {"c2": (8, 256, 64, 64), "c1_l3": (2, 512, 64, 64), "c1_l4": (2, 1024, 32, 32), "c1_l5": (2, 2048, 16, 16)}
K = 512
L2_BYTES = 126 << 20
ARMS = {"no_ema": None, "ema": {}, "ema_expire": {"threshold_ema_dead_code": 1.0}}


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
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ema_expire.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    name, power = device_info()
    per_round = max(1, args.iters // args.rounds)
    result = {"device": name, "power_limit": power, "iters_per_arm": per_round * args.rounds, "shapes": {}}
    for sname, (b, c, h, w) in SHAPES.items():
        g = torch.Generator(device=dev).manual_seed(42)
        init = torch.randn(K, c, generator=g, device=dev)
        nbuf = max(2, -(-2 * L2_BYTES // (b * c * h * w * 4)))
        xs = [torch.randn(b, c, h, w, generator=g, device=dev).requires_grad_(True) for _ in range(nbuf)]
        gq = torch.randn(b, c, h, w, generator=g, device=dev)
        one = torch.ones(1, device=dev)
        mods = {}
        for arm, kw in ARMS.items():
            m = V.VectorQuantizer(dim=c, num_embeddings=K).to(dev).train()
            m.codebook.embedding.weight.data.copy_(init)
            if kw is not None:
                m.enable_ema(**kw)
            mods[arm] = m

        def steps(m, n, start):
            for i in range(n):
                x = xs[(start + i) % nbuf]
                q, idx, loss, usage = m(x)
                torch.autograd.backward((q, loss), (gq, one))
                x.grad = None

        for m in mods.values():
            steps(m, args.warmup, 0)
        torch.cuda.synchronize()
        ms = {arm: 0.0 for arm in ARMS}
        for r in range(args.rounds):
            for arm, m in mods.items():
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                steps(m, per_round, r * per_round)
                e.record()
                torch.cuda.synchronize()
                ms[arm] += a.elapsed_time(e)
        us = {arm: ms[arm] * 1e3 / (per_round * args.rounds) for arm in ARMS}
        cb = mods["ema_expire"].codebook
        result["shapes"][sname] = {
            "shape": [b, c, h, w], "input_buffers": nbuf,
            **{f"{arm}_us": round(v, 2) for arm, v in us.items()},
            "ema_added_us": round(us["ema"] - us["no_ema"], 2),
            "expire_added_us": round(us["ema_expire"] - us["ema"], 2),
            "codes_expired_total": int(cb.codes_expired_total)}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
