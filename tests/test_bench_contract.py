"""Guard of the entry points: bench.py / __graft_entry__.py parse, the reference arm runs on the host cores and
prints ONE JSON line with the expected keys, the GPU arm refuses to run without a GPU, and both arms write the
outputs of their last timed step with --dump-outputs."""
import ast
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check_dump(out_dir, golden):
    """The dumped step ran the seed-0 C2 batch: its outputs are the reference's of golden case c2_randn."""
    arrs = {n: np.load(os.path.join(out_dir, n + ".npy")) for n in ("quantize", "embed_index", "loss", "code_usage")}
    assert all(a.dtype in (np.float32, np.float64) for a in arrs.values())
    assert sum(a.nbytes for a in arrs.values()) <= 64 << 20
    rec = golden["forward"]["c2_randn"]
    assert arrs["quantize"].shape == rec["shape"] and cases.sha(torch.from_numpy(arrs["quantize"])) == rec["q_eval_sha"]
    assert torch.equal(torch.from_numpy(arrs["embed_index"]).to(torch.int32), rec["idx"])
    assert torch.equal(torch.from_numpy(arrs["loss"]).reshape(1), rec["loss_eval"])
    assert torch.equal(torch.from_numpy(arrs["code_usage"]).reshape(()), rec["usage"])


def test_entry_scripts_parse():
    for f in ("bench.py", "__graft_entry__.py", "scripts/gpu_dev.py", "scripts/bench_layers.py"):
        ast.parse(open(os.path.join(ROOT, f)).read(), filename=f)


def test_reference_arm_prints_contract_line(tmp_path, golden):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "vq_lookup_vectors_per_sec" and d["unit"] == "vectors/s"
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0 and "workload" in d["config"]
    assert d["steps"] == 2
    _check_dump(tmp_path, golden)


def test_gpu_arm_needs_a_gpu():
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU path" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(tmp_path, golden):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    # a ring of 8 input batches: the 9th step reads slot 0 again, the seed-0 batch
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "9", "--warmup", "1", "--no-extras",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=200, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 9
    _check_dump(tmp_path, golden)
