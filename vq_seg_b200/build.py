"""Builds libvqseg.so (hand-written sm_100a CUDA behind the C ABI of include/vqseg.h) in-tree.

    python -m vq_seg_b200.build            # incremental
    python -m vq_seg_b200.build --force
    python -m vq_seg_b200.build --dev      # libvqseg_dev.so: same sources with -DVQSEG_DEV (pipeline trace hooks)

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with gpurun.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvqseg.so")
DEV_LIB = os.path.join(HERE, "libvqseg_dev.so")
SOURCES = ["api.cu", "exact.cu", "assign_tc.cu", "assign_tc2.cu", "assign_tc3.cu", "assign_tc4.cu", "ops.cu", "seghead.cu", "seghead_tiled.cu"]
HEADERS = ["common.cuh", "tc_common.cuh", "kernels.cuh", "codebook_prep.cuh", "filter_epilogue.cuh", "exact_chain.cuh", os.path.join("..", "..", "include", "vqseg.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def _digest():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False, dev=False):
    LIB = DEV_LIB if dev else globals()["LIB"]
    # the stamp lives in the (git-ignored) build directory: a fresh clone always compiles
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    stamp = os.path.join(HERE, "build", os.path.basename(LIB) + ".stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".dev.o" if dev else ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *(["-DVQSEG_DEV"] if dev else []), "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    failed = None
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src}\n{out}")
        if p.returncode != 0 and failed is None:
            failed = src
    if failed:
        sys.stderr.write("\n".join(log))
        raise RuntimeError(f"nvcc failed on {failed}")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append(r.stdout)
    if r.returncode != 0:
        sys.stderr.write("\n".join(log))
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "build", "ptxas_dev.log" if dev else "ptxas.log"), "w") as fh:
        fh.write("\n".join(log))
    with open(stamp, "w") as fh:
        fh.write(dig)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, dev="--dev" in sys.argv))
