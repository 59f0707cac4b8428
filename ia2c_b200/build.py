"""Build recipe for libia2c_b200.so (hand-written CUDA for sm_100a, C ABI in include/ia2c_b200.h).

nvcc cross-compiles here without a GPU; the .so is built IN-TREE (ia2c_b200/libia2c_b200.so) so that it
travels to the GPU box with the repo snapshot.  Run:  python -m ia2c_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import argparse
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
BUILD = os.path.join(PKG, "build")
LIB = os.path.join(PKG, "libia2c_b200.so")
SOURCES = ["runtime.cu", "org_env.cu", "belief.cu", "mlp.cu", "loss.cu", "trainer.cu", "rollout_fused.cu", "actor_pipe.cu", "debug.cu", "net_update.cu", "a2c.cu", "evaluate.cu", "history.cu", "pbt.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "--expt-relaxed-constexpr"]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _digest():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(ROOT, "include", "ia2c_b200.h")]
    for f in files:
        h.update(f.encode())
        h.update(open(f, "rb").read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(BUILD, exist_ok=True)
    stamp = os.path.join(BUILD, "digest.txt")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    if not os.path.exists(NVCC):
        raise RuntimeError(f"nvcc not found at {NVCC}; libia2c_b200.so must be built where CUDA 12.9 is installed")

    def compile_one(src):
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(_sources()))) as ex:
        objs = list(ex.map(compile_one, _sources()))
    # the link step gets the same -gencode: without it nvcc adds an (empty) default-architecture device-link stub
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB, *objs, "-lcudart"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    open(stamp, "w").write(dig)
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose))
