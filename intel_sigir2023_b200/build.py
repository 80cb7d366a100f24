"""Build libintel_b200.so (sm_100a) in-tree with nvcc.

    python -m intel_sigir2023_b200.build        # or __graft_entry__.build()

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libintel_b200.so")
SOURCES = ["batch.cu", "api_misc.cu", "api_model.cu", "attn.cu", "bert_fused.cu", "embed.cu", "eval.cu", "fuse.cu", "gemm.cu", "gemm_rows_tc.cu", "gemm_wgrad_tc.cu", "gru.cu", "gru_tc.cu", "host_pack.cu", "loss.cu", "mha.cu", "optim.cu", "rowset.cu", "trunk.cu", "trunk_tc.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
         "-I", CSRC, "-I", os.path.join(ROOT, "include")]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(ROOT, "include", "intel_b200.h"))
    objs, jobs = [], []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [os.path.join(CSRC, src)] + headers):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for out in ex.map(run, jobs):
            if verbose and out:
                print(out)
    if jobs or force or _stale(LIB, objs):
        run([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
