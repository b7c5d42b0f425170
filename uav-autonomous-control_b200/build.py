"""Build libuavb.so (the C-ABI CUDA library) for sm_100a with nvcc, in-tree.

    python uav-autonomous-control_b200/build.py [--force] [--verbose]

Output: uav-autonomous-control_b200/lib/libuavb.so (git-ignored; travels to the GPU box with gpurun).
nvcc cross-compiles without a GPU; cudart is linked statically so the library loads on a GPU-less
host (where every compute entry point then fails with UAVB_ENODEVICE).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libuavb.so")
SOURCES = ["capi.cu", "minsnap_kernels.cu", "minsnap_correct.cu", "rollout_kernels.cu", "rollout_sliced.cu", "rollout_log.cu", "rollout_traj.cu", "rollout_tables.cu", "rollout_tables_log.cu", "rollout_scalar.cu", "rollout_f64.cu", "stage_kernels.cu",
           "mc_kernels.cu", "host_api.cu", "rrt_kernels.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--extended-lambda",
              "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _fingerprint() -> str:
    h = hashlib.sha256()
    names = sorted(os.listdir(CSRC)) + ["../../include/uavb.h"]
    for n in names:
        with open(os.path.join(CSRC, n), "rb") as f:
            h.update(n.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "libuavb.stamp")
    fp = _fingerprint()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == fp:
        return LIB
    objs = []
    objdir = os.path.join(ROOT, "build", "uavb")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, cmd, p in procs:
        out, _ = p.communicate()
        log.append(f"$ {' '.join(cmd)}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append(f"$ {' '.join(link)}\n{r.stdout}")
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(os.path.join(LIBDIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    with open(stamp, "w") as f:
        f.write(fp)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
