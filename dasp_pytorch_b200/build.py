"""Build libdasp_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m dasp_pytorch_b200.build [--force] [--verbose]

The shared library lands next to this file so that it travels to the GPU box with the
repository snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libdasp_b200.so")
SOURCES = ["abi.cu", "pointwise.cu", "stereo.cu", "dynamics.cu", "biquad.cu", "reverb.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-O3,-Wall",
    "-Xptxas", "-v",
    # compress every cubin in the fatbinary: the default heuristic leaves some large ones (reverb.cu: 9 MB) uncompressed
    "-Xfatbin=-compress-all",
]


def _nvcc() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")
    return cand


def _stale(objs_srcs) -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "dasp_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if not force and not _stale(srcs):
        return LIB
    nvcc = _nvcc()
    cuda_lib = os.path.join(os.path.dirname(os.path.dirname(nvcc)), "lib64")
    objs = []
    logs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in srcs:
        obj = os.path.join(HERE, "build", os.path.basename(src) + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-I", INCLUDE, "-I", CSRC, "-c", src, "-o", obj]
        procs.append((src, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, cmd, p in procs:
        out, _ = p.communicate()
        logs.append(f"$ {' '.join(cmd)}\n{out}")
        if p.returncode != 0:
            sys.stderr.write(logs[-1])
            raise RuntimeError(f"nvcc failed on {src}")
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB, *objs, "-L", cuda_lib, "-lcufft", "-lcudart",
            "-Xlinker", f"-rpath={cuda_lib}"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    logs.append(f"$ {' '.join(link)}\n{r.stdout}")
    if r.returncode != 0:
        sys.stderr.write(logs[-1])
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "build", "build.log"), "w") as f:
        f.write("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
