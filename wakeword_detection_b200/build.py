"""In-tree build of libwwb200.so (nvcc, sm_100a only) and of the oracle's C restatement.

    python -m wakeword_detection_b200.build [--force]

The library is built next to this file so that it travels with the repository
snapshot to the GPU box; nothing is installed into site-packages.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libwwb200.so")
SOURCES = ["api.cu", "filter.cu", "crnn_simt.cu", "wavenet_simt.cu", "counts.cu", "wavenet_tc.cu", "crnn_tc.cu", "host_pipeline.cu", "context.cu",
           "stream_state.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
        [os.path.join(ROOT, "include", "wwb200.h")]
    if not force and not _stale(LIB, deps):
        return LIB
    objs = []
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")] + os.environ.get("NVCC_EXTRA", "").split()
    procs = []
    for s in srcs:
        o = os.path.join(CSRC, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        if force or _stale(o, deps):
            cmd = [_nvcc()] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed on %s" % s)
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of libwwb200.so failed")
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
