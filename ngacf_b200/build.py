"""Builds ngacf_b200/libngacf_b200.so (the C-ABI library of include/ngacf_b200.h) with nvcc for sm_100a.

The library is built IN-TREE so that it travels to the GPU box with the source snapshot; nothing is
JIT-compiled at import time.  `python -m ngacf_b200.build` rebuilds it.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libngacf_b200.so")
SOURCES = ["util.cu", "graph_build.cu", "propagate_fwd.cu", "propagate_bwd.cu", "pruned_stage.cu", "laplacian.cu", "spgat.cu", "transform_bwd_split.cu", "transform_tc.cu", "train_misc.cu", "neg_sampling.cu", "eval_topk.cu",
           "eval_topk_tc.cu", "recommend.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; ngacf_b200 has no CPU fallback and cannot be built without it")


def _stale(objs_srcs):
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "ngacf_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if not force and not _stale(srcs):
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    flags += os.environ.get("NGACF_NVCC_EXTRA", "").split()       # debug builds only (e.g. -DNGACF_TOPK_TRACE for scripts/probe/trace_topk.py)
    procs = []
    objs = []
    for s in srcs:
        o = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(o)
        cmd = [nvcc] + flags + ["-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            print(" ".join(cmd))
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (s, out.decode(errors="replace")))
        if verbose and out:
            print(out.decode(errors="replace"))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcuda"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s" % r.stdout.decode(errors="replace"))
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
