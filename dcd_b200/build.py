"""Build libdcd_b200.so in-tree with nvcc for sm_100a (no torch headers, no JIT cache).

    python -m dcd_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdcd_b200.so")
SOURCES = ["abi.cu", "edge_solve.cu", "edge_select.cu", "dgde_locate.cu", "gmw_aggregate.cu", "gmw_transport.cu", "gmw_transport_bwd.cu", "gmw_mlp_tc.cu", "gmw_mlp_fused.cu", "gmw_mlp_bwd_tc.cu"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    inc = os.path.join(HERE, "..", "include")
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(inc, f) for f in os.listdir(inc)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False, out: str = LIB, extra=()) -> str:
    """Compile every CUDA source into one shared library; returns its path.  `out` / `extra` build a variant (e.g. the
    in-kernel trace build, extra=["-DDCD_FUSED_TRACE"]) next to the product library without touching it."""
    variant = out != LIB
    if not force and not variant and not _stale():
        return LIB
    objs = []
    procs = []
    bdir = os.path.join(HERE, "build", os.path.basename(out).replace(".so", "") if variant else "")
    os.makedirs(bdir, exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(bdir, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + list(extra) + os.environ.get("DCD_B200_NVCC_EXTRA", "").split() + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        log, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("[%s]\n%s\n" % (src, log))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libdcd_b200.so")
    cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out] + objs
    subprocess.run(cmd, check=True)
    return out


if __name__ == "__main__":
    if "--scalar" in sys.argv:      # A/B variant: scalar instead of packed FP32 in the edge solve (profiles/ab_edge.py)
        print(build_library(force=True, out=os.path.join(HERE, "libdcd_b200_scalar.so"), extra=["-DDCD_SCALAR_FP32"]))
    elif "--trace" in sys.argv:       # debug variant with the in-kernel timeline of the fused forward (profiles/trace_fused.py)
        print(build_library(force=True, out=os.path.join(HERE, "libdcd_b200_trace.so"), extra=["-DDCD_FUSED_TRACE"]))
    else:
        print(build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
