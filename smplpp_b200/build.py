"""Builds smplpp_b200/libsmplpp_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch headers)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsmplpp_b200.so")
SOURCES = ["model.cu", "forward.cu", "skin_tc3.cu", "lbs_tma.cu", "lbs_tc.cu", "host_pipe.cu", "vposer.cu", "vposer_tc.cu", "ik.cu", "ik_solve_mma.cu", "ik_poseblend_tc.cu", "ik2.cu", "ik_host.cu", "task_forward.cu", "closest.cu", "sweep.cu", "io.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-Xcompiler", "-O3"]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False) -> str:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "smplpp_b200.h"))
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs, procs = [], []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== nvcc %s ==\n%s\n" % (s, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(LIB, objs):
        subprocess.check_call([nvcc, "-shared", "-o", LIB] + objs + ["-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
