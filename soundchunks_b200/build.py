"""Build libgsc_cuda.so in-tree with nvcc for sm_100a (no JIT cache, the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libgsc_cuda.so")
SOURCES = ["gsc_api.cu"]
DEPS = ["gsc_api.cu", "gsc_kernels.cuh", "gsc_online.cuh", "gsc_kdtree.cuh", "gsc_device.cuh", os.path.join("..", "..", "include", "gsc_cuda.h")]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build_variant(out: str, maxrreg: int, checks: bool = False) -> list:
    """Debug build with a register cap (tools/spill_probe.py): the online k-means shapes then spill on purpose, to
    show that the results do not depend on the register allocation.  Returns the spilling k_online shapes."""
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
           "-fmad=false", "-Xcompiler", "-fPIC,-O2,-fvisibility=default", "-shared", "-o", out,
           "-Xptxas", "-v"]
    cmd += [f"-DGSC_ONLINE_MAXNREG={maxrreg}"] if maxrreg else []
    cmd += ["-DGSC_ONLINE_CHECKS"] if checks else []
    cmd += [os.path.join(CSRC, s) for s in SOURCES] + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building " + out)
    return online_spills(r.stdout + r.stderr)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return SO
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
           "-fmad=false", "-Xcompiler", "-fPIC,-O2,-fvisibility=default", "-shared", "-o", SO]
    cmd += ["-Xptxas", "-v"]
    cmd += [os.path.join(CSRC, s) for s in SOURCES]
    cmd += ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building libgsc_cuda.so")
    spilled = online_spills(r.stdout + r.stderr)
    if spilled:
        os.remove(SO)
        raise RuntimeError("k_online variants with register spills (the dispatch in gsc_api.cu must only use "
                           "spill-free shapes): " + ", ".join(spilled))
    return SO


def online_spills(ptxas_log: str) -> list:
    """Names of k_online instantiations that ptxas compiled with spill stores.

    The online k-means kernel sits at the 255-register limit.  Round 1 reported that a spilling build of its largest
    shape gave different results; round 2 could not reproduce that (147 of 147 forced-spill runs bit-identical,
    profiles/r2_spill_probe.md, DESIGN.md section 2.1), so spills are a PERFORMANCE matter: local-memory traffic in
    the innermost loops of a latency-bound kernel.  A spilling shape is still treated as a build error so that a
    compiler update cannot slow the dispatched shapes down unnoticed."""
    bad, cur = [], None
    for line in ptxas_log.splitlines():
        if "Compiling entry function" in line:
            cur = line.split("'")[1] if "'" in line else None
        elif cur and "k_online" in cur and "spill stores" in line:
            n = int(line.split("bytes stack frame,")[1].split("bytes spill stores")[0])
            if n > 0:
                bad.append(cur)
    return bad


def build_host(force: bool = False) -> str:
    """libgsc_host.so + gsc_encode / gsc_decode (host/Makefile, g++ only)."""
    host = os.path.join(os.path.dirname(HERE), "host")
    out = os.path.join(host, "_build", "libgsc_host.so")
    build(force=False)
    r = subprocess.run(["make", "-C", host, "-s"] + (["-B"] if force else []), capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("building the host library failed")
    return out


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
    print(build_host(force=True))
