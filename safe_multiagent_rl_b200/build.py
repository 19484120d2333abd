"""Build libsmarl.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m safe_multiagent_rl_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  An object is rebuilt only when its own source or some header
is newer, so code that several sources share lives in headers (.cuh): a source never includes
another .cu file (tests/test_no_cu_includes.py checks this).  The library lands in
safe_multiagent_rl_b200/_lib/libsmarl.so (git-ignored).

A heavy source (32 agent-count instantiations per kernel) is compiled as several translation units in parallel, once
per -DSMARL_TU=k.  Its `#if SMARL_TU_IS(k)` guards say what each unit holds, and its unit count is 1 + the largest k
it names (1 for a source that names none).  The library is linked with --no-undefined, so a unit or an explicit
instantiation that goes missing fails here rather than when the library is loaded.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG), "include")
OUT_DIR = os.path.join(PKG, "_lib")
OBJ_DIR = os.path.join(OUT_DIR, "obj")
LIB_PATH = os.path.join(OUT_DIR, "libsmarl.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
          "-I", INCLUDE]
# Per-file extras.  collision.cu restates the reference's float64 arithmetic operation by
# operation, so the compiler must not contract a*b+c into an FMA there.
EXTRA = {"collision.cu": ["-fmad=false"], "collision_coop.cu": ["-fmad=false"], "collision_policy.cu": ["-fmad=false"],
         "coverage_float.cu": ["-fmad=false"], "coverage_float_policy.cu": ["-fmad=false"],
         "coverage_discretized_policy.cu": ["-fmad=false"]}
TU_INDEX = re.compile(r"\bSMARL_TU_IS\((\d+)\)")


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libsmarl.so cannot be built")
    return nvcc


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def tu_count(src: str) -> int:
    """Translation units of csrc/<src>: 1 + the largest k it names in SMARL_TU_IS(k), or 1."""
    with open(os.path.join(CSRC, src)) as f:
        return 1 + max((int(k) for k in TU_INDEX.findall(f.read())), default=0)


def _headers_mtime() -> float:
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs += [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    return max(os.path.getmtime(h) for h in hs)


def build(force: bool = False, verbose: bool = False) -> str:
    hm = _headers_mtime()
    newest = max([hm] + [os.path.getmtime(os.path.join(CSRC, f)) for f in sources()])
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= newest:
        return LIB_PATH            # up to date (e.g. the prebuilt library shipped to the GPU box without objects)
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    jobs = []
    objs = []
    for src in sources():
        s = os.path.join(CSRC, src)
        n_tu = tu_count(src)
        for tu in range(n_tu):
            o = os.path.join(OBJ_DIR, src[:-3] + (f".tu{tu}" if n_tu > 1 else "") + ".o")
            objs.append(o)
            if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hm):
                cmd = [nvcc, *ARCH, *COMMON, *EXTRA.get(src, []), "-c", s, "-o", o]
                if n_tu > 1:
                    cmd.insert(1, f"-DSMARL_TU={tu}")
                if verbose:
                    cmd.insert(1, "-Xptxas=-v")
                jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        for cmd, r in ex.map(run, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {cmd[-3]}: " + r.stderr[-2000:])
    if jobs or not os.path.exists(LIB_PATH):
        cmd = [nvcc, *ARCH, "-shared", "-Xlinker", "--no-undefined", "-o", LIB_PATH, *objs, "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link of libsmarl.so failed")
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
