"""Build libquadsim.so in-tree with nvcc for sm_100a (cross-compiles on a box without a GPU).

    python -m rl_aerial_manipulator_b200._build        (or __graft_entry__.build())

Objects go to rl-aerial-manipulator_b200/_obj/, the library to rl-aerial-manipulator_b200/lib/libquadsim.so.
Both are git-ignored but travel with the gpurun snapshot.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIBDIR = os.path.join(HERE, "lib")
# QS_NVCC_DEFINES="-DQS_RO_TRACE=1 ..." + QS_LIB_TAG=foo build a trace variant lib/libquadsim_foo.so (the clock64 phase traces of
# tools/rollout_trace.py and tools/policy_trace3.py; load it with QS_LIB_PATH).  The product build uses neither.
TAG = os.environ.get("QS_LIB_TAG", "")
DEFINES = os.environ.get("QS_NVCC_DEFINES", "").split()
OBJ = OBJ + ("_" + TAG if TAG else "")
LIB = os.path.join(LIBDIR, f"libquadsim{'_' + TAG if TAG else ''}.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-I", INCLUDE]
# per-file extra flags: the LSODA parity kernel must not contract a*b+c (see csrc/qs_step_lsoda.cu)
EXTRA = {"qs_step_lsoda.cu": ["-fmad=false"]}


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libquadsim needs the CUDA 12.9 toolkit to build")
    return exe


def sources() -> list[str]:
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _newest_header() -> float:
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(INCLUDE, "quadsim.h"))
    hs.append(os.path.abspath(__file__))
    return max(os.path.getmtime(h) for h in hs)


def _compile(src: str, verbose: bool) -> str:
    obj = os.path.join(OBJ, src[:-3] + ".o")
    cmd = [nvcc(), *ARCH, *COMMON, *DEFINES, *EXTRA.get(src, []), "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    with open(obj + ".log", "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{log}")
    if verbose:
        print(f"[build] {src} ok")
    return obj


def build(force: bool = False, verbose: bool = True) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    srcs = sources()
    hdr_time = _newest_header()
    todo = []
    for s in srcs:
        obj = os.path.join(OBJ, s[:-3] + ".o")
        stale = force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(os.path.join(CSRC, s)), hdr_time)
        if stale:
            todo.append(s)
    if todo:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(todo))) as ex:
            list(ex.map(lambda s: _compile(s, verbose), todo))
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in srcs]
    if todo or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        cmd = [nvcc(), *ARCH, "-shared", "-o", LIB, *objs, "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
        if verbose:
            print(f"[build] linked {LIB}")
    return LIB


def ptxas_report() -> str:
    """Registers / spills / smem per kernel from the last compile logs (for profiles/)."""
    out = []
    for s in sources():
        log = os.path.join(OBJ, s[:-3] + ".o.log")
        if os.path.exists(log):
            lines = open(log).read().splitlines()
            for i, ln in enumerate(lines):
                if "Compiling entry function" in ln:
                    out.append(s + ": " + ln.split("'")[1])
                    out.extend("    " + x.strip() for x in lines[i + 1:i + 3])
    return "\n".join(out)


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    if "--report" in sys.argv:
        print(ptxas_report())
