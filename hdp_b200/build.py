"""Build libhdp_b200.so (hand-written sm_100a CUDA + the C ABI of include/hdp_b200.h) in-tree.

    python -m hdp_b200.build [--force]

The library is compiled for sm_100a only; there is no other back end and no CPU fallback.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libhdp_b200.so")
SOURCES = ["abi.cu", "threshold.cu", "thr_net.cu", "metric.cu", "compound.cu", "intensity.cu", "seams.cu", "measure.cu", "trend.cu", "extent.cu", "host.cu"]
HEADERS = ["common.cuh", "thr_net.cuh", "thr_net_gen.cuh", "seams.h", "metric.cuh", "intensity.h", "trend.h", "scan.cuh"]
OBJ = os.path.join(HERE, "_obj")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",                 # the f64 interpolation must stay separately rounded (bit-exact parity)
    "-Xcompiler", "-fPIC,-O2,-Wall,-fvisibility=default",
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static"]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libhdp_b200.so cannot be built")


def sources() -> list:
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _common_deps() -> list:
    return [os.path.join(CSRC, h) for h in HEADERS if os.path.exists(os.path.join(CSRC, h))] + [os.path.join(INCLUDE, "hdp_b200.h"), __file__]


def _obj_of(src: str) -> str:
    return os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")


def _stale(target: str, deps: list) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _extra_flags(verbose: bool = False) -> list:
    extra = ["-Xptxas=-v"] if verbose else []
    if os.environ.get("HDP_B200_NET_DEV"):            # kernel iterations: only four instances of k_thr_net (thr_net.cu) instead of 64
        extra.append("-DHDP_NET_DEV")
    return extra


def _cmd_of(s: str, extra: list) -> list:
    return [nvcc(), *NVCC_FLAGS, *extra, "-I", INCLUDE, "-I", CSRC, "-c", "-o", _obj_of(s), s]


def _same_flags(s: str, extra: list) -> bool:
    """An object built with other flags is stale whatever its time stamp says."""
    try:
        with open(_obj_of(s) + ".cmd") as f:
            return f.read() == " ".join(_cmd_of(s, extra))
    except OSError:
        return False


def up_to_date() -> bool:
    if _stale(LIB, sources() + _common_deps()):
        return False
    if not os.path.isdir(OBJ):                        # a shipped library without its objects (the GPU box): nothing to compare
        return True
    extra = _extra_flags()
    return all(_same_flags(s, extra) for s in sources())


def _run(cmd: list, verbose: bool) -> None:
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        print(" ".join(cmd))
        print(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)


def build(force: bool = False, verbose: bool = False) -> str:
    """One object per source (compiled in parallel, only what changed), then one link: an edit of one kernel file does
    not recompile the others."""
    if not force and up_to_date():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ, exist_ok=True)
    common = _common_deps()
    extra = _extra_flags(verbose)
    todo = [s for s in sources() if force or _stale(_obj_of(s), [s] + common) or not _same_flags(s, _extra_flags())]

    def compile_one(s):
        _run(_cmd_of(s, extra), verbose)
        with open(_obj_of(s) + ".cmd", "w") as f:
            f.write(" ".join(_cmd_of(s, _extra_flags())))

    with ThreadPoolExecutor(max(1, min(len(todo), os.cpu_count() or 1))) as pool:
        list(pool.map(compile_one, todo))
    _run([nvcc(), *LINK_FLAGS, "-o", LIB + ".tmp", *[_obj_of(s) for s in sources()]], verbose)
    os.replace(LIB + ".tmp", LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
