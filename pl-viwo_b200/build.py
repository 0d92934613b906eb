"""Builds pl-viwo_b200/libplviwo_fe.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libplviwo_fe.so")
OBJ = os.path.join(HERE, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off"]
# (source, extra flags).  The per-feature kernels must round float expressions where the reference's SSE build
# rounds them, so no fused multiply-add contraction there.
SOURCES = [
    ("kernels_image.cu", []),
    ("kernels_fast.cu", []),
    ("kernels_track.cu", ["--fmad=false"]),
    ("kernels_lines.cu", ["--fmad=false"]),
    ("fe_context.cu", []),
    ("fe_stereo.cu", []),
    ("fe_group.cu", []),
    ("kernels_glue.cu", ["--fmad=false"]),
    ("fe_capi.cu", []),
    ("ransac.cpp", []),
    ("host_simd.cpp", []),
]
HEADERS = ["fe_kernels.h", "fe_group_dev.h", "fe_group.h", "ransac_core.h", "fe_context.h", "fe_stereo.h", "tma_bulk.h", "introsort.h", os.path.join("..", "..", "include", "plviwo_fe.h")]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for src, extra in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, os.path.splitext(src)[0] + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + ARCH + COMMON + extra + os.environ.get("PLVIWO_NVCC_FLAGS", "").split() + ["-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for out in ex.map(run, jobs):
                if verbose and out:
                    print(out)
    if force or jobs or _stale(OUT, objs):
        run([nvcc] + ARCH + ["-shared", "-o", OUT] + objs + ["-Xcompiler", "-fPIC"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
