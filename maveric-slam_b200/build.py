"""Builds libmaveric_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python maveric-slam_b200/build.py [--force]

Every .cu is compiled with -fmad=false: the bit-exact kernels must not contract
mul+add into FMA, and the PnP kernel states its FMAs explicitly (see csrc/pnp_gn.cu).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libmaveric_b200.so")
OBJ = os.path.join(HERE, "build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function",
          "-I", os.path.join(HERE, "..", "include")]
# A/B builds of a tuning constant: MV_EXTRA_NVCC="-DMV_LEAD_CTAS=2" MV_OUT=/path/variant.so python build.py
# (objects go to a directory of their own; load the variant with MV_LIB_PATH=/path/variant.so)
if os.environ.get("MV_EXTRA_NVCC"):
    COMMON += os.environ["MV_EXTRA_NVCC"].split()
if os.environ.get("MV_OUT"):
    OUT = os.path.abspath(os.environ["MV_OUT"])
    OBJ = OUT + ".obj"
SOURCES = ["api.cu", "detector.cu", "match.cu", "match_tc.cu", "ransac.cu", "pnp_gn.cu", "traj.cu", "nms.cu", "lba.cu", "bow.cu", "lcd.cu", "synth.cu", "pool.cpp"]


def _newer(src_list, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_list)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers += [os.path.join(HERE, "..", "include", f) for f in os.listdir(os.path.join(HERE, "..", "include"))]
    jobs = []
    objs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        if not os.path.exists(src):
            continue
        obj = os.path.join(OBJ, os.path.splitext(s)[0] + ".o")
        objs.append(obj)
        if force or _newer([src] + headers, obj):
            cmd = [NVCC] + ARCH + COMMON + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            if s.endswith(".cpp"):
                cmd = [NVCC, "-O2", "-std=c++17", "-Xcompiler", "-fPIC,-Wall", "-I", os.path.join(HERE, "..", "include"),
                       "-c", src, "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        return r.stderr

    with ThreadPoolExecutor(max_workers=8) as ex:
        logs = list(ex.map(run, jobs))
    if verbose:
        for l in logs:
            sys.stderr.write(l)
    if jobs or force or _newer(objs, OUT):
        # static cudart + libcuda: the library carries its runtime and loads next to
        # torch's own without symbol clashes
        run([NVCC] + ARCH + ["-shared", "-o", OUT] + objs + ["-cudart", "static"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
