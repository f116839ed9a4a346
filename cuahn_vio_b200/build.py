"""Build cuahn_vio_b200/lib/libuahn.so with nvcc for sm_100a (no torch dependency; static cudart)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libuahn.so")
SOURCES = ["engine.cu", "image_kernels.cu", "conv_f32.cu", "conv_bf16.cu", "conv_bf16_tma.cu", "conv_fused_front.cu", "conv_s2_first.cu", "conv_small_m.cu", "head_kernels.cu", "ekf_update.cpp", "preproc_maps.cpp", "imu_propagate.cpp", "filter_bank.cu"]
FP64_EXACT = ["filter_bank.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr", "-cudart", "static"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", f) for f in ("uahn.h", "uahn_ekf.h", "uahn_preproc.h", "uahn_filter.h")] + [__file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    extra = os.environ.get("UAHN_NVCC_EXTRA", "").split()   # e.g. -DUAHN_FF_PROFILE=1 (per-role cycle counters)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, os.path.splitext(src)[0] + ".o")
        cmd = [NVCC, *FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if src.endswith(".cpp"):
            cmd[1:1] = ["-Xcompiler", "-ffp-contract=off"]   # host double math must round like the library it restates
        if src in FP64_EXACT:
            cmd[1:1] = ["-fmad=false"]   # device fp64 filter math rounds like the host build of ekf_math.h
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [NVCC, "-shared", "-o", LIB, *objs, "-cudart", "static", "-lcuda"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
