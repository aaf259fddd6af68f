"""Builds rust_bio_b200/csrc/libb200align.so in-tree with nvcc for sm_100a.

Usage: python -m rust_bio_b200.build [--force]
The K1 fill kernel is instantiated once per (lanes-per-pair, rows-per-lane) shape in its own
translation unit so the shapes compile in parallel; everything is linked into one shared library
that exports the C ABI of include/b200align.h.  cudart is linked statically so the library loads
(and reports B2A_E_NO_DEVICE) on a machine without a GPU driver.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
VARIANT = os.environ.get("B2A_VARIANT", "")  # dev knob: a differently configured build beside the default one
OBJ = os.path.join(CSRC, "build" + (("_" + VARIANT) if VARIANT else ""))
SO = os.path.join(CSRC, "libb200align%s.so" % (("_" + VARIANT) if VARIANT else ""))
SHAPES = [(1, 16), (1, 8), (1, 20), (2, 16), (2, 20), (4, 16), (8, 16), (8, 20), (32, 8), (32, 16)]
# minimum resident CTAs per SM asked of ptxas per shape (__launch_bounds__): measured choice, see DESIGN.md
MIN_BLOCKS = {(1, 16): int(os.environ.get("B2A_MINB_1_16", "3")), (8, 16): int(os.environ.get("B2A_MINB_8_16", "3")),
              (8, 20): int(os.environ.get("B2A_MINB_8_20", "1"))}  # 8x20 at 3 CTAs/SM (168 registers) measured 10 % slower
KS_DEFS = [f"-D{k}={os.environ[k]}" for k in ("B2A_KS_R", "B2A_KS_MINB") if os.environ.get(k)]  # strip-fill geometry knobs
W_8_20 = os.environ.get("B2A_W_8_20")  # warps per CTA of the 8x20 fill (default in b2a_common.cuh)
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fwrapv", "--expt-relaxed-constexpr"] + ([f"-DB2A_W_8_20={W_8_20}"] if W_8_20 else []) + KS_DEFS
HEADERS = ["b2a_common.cuh", "b2a_coop.cuh", "b2a_fill.cuh", "b2a_fill_pair16.cuh", "b2a_walk.cuh", "b2a_kernels.cuh", "b2a_plan.h", "b2a_banded.cuh", "b2a_banded_strip.cuh",
           "b2a_fill_launch.h", os.path.join("..", "..", "include", "b200align.h")]


def _stale(target: str, sources) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
    return r.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    objs = []
    for g, r in SHAPES:
        o = os.path.join(OBJ, f"fill_{g}_{r}.o")
        objs.append(o)
        src = os.path.join(CSRC, "b2a_fill_inst.cu")
        if force or _stale(o, hdrs + [src]):
            jobs.append([NVCC, *FLAGS, f"-DB2A_G={g}", f"-DB2A_R={r}", f"-DB2A_MINB={MIN_BLOCKS.get((g, r), 1)}", "-c", src, "-o", o])
    # the pair-packed 1x16 fill: 3 CTAs per SM like the int32 1x16 kernel
    p16o = os.path.join(OBJ, "fill_pair16.o")
    objs.append(p16o)
    p16src = os.path.join(CSRC, "b2a_fill_pair16.cu")
    if force or _stale(p16o, hdrs + [p16src]):
        jobs.append([NVCC, *FLAGS, f"-DB2A_MINB={MIN_BLOCKS[(1, 16)]}", "-c", p16src, "-o", p16o])
    eo = os.path.join(OBJ, "engine.o")
    objs.append(eo)
    esrc = os.path.join(CSRC, "b2a_engine.cu")
    if force or _stale(eo, hdrs + [esrc]):
        jobs.append([NVCC, *FLAGS, "-c", esrc, "-o", eo])
    mo = os.path.join(OBJ, "multi.o")
    objs.append(mo)
    msrc = os.path.join(CSRC, "b2a_multi.cu")
    if force or _stale(mo, [msrc, os.path.join(CSRC, "..", "..", "include", "b200align.h")]):
        jobs.append([NVCC, *FLAGS, "-c", msrc, "-o", mo])
    po = os.path.join(OBJ, "peak.o")
    objs.append(po)
    psrc = os.path.join(CSRC, "b2a_peak.cu")
    if force or _stale(po, [psrc]):
        jobs.append([NVCC, *FLAGS, "-c", psrc, "-o", po])
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for log in ex.map(_run, jobs):
                if verbose and log:
                    print(log, file=sys.stderr)
    if jobs or force or _stale(SO, objs):
        _run([NVCC, "-shared", "-o", SO, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-ldl"])
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
