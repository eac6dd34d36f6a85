"""In-tree build of libqekf.so with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

The heavy kernel templates are split over translation units (one per real type x est_bias x
direct_orien_method) that compile in parallel; objects go to quadrotor_landing_b200/build/.
"""
from __future__ import annotations

import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "build")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libqekf.so")
BIN_DIR = os.path.join(HERE, "bin")
REPLAY = os.path.join(BIN_DIR, "qekf_replay")
ROOT = os.path.dirname(HERE)
REPLAY_SRC = [os.path.join(ROOT, "tools", "replay_driver.cpp"), os.path.join(ROOT, "include", "relative_pose_ekf_gpu.hpp"),
              os.path.join(ROOT, "include", "qekf.h")]
HEADERS = ["ekf_core.cuh", "ekf_synth.cuh", "ekf_kernels.cuh", "ekf_params.hpp", "scenario.hpp", "preset.hpp", "launch.hpp",
           "launch_coop.hpp", os.path.join("..", "..", "include", "qekf.h")]
COOP_HEADERS = ["ekf_coop.cuh", "ekf_duo.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
NVCC_FLAGS += os.environ.get("QEKF_NVCC_EXTRA", "").split()     # experiments only (e.g. -DQEKF_EXP8)


def _units():
    units = [("qekf_capi", "qekf_capi.cu", []), ("inst_misc", "inst_misc.cu", [])]
    # the cooperative kernel's units first: the benchmark variant (b1 d1 s1) is the longest compile
    for b, d, sy in ((1, 1, 1), (1, 1, 0), (1, 0, 1), (1, 0, 0), (0, 1, 1), (0, 1, 0), (0, 0, 1), (0, 0, 0)):
        for kind in ("duo", "coop"):
            units.append(("inst_%s_b%d_d%d_s%d" % (kind, b, d, sy), "inst_%s.cu" % kind,
                          ["-DQ_BIAS=%d" % b, "-DQ_DIRECT=%d" % d, "-DQ_SYNTH=%d" % sy]))
    for t in ("double", "float"):
        for b in (1, 0):
            for d in (1, 0):
                for m in (0, 1):
                    units.append(("inst_run_%s_b%d_d%d_m%d" % (t, b, d, m), "inst_run.cu",
                                  ["-DQ_T=%s" % t, "-DQ_BIAS=%d" % b, "-DQ_DIRECT=%d" % d, "-DQ_MR=%d" % m]))
                    units.append(("inst_step_%s_b%d_d%d_m%d" % (t, b, d, m), "inst_step.cu",
                                  ["-DQ_T=%s" % t, "-DQ_BIAS=%d" % b, "-DQ_DIRECT=%d" % d, "-DQ_MR=%d" % m]))
    return units


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    srcs = HEADERS + COOP_HEADERS + ["qekf_capi.cu", "inst_misc.cu", "inst_run.cu", "inst_step.cu", "inst_coop.cu",
                                      "inst_duo.cu"]
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in srcs)


def _deps(src):
    return [src] + HEADERS + (COOP_HEADERS if src in ("inst_coop.cu", "inst_duo.cu") else [])


def _compile(unit, verbose, force=False):
    name, src, defs = unit
    obj = os.path.join(OBJ_DIR, name + ".o")
    if not force and not verbose and os.path.exists(obj) and all(
            os.path.getmtime(os.path.join(CSRC, f)) <= os.path.getmtime(obj) for f in _deps(src)):
        return obj, ""          # up to date: only units whose sources changed are recompiled
    cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + defs + ["-c", os.path.join(CSRC, src), "-o", obj]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (name, res.stdout))
    return obj, res.stdout


def build_replay_driver(force: bool = False) -> str:
    """The ROS-free replay driver (C++ host code over the C ABI), linked against the in-tree libqekf.so."""
    stale = (not os.path.exists(REPLAY)) or any(os.path.getmtime(f) > os.path.getmtime(REPLAY) for f in REPLAY_SRC + [LIB])
    if force or stale:
        os.makedirs(BIN_DIR, exist_ok=True)
        cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "include"), REPLAY_SRC[0], "-L" + LIB_DIR,
               "-lqekf", "-Wl,-rpath,$ORIGIN/../lib", "-o", REPLAY]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0:
            raise RuntimeError("replay driver build failed:\n" + res.stdout)
    return REPLAY


def build(force: bool = False, verbose: bool = False) -> str:
    if not (force or is_stale()):
        build_replay_driver(force)
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(OBJ_DIR, exist_ok=True)
    with ThreadPoolExecutor(max_workers=min(10, os.cpu_count() or 4)) as ex:
        results = list(ex.map(lambda u: _compile(u, verbose, force), _units()))
    objs = [r[0] for r in results]
    if verbose:
        for r in results:
            print(r[1])
    res = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout)
    build_replay_driver(True)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
