"""ctypes loader for the host-instantiated explicit-stream replay scored against per-filter truth
(tests/host_core/host_truth.cu).  TEST ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _dp

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {64: os.path.join(_HERE, "libhost_truth64.so"), 32: os.path.join(_HERE, "libhost_truth32.so")}
_SRC = [os.path.join(_HERE, "host_truth.cu")] + [
    os.path.join(_HERE, "..", "..", "quadrotor_landing_b200", "csrc", f)
    for f in ("ekf_core.cuh", "ekf_synth.cuh", "ekf_kernels.cuh", "ekf_params.hpp")
]


def _build_one(prec):
    res = subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                          "-DHT_ONLY_PREC=%d" % prec, "-Xcompiler", "-fPIC", "-shared", "-o", _LIBS[prec], _SRC[0]],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("host_truth build failed:\n" + res.stdout)


def build(force=False):
    """One library per precision, compiled in parallel (as host_core.build)."""
    todo = [pr for pr, lib_ in _LIBS.items()
            if force or not os.path.exists(lib_) or any(os.path.getmtime(s) > os.path.getmtime(lib_) for s in _SRC)]
    if todo:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=2) as ex:
            list(ex.map(_build_one, todo))
    return _LIBS[64]


_libs = {}


def lib(prec=64):
    if prec not in _libs:
        build()
        _libs[prec] = C.CDLL(_LIBS[prec])
    return _libs[prec]


def run_truth(hb, k0, n_steps, st, truth, acc, stride):
    """hb (host_core.HostBatch) advanced by hc_run_truth: the product's explicit-stream replay scored against per-filter
    truth [n_bins][16][N] into acc [32][n_bins][20]."""
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    i32 = lambda a: a.ctypes.data_as(ip)
    f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    imu, pose, stamp, tr = f64(st["imu"]), f64(st["tag_pose"]), f64(st["tag_stamp"]), f64(truth)
    step = np.ascontiguousarray(st["tag_step"], dtype=np.int32)
    valid = np.ascontiguousarray(st["tag_valid"], dtype=np.uint8)
    L = lib(hb.prec)
    L.hc_run_truth.argtypes = ([C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, dp, C.c_int64, ip, dp, dp,
                                C.POINTER(C.c_uint8), C.c_double] + [dp] * 4 + [ip] * 2 + [dp] * 3 + [ip] * 3 +
                               [C.c_int32, C.c_int32] + [dp] * 5 + [dp, dp, C.c_int32, C.c_int32])
    if hb.p.multirate_ekf:
        h = hb._history()
        hist = [_dp(h["xc"]), _dp(h["Pc"]), _dp(h["ring"]), i32(h["nh"]), i32(h["hpos"]), i32(h["hlen"]),
                h["ring_len"], h["dmax"]]
    else:
        hist = [None, None, None, None, None, None, 0, 1]
    pf = [_dp(a) for a in hb.pf] if hb.pf is not None else [None] * 5
    L.hc_run_truth(C.byref(hb.p), int(hb.prec), hb.N, int(k0), int(n_steps), _dp(imu), step.shape[0], i32(step),
                   _dp(pose), _dp(stamp), valid.ctypes.data_as(C.POINTER(C.c_uint8)), 0.0, _dp(hb.x), _dp(hb.Ppk),
                   _dp(hb.aux), _dp(hb.pend), i32(hb.flags), i32(hb.upds), *hist, *pf, _dp(tr), _dp(acc),
                   acc.shape[1], int(stride))
