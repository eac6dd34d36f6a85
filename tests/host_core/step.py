"""ctypes loader for the host-instantiated per-tick step of qekf_step (tests/host_core/host_step.cu).  TEST ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import _dp

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {64: os.path.join(_HERE, "libhost_step64.so"), 32: os.path.join(_HERE, "libhost_step32.so")}
_SRC = [os.path.join(_HERE, "host_step.cu")] + [
    os.path.join(_HERE, "..", "..", "quadrotor_landing_b200", "csrc", f)
    for f in ("ekf_core.cuh", "ekf_synth.cuh", "ekf_kernels.cuh", "ekf_params.hpp")
]


def _build_one(prec):
    res = subprocess.run(["nvcc", "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                          "-DHS_ONLY_PREC=%d" % prec, "-Xcompiler", "-fPIC", "-shared", "-o", _LIBS[prec], _SRC[0]],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("host_step build failed:\n" + res.stdout)


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


def step(hb, t_curr, imu, arrived=None, tag=None, counts=None, outputs=True):
    """hb (host_core.HostBatch) advanced by one qekf_step: imu [6][N], arrived [N] uint8 or None, tag [8][N].
    counts: int64 array [2] that gains (predictions, corrections).  Returns the outputs (x [16][N], cov [NP][N],
    aux [11][N], flags [6][N]) or None."""
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    i32 = lambda a: a.ctypes.data_as(ip)
    f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    N = hb.N
    imu = f64(imu)
    assert imu.shape == (6, N)
    u8 = C.POINTER(C.c_uint8)
    if arrived is not None:
        arrived = np.ascontiguousarray(arrived, dtype=np.uint8)
        tag = f64(tag)
        assert arrived.shape == (N,) and tag.shape == (8, N)
    if counts is None:
        counts = np.zeros(2, dtype=np.int64)
    out = None
    if outputs:
        out = (np.zeros((16, N)), np.zeros((hb.np_, N)), np.zeros((11, N)), np.zeros((6, N), dtype=np.int32))
    L = lib(hb.prec)
    L.hc_step.argtypes = ([C.c_void_p, C.c_int, C.c_int64, C.c_double, dp, u8, dp] + [dp] * 4 + [ip] * 2 + [dp] * 3 +
                          [ip] * 3 + [C.c_int32, C.c_int32] + [dp] * 5 + [C.POINTER(C.c_int64), dp, dp, dp, ip])
    if hb.p.multirate_ekf:
        h = hb._history()
        hist = [_dp(h["xc"]), _dp(h["Pc"]), _dp(h["ring"]), i32(h["nh"]), i32(h["hpos"]), i32(h["hlen"]),
                h["ring_len"], h["dmax"]]
    else:
        hist = [None, None, None, None, None, None, 0, 1]
    pf = [_dp(a) for a in hb.pf] if hb.pf is not None else [None] * 5
    outs = [_dp(out[0]), _dp(out[1]), _dp(out[2]), i32(out[3])] if out is not None else [None] * 4
    L.hc_step(C.byref(hb.p), int(hb.prec), N, float(t_curr), _dp(imu),
              arrived.ctypes.data_as(u8) if arrived is not None else None, _dp(tag) if arrived is not None else None,
              _dp(hb.x), _dp(hb.Ppk), _dp(hb.aux), _dp(hb.pend), i32(hb.flags), i32(hb.upds), *hist, *pf,
              counts.ctypes.data_as(C.POINTER(C.c_int64)), *outs)
    return out
