"""Host-side mirror of the reference estimator interface over the libqekf C ABI.

`RelativePoseEKF` keeps the public names of the reference class
(quad_state_estimation/include/relative_pose_EKF.hpp:20-133 and its Python twin
quad_state_estimation/test/rel_pose_EKF_test_class.py:27-170): parameter members, `initialize_params`,
`initialize_state`, `filter_update`, and the state members the node reads after every tick
(relative_pose_EKF_node.cpp:184-281).  It is backed by a batch of one filter on the GPU.

`BatchEKF` is the product interface: N independent filters replaying whole input streams inside one
kernel launch per call.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat
from ._native import QekfNoiseSpec, QekfParams, QekfSharedStreams, QekfStreams, check


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _dp(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_double))


_VEC_FIELDS = {"Q_a": 3, "Q_w": 3, "Q_ab": 3, "Q_wb": 3, "R_r": 3, "R_ang": 3, "ab_static": 3, "wb_static": 3,
               "r_v_cv": 3, "q_vc": 4, "camera_K": 9, "g": 3}
_SCALAR_FIELDS = ["update_freq", "measurement_freq", "measurement_delay", "measurement_delay_max",
                  "dyn_measurement_delay_offset", "r_cov_init", "v_cov_init", "ang_cov_init", "ab_cov_init",
                  "wb_cov_init", "tag_in_view_margin", "small_ang_tol", "camera_width", "camera_height", "n_tags",
                  "est_bias", "limit_measurement_freq", "corner_margin_enbl", "direct_orien_method",
                  "multirate_ekf", "dynamic_meas_delay"]


class BatchEKF:
    """N independent relative-pose EKFs on one GPU (handle of include/qekf.h)."""

    def __init__(self, params: QekfParams | None = None, n_filters: int = 1, device: int = 0,
                 precision: int = nat.QEKF_FP64):
        self._L = nat.lib()
        self.params = params if params is not None else nat.default_params()
        self.N = int(n_filters)
        self._h = C.c_void_p()
        check(self._L.qekf_create(C.byref(self.params), self.N, int(device), int(precision), C.byref(self._h)))
        self.precision = precision
        self._device = int(device)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.qekf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def n(self) -> int:
        return int(self._L.qekf_num_states(self._h))

    def set_params(self, params: QekfParams):
        check(self._L.qekf_set_params(self._h, C.byref(params)))
        self.params = params

    def set_filter_params(self, field: int, values):
        v = _f64(values)
        assert v.shape[-1] == self.N
        check(self._L.qekf_set_filter_params(self._h, int(field), _dp(v)))

    def set_mapping(self, lanes_per_filter: int = 1, groups: int = 0):
        """1 = one thread per filter (default, fastest), 2 = two role-specialised warps per 32 filters, 3 = three lanes per
        filter (FP64 single-rate handles); groups: 32-filter groups per CTA."""
        nat.check(self._L.qekf_set_mapping(self._h, int(lanes_per_filter), int(groups)))

    def set_stream(self, cuda_stream: int):
        check(self._L.qekf_set_stream(self._h, C.c_void_p(int(cuda_stream))))

    def sync(self):
        check(self._L.qekf_sync(self._h))

    def reset_filters(self):
        check(self._L.qekf_reset_filters(self._h))

    def step_counts(self, reset=False):
        """(prediction_step calls, correction_step calls) executed by the fused kernels."""
        a, b = C.c_int64(), C.c_int64()
        check(self._L.qekf_step_counts(self._h, C.byref(a), C.byref(b), int(reset)))
        return a.value, b.value

    @property
    def launch_count(self) -> int:
        return int(self._L.qekf_launch_count(self._h))

    # ---- reference per-tick interface (same input for every filter) ----
    def set_imu(self, accel, gyro):
        a, w = _f64(accel), _f64(gyro)
        check(self._L.qekf_set_imu(self._h, _dp(a), _dp(w)))

    def set_tag(self, pos, quat_xyzw, stamp=0.0):
        p, q = _f64(pos), _f64(quat_xyzw)
        check(self._L.qekf_set_tag(self._h, _dp(p), _dp(q), float(stamp)))

    def initialize_state(self, reinit_bias=False):
        check(self._L.qekf_initialize_state(self._h, int(bool(reinit_bias))))

    def filter_update(self, t_curr=0.0):
        check(self._L.qekf_filter_update(self._h, float(t_curr)))

    # ---- batch replay ----
    def run(self, k0, n_steps, imu, tag_step, tag_pose, tag_stamp, tag_valid=None, t_start=0.0, truth=None):
        """Host (numpy) streams: imu [T][6][N], tag_step [M], tag_pose [M][7][N], tag_stamp [M],
        tag_valid [M][N] or None.  truth: [n_bins][16][N] per-filter true states (r v q_tv ab wb) after the sampling
        tick of each statistics bin, or None; scores the replay into the statistics of stats_configure()."""
        imu = _f64(imu)
        T = imu.shape[0]
        assert imu.shape == (T, 6, self.N), imu.shape
        tag_step = np.ascontiguousarray(tag_step, dtype=np.int32)
        M = int(tag_step.shape[0])
        tag_pose = _f64(tag_pose).reshape(M, 7, self.N)
        tag_stamp = _f64(tag_stamp).reshape(M)
        s = QekfStreams()
        s.T = T
        s.imu = imu.ctypes.data
        s.M = M
        s.tag_step = tag_step.ctypes.data if M else None
        s.tag_pose = tag_pose.ctypes.data if M else None
        s.tag_stamp = tag_stamp.ctypes.data if M else None
        if tag_valid is not None:
            tag_valid = np.ascontiguousarray(tag_valid, dtype=np.uint8)
            assert tag_valid.shape == (M, self.N)
            s.tag_valid = tag_valid.ctypes.data
        s.t_start = float(t_start)
        s.on_device = 0
        tp = None
        if truth is not None:
            truth = _f64(truth)
            assert truth.ndim == 3 and truth.shape[1:] == (16, self.N), truth.shape
            tp = truth.ctypes.data
        check(self._L.qekf_run_with_truth(self._h, C.byref(s), tp, int(k0), int(n_steps)))
        self.sync()   # the host buffers above must outlive the asynchronous copies

    def run_device(self, k0, n_steps, T, imu_ptr, M, tag_step_ptr, tag_pose_ptr, tag_stamp_ptr,
                   tag_valid_ptr=None, t_start=0.0, truth_ptr=None):
        """Device-resident streams given as raw device pointers (e.g. torch tensors' data_ptr()).  truth_ptr: device
        pointer to the [n_bins][16][N] per-filter truth of run(), or None."""
        s = QekfStreams()
        s.T, s.imu, s.M = int(T), int(imu_ptr), int(M)
        s.tag_step, s.tag_pose, s.tag_stamp = tag_step_ptr, tag_pose_ptr, tag_stamp_ptr
        s.tag_valid = tag_valid_ptr
        s.t_start = float(t_start)
        s.on_device = 1
        tp = int(truth_ptr) if truth_ptr is not None else None
        check(self._L.qekf_run_with_truth(self._h, C.byref(s), tp, int(k0), int(n_steps)))

    # ---- per-tick step with device-resident per-filter inputs and outputs (closed-loop simulation) ----
    def step(self, t_curr, imu, tag=None, arrived=None, x=None, cov=None, aux=None, flags=None):
        """One timer tick of every filter (qekf_step): for filter i, the tag callback with tag[:, i] where arrived[i] is
        nonzero, then the IMU sample imu[:, i] and filter_update(t_curr).  All arguments are contiguous torch CUDA tensors
        on this handle's device: imu [6][N] float64; tag [8][N] float64 (r_c_tc xyz, q_ct xyzw, capture stamp); arrived
        [N] uint8 or bool.  Outputs, written where given and never allocated here: x [16][N], cov [n(n+1)/2][N] (upper
        triangle of cov_pert, row by row), aux [11][N] float64, flags [6][N] int32 -- the accessors' layouts.  Returns
        (x, cov, aux, flags).

        Asynchronous on the handle's stream, with no host synchronisation, so it can be captured into a CUDA graph.  To
        order it with torch work, run it on torch's stream: set_stream(torch.cuda.current_stream().cuda_stream)."""
        import torch
        dev = torch.device("cuda", self._device)
        N = self.N

        def ptr(t, name, rows, dtypes):
            if t is None:
                return None
            if not isinstance(t, torch.Tensor) or t.device != dev:
                raise ValueError("%s must be a torch tensor on %s" % (name, dev))
            if t.dtype not in dtypes:
                raise ValueError("%s must be %s, not %s" % (name, " or ".join(str(d) for d in dtypes), t.dtype))
            shape = (N,) if rows is None else (rows, N)
            if tuple(t.shape) != shape:
                raise ValueError("%s must have shape %s, not %s" % (name, shape, tuple(t.shape)))
            if not t.is_contiguous():
                raise ValueError("%s must be contiguous" % name)
            return t.data_ptr()

        if imu is None:
            raise ValueError("imu is required")
        if arrived is not None and tag is None:
            raise ValueError("arrived given without tag")
        f64, n = (torch.float64,), self.n
        io = nat.QekfStepIO()
        io.imu = ptr(imu, "imu", 6, f64)
        io.tag = ptr(tag, "tag", 8, f64)
        io.arrived = ptr(arrived, "arrived", None, (torch.uint8, torch.bool))
        io.x_out = ptr(x, "x", 16, f64)
        io.cov_out = ptr(cov, "cov", n * (n + 1) // 2, f64)
        io.aux_out = ptr(aux, "aux", 11, f64)
        io.flags_out = ptr(flags, "flags", 6, (torch.int32,))
        check(self._L.qekf_step(self._h, float(t_curr), C.byref(io)))
        return x, cov, aux, flags

    # ---- Monte-Carlo replay: shared clean scenario + in-kernel per-filter noise ----
    def _shared(self, scn, with_truth=True):
        """scn: quadrotor_landing_b200.scenario.Scenario (host numpy arrays).  Returns the C struct and the
        arrays it points to (which must outlive the call)."""
        imu = _f64(scn.imu_clean); pose = _f64(scn.tag_pose_clean); stamp = _f64(scn.tag_stamp)
        step = np.ascontiguousarray(scn.tag_step, dtype=np.int32)
        truth = _f64(scn.truth) if (with_truth and scn.truth is not None) else None
        s = QekfSharedStreams()
        s.T, s.imu_clean, s.M = imu.shape[0], imu.ctypes.data, step.shape[0]
        s.tag_step, s.tag_pose_clean, s.tag_stamp = step.ctypes.data, pose.ctypes.data, stamp.ctypes.data
        s.truth = truth.ctypes.data if truth is not None else None
        s.t_start = float(scn.spec.t_start)
        s.on_device = 0
        return s, (imu, pose, stamp, step, truth)

    def run_monte_carlo(self, scn, noise: QekfNoiseSpec, k0=0, n_steps=None, sync=True):
        n_steps = scn.T - k0 if n_steps is None else n_steps
        s, keep = self._shared(scn)
        check(self._L.qekf_run_monte_carlo(self._h, C.byref(s), C.byref(noise), int(k0), int(n_steps)))
        if sync:
            self.sync()
        return keep

    def run_monte_carlo_device(self, shared: QekfSharedStreams, noise: QekfNoiseSpec, k0, n_steps):
        """Device-resident shared scenario (shared.on_device = 1); asynchronous on the handle's stream."""
        check(self._L.qekf_run_monte_carlo(self._h, C.byref(shared), C.byref(noise), int(k0), int(n_steps)))

    def synthesize_streams(self, scn, noise: QekfNoiseSpec, first=0, count=None):
        """The realisation of filters [first, first+count) as explicit host streams (qekf_streams layout)."""
        count = self.N - first if count is None else count
        s, keep = self._shared(scn, with_truth=False)
        T, M = s.T, s.M
        imu = np.zeros((T, 6, count)); pose = np.zeros((M, 7, count))
        valid = np.zeros((M, count), dtype=np.uint8); bias = np.zeros((6, count))
        check(self._L.qekf_synthesize_streams(self._h, C.byref(s), C.byref(noise), int(first), int(count), _dp(imu),
                                              _dp(pose), valid.ctypes.data_as(C.POINTER(C.c_uint8)), _dp(bias)))
        return dict(imu=imu, tag_step=keep[3].copy(), tag_pose=pose, tag_stamp=keep[2].copy(), tag_valid=valid, bias=bias)

    def stats_configure(self, n_bins: int, stride: int):
        check(self._L.qekf_stats_configure(self._h, int(n_bins), int(stride)))
        self._stats_bins = int(n_bins)

    def stats_reset(self):
        check(self._L.qekf_stats_reset(self._h))

    def stats(self) -> np.ndarray:
        out = np.zeros((self._stats_bins, nat.STAT_DIM))
        check(self._L.qekf_get_stats(self._h, _dp(out)))
        return out

    def copy_stats_device(self, dst_ptr: int):
        check(self._L.qekf_copy_stats_device(self._h, C.c_void_p(int(dst_ptr))))

    def stats_tensor(self):
        """The reduced statistics as a torch tensor on this handle's GPU (what a multi-GPU job all-reduces)."""
        import torch
        t = torch.zeros((self._stats_bins, nat.STAT_DIM), dtype=torch.float64, device=torch.device("cuda", self._device))
        self.copy_stats_device(t.data_ptr())
        self.sync()
        return t

    # ---- stateless steps ----
    def prediction_step(self, u):
        u = _f64(u)
        assert u.shape == (6, self.N)
        check(self._L.qekf_prediction_step(self._h, _dp(u)))

    def correction_step(self, tag_pose):
        t = _f64(tag_pose)
        assert t.shape == (7, self.N)
        check(self._L.qekf_correction_step(self._h, _dp(t)))

    # ---- accessors ----
    def state(self, first=0, count=None) -> np.ndarray:
        count = self.N - first if count is None else count
        x = np.zeros((16, count))
        check(self._L.qekf_get_state(self._h, first, count, _dp(x)))
        return x

    def cov(self, first=0, count=None) -> np.ndarray:
        count = self.N - first if count is None else count
        n = self.n
        P = np.zeros((n * n, count))
        check(self._L.qekf_get_cov(self._h, first, count, _dp(P)))
        return P.reshape(n, n, count)

    def aux(self, first=0, count=None) -> np.ndarray:
        count = self.N - first if count is None else count
        a = np.zeros((11, count))
        check(self._L.qekf_get_aux(self._h, first, count, _dp(a)))
        return a

    def flags(self, first=0, count=None) -> np.ndarray:
        count = self.N - first if count is None else count
        f = np.zeros((6, count), dtype=np.int32)
        check(self._L.qekf_get_flags(self._h, first, count, f.ctypes.data_as(C.POINTER(C.c_int32))))
        return f

    def set_state(self, x16, P, first=0):
        x = _f64(x16)
        count = x.shape[1]
        n = self.n
        Pm = _f64(P).reshape(n * n, count)
        check(self._L.qekf_set_state(self._h, first, count, _dp(x), _dp(Pm)))

    def export_state(self) -> np.ndarray:
        """Exact checkpoint (qekf_export_state): state, covariance, latched inputs, flags, counters, the delayed-fusion
        history and the statistics accumulators as one host blob."""
        n = int(self._L.qekf_export_size(self._h))
        buf = np.empty(n, dtype=np.uint8)
        check(self._L.qekf_export_state(self._h, buf.ctypes.data_as(C.c_void_p), n))
        return buf

    def import_state(self, blob):
        """Resume from an export_state() blob of a handle with the same parameters, size and precision."""
        buf = np.ascontiguousarray(blob, dtype=np.uint8)
        check(self._L.qekf_import_state(self._h, buf.ctypes.data_as(C.c_void_p), buf.size))
        nb, stride = C.c_int32(), C.c_int32()
        check(self._L.qekf_stats_config(self._h, C.byref(nb), C.byref(stride)))
        if nb.value:
            self._stats_bins = nb.value


class RelativePoseEKF:
    """The reference's single estimator, same member names, backed by a batch of one on the GPU.

    Usage follows the node (relative_pose_EKF_node.cpp:53-182): write parameter members, call
    `initialize_params()`, feed `set_imu` / `set_tag` from the sensor callbacks, call
    `filter_update(t)` from the timer, read the state members.
    """

    def __init__(self, device: int = 0, precision: int = nat.QEKF_FP64):
        object.__setattr__(self, "_params", nat.default_params())
        object.__setattr__(self, "_device", device)
        object.__setattr__(self, "_precision", precision)
        object.__setattr__(self, "_batch", BatchEKF(self._params, 1, device, precision))
        object.__setattr__(self, "apriltag_time", 0.0)

    # parameter members read/write through to the qekf_params block
    def __getattr__(self, name):
        if name in _VEC_FIELDS:
            return np.array(list(getattr(self._params, name)))
        if name in _SCALAR_FIELDS:
            return getattr(self._params, name)
        if name == "tag_widths":
            return np.array(list(self._params.tag_widths))[: self._params.n_tags]
        if name == "tag_positions":
            return np.array(list(self._params.tag_positions))[: 3 * self._params.n_tags].reshape(-1, 3).T
        raise AttributeError(name)

    def __setattr__(self, name, value):
        if name in _VEC_FIELDS:
            v = np.asarray(value, dtype=np.float64).flatten()
            assert v.size == _VEC_FIELDS[name]
            for i in range(v.size):
                getattr(self._params, name)[i] = float(v[i])
        elif name in _SCALAR_FIELDS:
            setattr(self._params, name, type(getattr(self._params, name))(value))
        elif name == "tag_widths":
            v = np.asarray(value, dtype=np.float64).flatten()
            for i in range(v.size):
                self._params.tag_widths[i] = float(v[i])
        elif name == "tag_positions":   # 3 x n_tags, as the reference's MatrixXd
            v = np.asarray(value, dtype=np.float64)
            for i in range(v.shape[1]):
                for j in range(3):
                    self._params.tag_positions[3 * i + j] = float(v[j, i])
        else:
            object.__setattr__(self, name, value)

    def initialize_params(self):
        self._batch.set_params(self._params)

    # sensor callbacks (node.cpp:144-176)
    def set_imu(self, accel, gyro):
        self._batch.set_imu(accel, gyro)

    def set_tag(self, pos, quat_xyzw, stamp=0.0):
        object.__setattr__(self, "apriltag_time", float(stamp))
        self._batch.set_tag(pos, quat_xyzw, stamp)

    def initialize_state(self, reinit_bias=False):
        self._batch.initialize_state(reinit_bias)

    def filter_update(self, t_curr=0.0):
        self._batch.filter_update(t_curr)

    # state members (read after every tick by the node, node.cpp:184-281)
    @property
    def _x(self):
        return self._batch.state()[:, 0]

    r_nom = property(lambda self: self._x[0:3])
    v_nom = property(lambda self: self._x[3:6])
    q_nom = property(lambda self: self._x[6:10])        # x, y, z, w
    ab_nom = property(lambda self: self._x[10:13])
    wb_nom = property(lambda self: self._x[13:16])
    cov_pert = property(lambda self: self._batch.cov()[:, :, 0])
    accel_rel = property(lambda self: self._batch.aux()[0:3, 0])
    r_t_vt_obs = property(lambda self: self._batch.aux()[3:6, 0])
    q_tv_obs = property(lambda self: self._batch.aux()[6:10, 0])
    measurement_delay_curr = property(lambda self: float(self._batch.aux()[10, 0]))
    state_initialized = property(lambda self: bool(self._batch.flags()[0, 0]))
    measurement_ready = property(lambda self: bool(self._batch.flags()[1, 0]))
    performed_correction = property(lambda self: bool(self._batch.flags()[2, 0]))
    filter_active = property(lambda self: bool(self._batch.flags()[3, 0]))
    upds_since_correction = property(lambda self: int(self._batch.flags()[4, 0]))
    num_states = property(lambda self: self._batch.n)

    def pose_covariance_6x6(self):
        """The 6x6 the node publishes: rows/cols {r, theta} of cov_pert, row-major (node.cpp:203-210)."""
        P = self.cov_pert
        idx = [0, 1, 2, 6, 7, 8]
        return P[np.ix_(idx, idx)].reshape(-1)
