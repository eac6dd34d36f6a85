"""ctypes binding of libqekf.so (the C ABI of include/qekf.h).

The library is the product; this module only loads it.  There is no fallback: if the shared object is
missing the import fails loudly, and qekf_create fails with QEKF_ERR_NO_DEVICE without a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libqekf.so")
MAX_TAGS = 16

QEKF_FP64, QEKF_FP32 = 64, 32
PF_Q, PF_R, PF_R_V_CV, PF_Q_VC, PF_DELAY = range(5)

STATUS = {0: "QEKF_OK", 1: "QEKF_ERR_BAD_ARG", 2: "QEKF_ERR_CUDA", 3: "QEKF_ERR_NOT_INITIALIZED",
          4: "QEKF_ERR_UNSUPPORTED", 5: "QEKF_ERR_NO_DEVICE", 6: "QEKF_ERR_ALLOC"}


class QekfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (STATUS.get(code, code), msg))
        self.code = code


class QekfParams(C.Structure):
    """qekf_params (include/qekf.h) == the reference's public parameter members
    (quad_state_estimation/include/relative_pose_EKF.hpp:67-133)."""

    _fields_ = [
        ("update_freq", C.c_double),
        ("measurement_freq", C.c_double),
        ("measurement_delay", C.c_double),
        ("measurement_delay_max", C.c_double),
        ("dyn_measurement_delay_offset", C.c_double),
        ("Q_a", C.c_double * 3),
        ("Q_w", C.c_double * 3),
        ("Q_ab", C.c_double * 3),
        ("Q_wb", C.c_double * 3),
        ("R_r", C.c_double * 3),
        ("R_ang", C.c_double * 3),
        ("r_cov_init", C.c_double),
        ("v_cov_init", C.c_double),
        ("ang_cov_init", C.c_double),
        ("ab_cov_init", C.c_double),
        ("wb_cov_init", C.c_double),
        ("ab_static", C.c_double * 3),
        ("wb_static", C.c_double * 3),
        ("r_v_cv", C.c_double * 3),
        ("q_vc", C.c_double * 4),
        ("camera_K", C.c_double * 9),
        ("tag_in_view_margin", C.c_double),
        ("tag_widths", C.c_double * MAX_TAGS),
        ("tag_positions", C.c_double * (3 * MAX_TAGS)),
        ("small_ang_tol", C.c_double),
        ("g", C.c_double * 3),
        ("camera_width", C.c_int32),
        ("camera_height", C.c_int32),
        ("n_tags", C.c_int32),
        ("est_bias", C.c_int32),
        ("limit_measurement_freq", C.c_int32),
        ("corner_margin_enbl", C.c_int32),
        ("direct_orien_method", C.c_int32),
        ("multirate_ekf", C.c_int32),
        ("dynamic_meas_delay", C.c_int32),
        ("reserved", C.c_int32),
    ]


class QekfStreams(C.Structure):
    _fields_ = [
        ("T", C.c_int64),
        ("imu", C.c_void_p),
        ("M", C.c_int64),
        ("tag_step", C.c_void_p),
        ("tag_pose", C.c_void_p),
        ("tag_stamp", C.c_void_p),
        ("tag_valid", C.c_void_p),
        ("t_start", C.c_double),
        ("on_device", C.c_int32),
        ("reserved", C.c_int32),
    ]


class QekfScenarioSpec(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "duration_s", "hover_s", "z_start", "z_end", "sway_ax", "sway_wx", "sway_ay", "sway_wy", "sway_phase_y",
        "yaw_amp", "yaw_w", "tag_rate_hz", "tag_latency_s", "t_start")]


class QekfNoiseSpec(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("first_global_id", C.c_int64),
        ("sigma_accel", C.c_double), ("sigma_gyro", C.c_double),
        ("sigma_bias_accel", C.c_double), ("sigma_bias_gyro", C.c_double),
        ("sigma_tag_pos", C.c_double), ("sigma_tag_ang", C.c_double),
        ("dropout_k0", C.c_int32), ("dropout_k1", C.c_int32),
        ("rand_dropout_len", C.c_int32), ("rand_dropout_lo", C.c_int32), ("rand_dropout_hi", C.c_int32),
        ("edge_loss", C.c_int32),
        ("range_ref", C.c_double), ("range_exp_pos", C.c_double), ("range_exp_ang", C.c_double),
    ]


class QekfStepIO(C.Structure):
    """qekf_step_io: device pointers of one qekf_step call (NULL = not given)."""
    _fields_ = [
        ("imu", C.c_void_p),
        ("arrived", C.c_void_p),
        ("tag", C.c_void_p),
        ("x_out", C.c_void_p),
        ("cov_out", C.c_void_p),
        ("aux_out", C.c_void_p),
        ("flags_out", C.c_void_p),
    ]


class QekfSharedStreams(C.Structure):
    _fields_ = [
        ("T", C.c_int64),
        ("imu_clean", C.c_void_p),
        ("M", C.c_int64),
        ("tag_step", C.c_void_p),
        ("tag_pose_clean", C.c_void_p),
        ("tag_stamp", C.c_void_p),
        ("truth", C.c_void_p),
        ("t_start", C.c_double),
        ("on_device", C.c_int32),
        ("reserved", C.c_int32),
    ]


STAT_DIM = 20

# every symbol include/qekf.h declares; tests assert the library exports all of them
EXPORTS = [
    "qekf_default_params", "qekf_create", "qekf_destroy", "qekf_set_params", "qekf_get_params",
    "qekf_set_filter_params", "qekf_last_error_string", "qekf_num_states", "qekf_num_filters",
    "qekf_set_mapping", "qekf_set_stream", "qekf_sync", "qekf_set_imu", "qekf_set_tag", "qekf_initialize_state",
    "qekf_filter_update", "qekf_latch_tag", "qekf_tick", "qekf_step", "qekf_run", "qekf_run_with_truth", "qekf_get_state", "qekf_get_cov", "qekf_get_aux", "qekf_get_flags",
    "qekf_set_state", "qekf_prediction_step", "qekf_correction_step",
    "qekf_scenario_default", "qekf_scenario_sizes", "qekf_scenario_generate",
    "qekf_noise_default", "qekf_run_monte_carlo", "qekf_synthesize_streams", "qekf_stats_configure",
    "qekf_stats_reset", "qekf_get_stats", "qekf_copy_stats_device",
    "qekf_reset_filters", "qekf_launch_count", "qekf_measure_fma_peak", "qekf_step_counts",
    "qekf_params_from_yaml", "qekf_params_from_yaml_text",
    "qekf_export_size", "qekf_export_state", "qekf_import_state", "qekf_stats_config",
]

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libqekf.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `python -m quadrotor_landing_b200.build`. There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, dp, ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)
    L.qekf_last_error_string.restype = C.c_char_p
    L.qekf_default_params.argtypes = [C.POINTER(QekfParams)]
    L.qekf_create.argtypes = [C.POINTER(QekfParams), C.c_int64, C.c_int, C.c_int, C.POINTER(vp)]
    L.qekf_destroy.argtypes = [vp]
    L.qekf_set_params.argtypes = [vp, C.POINTER(QekfParams)]
    L.qekf_get_params.argtypes = [vp, C.POINTER(QekfParams)]
    L.qekf_set_filter_params.argtypes = [vp, C.c_int, dp]
    L.qekf_num_states.argtypes = [vp]
    L.qekf_num_filters.argtypes = [vp]
    L.qekf_num_filters.restype = C.c_int64
    L.qekf_set_mapping.argtypes = [vp, C.c_int, C.c_int]
    L.qekf_set_stream.argtypes = [vp, vp]
    L.qekf_sync.argtypes = [vp]
    L.qekf_set_imu.argtypes = [vp, dp, dp]
    L.qekf_set_tag.argtypes = [vp, dp, dp, C.c_double]
    L.qekf_initialize_state.argtypes = [vp, C.c_int]
    L.qekf_filter_update.argtypes = [vp, C.c_double]
    L.qekf_latch_tag.argtypes = [vp, dp, dp, C.c_double]
    L.qekf_tick.argtypes = [vp, dp, dp, C.c_int, dp, dp, C.c_double, C.c_double, C.c_int, dp]
    L.qekf_step.argtypes = [vp, C.c_double, C.POINTER(QekfStepIO)]
    L.qekf_run.argtypes = [vp, C.POINTER(QekfStreams), C.c_int64, C.c_int64]
    L.qekf_run_with_truth.argtypes = [vp, C.POINTER(QekfStreams), vp, C.c_int64, C.c_int64]
    L.qekf_get_state.argtypes = [vp, C.c_int64, C.c_int64, dp]
    L.qekf_get_cov.argtypes = [vp, C.c_int64, C.c_int64, dp]
    L.qekf_get_aux.argtypes = [vp, C.c_int64, C.c_int64, dp]
    L.qekf_get_flags.argtypes = [vp, C.c_int64, C.c_int64, ip]
    L.qekf_set_state.argtypes = [vp, C.c_int64, C.c_int64, dp, dp]
    L.qekf_prediction_step.argtypes = [vp, dp]
    L.qekf_correction_step.argtypes = [vp, dp]
    L.qekf_scenario_default.argtypes = [C.POINTER(QekfScenarioSpec)]
    L.qekf_scenario_sizes.argtypes = [C.POINTER(QekfParams), C.POINTER(QekfScenarioSpec),
                                      C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.qekf_scenario_generate.argtypes = [C.POINTER(QekfParams), C.POINTER(QekfScenarioSpec), dp, dp, ip, dp, dp]
    L.qekf_noise_default.argtypes = [C.POINTER(QekfNoiseSpec)]
    L.qekf_run_monte_carlo.argtypes = [vp, C.POINTER(QekfSharedStreams), C.POINTER(QekfNoiseSpec), C.c_int64, C.c_int64]
    L.qekf_synthesize_streams.argtypes = [vp, C.POINTER(QekfSharedStreams), C.POINTER(QekfNoiseSpec), C.c_int64,
                                          C.c_int64, dp, dp, C.POINTER(C.c_uint8), dp]
    L.qekf_stats_configure.argtypes = [vp, C.c_int32, C.c_int32]
    L.qekf_stats_reset.argtypes = [vp]
    L.qekf_stats_config.argtypes = [vp, ip, ip]
    L.qekf_get_stats.argtypes = [vp, dp]
    L.qekf_copy_stats_device.argtypes = [vp, vp]
    L.qekf_reset_filters.argtypes = [vp]
    L.qekf_launch_count.argtypes = [vp]
    L.qekf_launch_count.restype = C.c_int64
    L.qekf_measure_fma_peak.argtypes = [C.c_int, C.c_int, dp]
    L.qekf_step_counts.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int]
    L.qekf_export_size.argtypes = [vp]
    L.qekf_export_size.restype = C.c_int64
    L.qekf_export_state.argtypes = [vp, vp, C.c_int64]
    L.qekf_import_state.argtypes = [vp, vp, C.c_int64]
    L.qekf_params_from_yaml.argtypes = [C.c_char_p, C.POINTER(QekfParams)]
    L.qekf_params_from_yaml_text.argtypes = [C.c_char_p, C.POINTER(QekfParams)]
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise QekfError(rc, lib().qekf_last_error_string().decode("utf-8", "replace"))


def measure_fma_peak(device: int = 0, precision: int = QEKF_FP64) -> float:
    """Self-measured FMA peak of the device in TFLOP/s (FMA = 2 flops)."""
    v = C.c_double()
    check(lib().qekf_measure_fma_peak(int(device), int(precision), C.byref(v)))
    return v.value


def default_noise() -> QekfNoiseSpec:
    n = QekfNoiseSpec()
    check(lib().qekf_noise_default(C.byref(n)))
    return n


PRESET_DIR = os.path.join(HERE, "presets")


def params_from_yaml(path: str) -> QekfParams:
    """The node's parameter file (or the name of a bundled preset: "rotors_sim", "hardware_bundle") -> params,
    filled as RelativePoseEKFNode's constructor does (relative_pose_EKF_node.cpp:35-136)."""
    if not os.path.exists(path) and os.path.exists(os.path.join(PRESET_DIR, path + ".yaml")):
        path = os.path.join(PRESET_DIR, path + ".yaml")
    p = QekfParams()
    check(lib().qekf_params_from_yaml(path.encode(), C.byref(p)))
    return p


def params_from_yaml_text(text: str) -> QekfParams:
    p = QekfParams()
    check(lib().qekf_params_from_yaml_text(text.encode(), C.byref(p)))
    return p


def default_params() -> QekfParams:
    p = QekfParams()
    check(lib().qekf_default_params(C.byref(p)))
    return p
