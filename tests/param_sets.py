"""Named, seeded parameter sets beyond the rotors preset, shared by the CPU tier (test_params_space_host.py) and the GPU
tier (test_gpu_params_space.py).

The rotors preset hides whole classes of indexing and scheduling mistakes: its per-axis constants are isotropic or zero,
it runs one rate ratio (200 Hz updates, 30 Hz gate and tags, upd_per_meas = 7) and one single-tag camera.  Each set here
moves one of those axes and keeps the tag in view for most of the scenario:

  aniso      rotors geometry with three distinct components in every per-axis constant (Q_*, R_*, ab_static,
             wb_static, g, r_v_cv), distinct initial variances per block, q_vc a few degrees off the preset and a camera
             with fx != fy and an off-centre principal point
  gate1      100 Hz update, 100 Hz gate (upd_per_meas = 1), 50 Hz tags
  slow_gate  400 Hz update, 25 Hz gate (upd_per_meas = 16), 20 Hz tags, fixed delay 47.5 ms (19 ticks), a capture
             latency that is not a whole number of ticks
  stale20    200 Hz, 20 Hz gate (upd_per_meas = 10), 30 Hz tags: a latched detection is overwritten before the gate opens
  stale50    200 Hz, 50 Hz gate (upd_per_meas = 4), 30 Hz tags: the gate waits for arrivals
  clamp      250 Hz, dynamic delay whose offset and latency exceed measurement_delay_max (0.1 s): the clamp and the
             largest ring
  bundle     the 13-tag hardware bundle at 200 Hz, margin 0.05, on a low descent that takes the big tags (and at the
             sides of the sway the centre tag) out of the image while other tags stay in

Every delay is kept at least 0.2 tick away from a half tick: the delay-to-steps rounding at exactly half a tick is
implementation-defined in the reference too."""
import numpy as np

from quadrotor_landing_b200 import scenario
from streams_np import noisy_streams, q_exp, q_mul, rotors_params

MODES = {"single": (False, False), "fixed": (True, False), "dynamic": (True, True)}

# update_freq, measurement_freq, tag rate (Hz); fixed delay, delay cap, dynamic offset (s); capture latency in whole
# ticks (s) and the extra sub-tick part of the stamps (ticks); scenario length and hover (s); delay modes
SETS = {
    "aniso":     dict(f=200.0, gate=30.0, tags=30.0, delay=0.030, dmax=0.200, off=0.005, lat=0.035, frac=0.3,
                      secs=(10.0, 2.0), modes=("single", "fixed", "dynamic")),
    "gate1":     dict(f=100.0, gate=100.0, tags=50.0, delay=0.030, dmax=0.200, off=0.002, lat=0.030, frac=0.0,
                      secs=(20.0, 3.0), modes=("single", "fixed", "dynamic")),
    "slow_gate": dict(f=400.0, gate=25.0, tags=20.0, delay=0.0475, dmax=0.200, off=0.0, lat=0.045, frac=0.3,
                      secs=(6.0, 1.5), modes=("single", "fixed", "dynamic")),
    "stale20":   dict(f=200.0, gate=20.0, tags=30.0, delay=0.030, dmax=0.200, off=0.005, lat=0.040, frac=0.25,
                      secs=(10.0, 2.0), modes=("single", "fixed", "dynamic")),
    "stale50":   dict(f=200.0, gate=50.0, tags=30.0, delay=0.030, dmax=0.200, off=0.005, lat=0.040, frac=0.25,
                      secs=(10.0, 2.0), modes=("single", "fixed", "dynamic")),
    "clamp":     dict(f=250.0, gate=50.0, tags=25.0, delay=0.060, dmax=0.100, off=0.030, lat=0.080, frac=0.3,
                      secs=(8.0, 2.0), modes=("fixed", "dynamic")),
    "bundle":    dict(f=200.0, gate=100.0, tags=30.0, delay=0.150, dmax=0.350, off=0.085, lat=0.060, frac=0.3,
                      secs=(10.0, 2.0), modes=("single", "fixed", "dynamic")),
}
NAMES = tuple(SETS)
# (set, mode) pairs, every set in every delay mode it supports
CASES = [(s, m) for s in NAMES for m in SETS[s]["modes"]]


def _aniso(p):
    """Three distinct components in every per-axis constant of p, in place."""
    for i, (fa, fw, fab, fwb) in enumerate(((1.0, 0.7, 1.3, 0.8), (1.6, 1.2, 0.6, 1.5), (0.6, 1.9, 2.1, 0.5))):
        p.Q_a[i] *= fa; p.Q_w[i] *= fw; p.Q_ab[i] *= fab; p.Q_wb[i] *= fwb
    p.R_r[0], p.R_r[1], p.R_r[2] = 0.011, 0.019, 0.027
    p.R_ang[0], p.R_ang[1], p.R_ang[2] = 0.0012, 0.0021, 0.033
    p.r_cov_init, p.v_cov_init, p.ang_cov_init, p.ab_cov_init, p.wb_cov_init = 0.13, 0.07, 0.17, 0.45, 0.08
    p.ab_static[0], p.ab_static[1], p.ab_static[2] = 0.21, -0.09, 0.04
    p.wb_static[0], p.wb_static[1], p.wb_static[2] = -0.018, 0.011, 0.006
    p.g[0], p.g[1], p.g[2] = 0.04, -0.025, -9.805
    p.r_v_cv[0], p.r_v_cv[1], p.r_v_cv[2] = 0.031, -0.017, -0.068
    qv = q_mul(np.array(list(p.q_vc)), q_exp(np.deg2rad(np.array([2.0, -3.0, 4.0]))))
    for i in range(4):
        p.q_vc[i] = float(qv[i])
    K = (250.3, 0.0, 361.2, 0.0, 233.9, 251.7, 0.0, 0.0, 1.0)
    for i in range(9):
        p.camera_K[i] = K[i]


def make(name, P, mode="single", est_bias=1, direct=1):
    """(params, scenario) of set `name` in delay mode `mode`; P: a fresh params struct (the product's or the oracle's
    layout).  The scenario's tag stamps carry the set's sub-tick latency."""
    s = SETS[name]
    mr, dyn = MODES[mode]
    assert mode in s["modes"], (name, mode)
    if name == "bundle":
        from quadrotor_landing_b200 import _native as nat
        src = nat.params_from_yaml("hardware_bundle")
        import ctypes as C
        C.memmove(C.addressof(P), C.addressof(src), C.sizeof(P))
        p = P
        p.limit_measurement_freq, p.corner_margin_enbl = 1, 1
        p.tag_in_view_margin = 0.05
        p.est_bias, p.direct_orien_method = int(est_bias), int(direct)
        p.multirate_ekf, p.dynamic_meas_delay = int(mr), int(dyn)
    else:
        p = rotors_params(P, est_bias=est_bias, direct=direct, multirate=mr, dynamic_delay=dyn)
    p.update_freq, p.measurement_freq = s["f"], s["gate"]
    p.measurement_delay, p.measurement_delay_max, p.dyn_measurement_delay_offset = s["delay"], s["dmax"], s["off"]
    if name == "aniso":
        _aniso(p)
    spec = scenario.default_spec()
    spec.duration_s, spec.hover_s = s["secs"]
    spec.tag_rate_hz = s["tags"]
    spec.tag_latency_s = s["lat"] if mr else 0.0
    if name == "bundle":
        spec.z_start, spec.z_end = 1.6, 0.35
        spec.sway_ax, spec.sway_ay, spec.sway_wx, spec.sway_wy = 0.22, 0.16, 0.9, 0.7
    scn = scenario.generate(p, spec)
    if mr:
        scn.tag_stamp -= s["frac"] / p.update_freq
    return p, scn


def upd_per_meas(p):
    return int(np.ceil(p.update_freq / p.measurement_freq))


def streams(scn, N, seed, T, ring_len):
    """Explicit per-filter streams with a common dropout and a private dropout per filter, both longer than the
    delayed-fusion ring (the ring-full path)."""
    d = ring_len + 7
    return noisy_streams(scn, N, seed=seed, T=T, dropout=(T // 3, T // 3 + d), random_dropout_ticks=d)


def cuts(T):
    """Chunk borders at odd ticks (through pending measurements and through the history)."""
    a, b = T // 3 + 1, (2 * T) // 3 - 2
    return ((0, 1), (1, a - 1), (a, 3), (a + 3, b - a - 3), (b, T - b))


# ---- what the sets are for: asserted by every test built on them ----------------------------------------------------

def corner_ok(p, pose):
    """Per-tag corner-margin decision (relative_pose_EKF.cpp:156-186) of tag poses [7][K], numpy float64: [n_tags][K]."""
    x, y, z, w = pose[3:7]
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    K = np.array(list(p.camera_K)).reshape(3, 3)
    m = p.tag_in_view_margin
    out = []
    for i in range(p.n_tags):
        hw, px, py = p.tag_widths[i] / 2, p.tag_positions[3 * i], p.tag_positions[3 * i + 1]
        u, v = [], []
        for cx, cy in ((hw, hw), (-hw, hw), (-hw, -hw), (hw, -hw)):
            pc = R[:, 0] * (cx + px) + R[:, 1] * (cy + py) + pose[0:3]
            uvw = K @ (pc / pc[2])
            u.append(uvw[0]); v.append(uvw[1])
        u, v = np.array(u), np.array(v)
        out.append((u.min(0) > p.camera_width * m) & (v.min(0) > p.camera_height * m) &
                   (u.max(0) < p.camera_width * (1 - m)) & (v.max(0) < p.camera_height * (1 - m)))
    return np.array(out)


def assert_exercised(name, p, st, T, ncorr, aux=None, ring_len=None):
    """Non-vacuity of one replay of set `name`: st the streams it replayed over T ticks, ncorr the oracle's corrections,
    aux the oracle's aux at the end, ring_len the delayed-fusion ring."""
    N = st["tag_valid"].shape[1]
    sel = st["tag_step"] < T
    arrivals = int(st["tag_valid"][sel].sum())
    gates = N * T / upd_per_meas(p)
    assert ncorr > 0.6 * min(arrivals, gates), (ncorr, arrivals, gates)
    rate = p.update_freq / SETS[name]["tags"]           # ticks between arrivals
    upm = upd_per_meas(p)
    assert upm == {"aniso": 7, "gate1": 1, "slow_gate": 16, "stale20": 10, "stale50": 4, "clamp": 5, "bundle": 2}[name]
    if name == "stale20":
        assert rate < upm and ncorr < 0.8 * arrivals     # detections overwritten before the gate opens
    if name in ("stale50", "gate1"):
        assert rate > upm and ncorr > 0.9 * arrivals     # the gate waits for arrivals
    if ring_len is not None and p.multirate_ekf:
        # some filter goes longer than the ring without a detection: the ring-full path
        steps = st["tag_step"][sel]
        gaps = [np.diff(steps[st["tag_valid"][sel][:, i] != 0]).max() for i in range(N)]
        assert max(gaps) > ring_len
        if name == "slow_gate" and not p.dynamic_meas_delay:
            assert ring_len == 19 + 2 * 16 + 1
    if name == "clamp" and p.dynamic_meas_delay:
        assert aux is not None and np.max(aux[10]) == p.measurement_delay_max
    if name == "bundle":
        v = st["tag_valid"][sel] != 0
        ok = corner_ok(p, np.moveaxis(st["tag_pose"][sel], 1, 0).reshape(7, -1)).reshape(p.n_tags, *v.shape)
        accepted = ok.any(axis=0) & v
        assert (v & ~ok.any(axis=0)).sum() > 0.01 * v.sum()      # the gate rejects
        assert accepted.sum() > 0.3 * v.sum()                    # and accepts
        assert (v & ~ok[0] & ok[1:].any(axis=0)).sum() > 0       # the centre tag alone would reject some
        assert ncorr < arrivals        # the gate waits for arrivals (upd_per_meas 2), so every miss is a rejection
