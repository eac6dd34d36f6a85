"""CPU tier of the FP32 mode: the product's per-filter code instantiated in float for the host (tests/host_core,
prec=32) against the FP64 oracle, so that a machine without a GPU catches FP32 regressions.  The GPU twin of every
test here is in test_gpu_fp32.py, which imports the comparison helpers below.

BASELINE.json promises FP32 within 1e-4 of the reference with every covariance symmetric positive-definite.  The
norm-relative bar of the other tiers (max|a - b| / max|b| over the batch) is dominated by the position and velocity
variances; on the accelerometer / gyro bias variances (1e-4 .. 1e-3 of those) it would allow percent errors.  So every
FP32 comparison goes through `assert_fp32_close`, which applies, per filter:
  state       max|x32 - x64| / max|x64| over the filter's 16 entries           <= TOL_STATE
  covariance  the same norm-relative error over the filter's n x n entries      <= TOL_COV
              |P32_ij - P64_ij| <= TOL_COV_SCALED * sqrt(P64_ii P64_jj)          (scale-aware: sees the bias blocks)
  SPD         eigvalsh of every returned FP32 covariance > 0 (float64, on the stored upper triangle)
and `assert_decisions_equal` requires the discrete decisions (state_initialized, measurement_ready,
performed_correction, filter_active, upds_since_correction and, with delayed fusion, the x_hist size) to equal the
oracle's: the frequency gate, the corner-margin gate and the delay-to-steps rounding.  If one of them flips, the
continuous comparison means nothing.

Measured worst cases behind the bars (host instantiation, 24 filters x 3,000 ticks, every (est_bias, direct) pair in
single rate, fixed and dynamic delay, per-filter sweeps): state 2.0e-6, covariance norm-relative 3.0e-5, covariance
scale-aware 4.9e-5 (in the per-filter sweeps, whose bias process noise reaches 10x the preset).  On one B200 the same
configurations at N = 400 reach 7.3e-5 scale-aware (test_gpu_fp32.py).  TOL_COV_SCALED = 2e-4 keeps a margin of 2.7
over the device and 4 over the host.  A perturbation confined to the gyro-bias block (Q_wb x 1.002 in the FP32
constants only) moves the scale-aware error to 1.1e-3 while the per-filter norm-relative error stays at 8.7e-5.
With the plain update instead of the Joseph form (QEKF_NO_JOSEPH), the host Joseph-form stress test
(test_core_host.test_fp32_joseph_form_keeps_covariance_positive) fails.
"""
import numpy as np
import pytest

import host_core as hc
import quadrotor_landing_b200 as q
from oracle import ekf_oracle as orc
from oracle import noise_np
from quadrotor_landing_b200 import scenario
from streams_np import noisy_streams, norm_rel, rotors_params
from test_core_host import rand_case
from test_multirate_host import delayed_scenario, sweep_values

TOL_STATE = 1e-4
TOL_COV = 1e-4
TOL_COV_SCALED = 2e-4
CHI2 = {1: (6.262137795043251, 27.488392863442982), 0: (2.7003894999803584, 19.02276779864163)}
U32 = float(np.finfo(np.float32).eps) / 2      # unit roundoff of float
# per-sample relative error allowed to the FP32 NEES: the derived bound (nees_tolerance) capped at 20x the worst error
# measured on the NEES sums (1.0e-6 on one B200, 5e-7 on the host), so that a moderate NEES error cannot pass
NEES_REL = 2e-5


def fp32_errors(x32, P32, x64, P64):
    """Per-filter errors of FP32 results against an FP64 reference: x [16][N], P [n][n][N]."""
    ex = np.max(np.abs(x32 - x64), axis=0) / np.max(np.abs(x64), axis=0)
    dP = np.abs(P32 - P64)
    eP = np.max(dP, axis=(0, 1)) / np.max(np.abs(P64), axis=(0, 1))
    d = np.sqrt(np.einsum("iin->in", P64))
    es = np.max(dP / (d[:, None] * d[None]), axis=(0, 1))
    return ex, eP, es


def assert_spd(P32):
    """Every covariance positive-definite, evaluated in float64 on the stored upper triangle (DESIGN.md section 7)."""
    U = np.triu(np.moveaxis(P32, 2, 0))
    S = U + np.triu(U, 1).transpose(0, 2, 1)
    lam = np.linalg.eigvalsh(S).min(axis=1)
    assert np.all(lam > 0), (np.argmin(lam), lam.min())


def assert_fp32_close(x32, P32, x64, P64, tol_state=TOL_STATE, tol_cov=TOL_COV, tol_scaled=TOL_COV_SCALED):
    """The FP32 bars of this module, per filter; returns the worst (state, covariance, scale-aware covariance)."""
    ex, eP, es = fp32_errors(x32, P32, x64, P64)
    assert ex.max() <= tol_state, ("state", int(np.argmax(ex)), ex.max())
    assert eP.max() <= tol_cov, ("covariance", int(np.argmax(eP)), eP.max())
    assert es.max() <= tol_scaled, ("scale-aware covariance", int(np.argmax(es)), es.max())
    assert_spd(P32)
    return ex.max(), eP.max(), es.max()


def host_flags(hb):
    """A HostBatch's flags in the oracle's layout [6][N]: init, ready, corrected, active, upds, x_hist size."""
    f = hb.flags
    return np.stack([f & 1, (f >> 1) & 1, (f >> 2) & 1, (f >> 3) & 1, hb.upds, hb.history_length()]).astype(np.int32)


def assert_decisions_equal(fl32, fl64, multirate):
    assert np.array_equal(fl32[0:5], fl64[0:5])
    if multirate:
        assert np.array_equal(fl32[5], fl64[5])


def test_fp32_joseph_form_keeps_covariance_positive_conventional_model():
    """test_core_host's Joseph-form stress case (measurements 1000x sharper than the preset, priors spread over three
    decades, 300 cases) for the conventional measurement model, whose innovation covariance reaches a condition number
    of 1.3e5 here (2e3 for the direct model): every updated covariance positive-definite and within the direct model's
    bars of the oracle (max 3e-6, median 2e-7).  Measured: max 2.0e-6, median 1.1e-7.  With the refined gain evaluated
    in float (before the conventional model's gain moved to double, ekf_core.cuh correction_step) 7 of the 300 were
    indefinite and the worst error was 4.9e-5, although every float-rounded oracle posterior is SPD."""
    rng = np.random.default_rng(3)
    p = q.default_params()
    p.direct_orien_method = 0
    for i in range(3):
        p.R_r[i] *= 1e-3
        p.R_ang[i] *= 1e-3
    f = orc.Filter(orc.params_from(p))
    qvc = orc.quat_norm(np.array(list(p.q_vc)))
    errs = []
    for t in range(300):
        x, P, u = rand_case(rng, 15, 1)
        d = 10.0 ** (rng.uniform(-1.5, 1.5, 15) / 2)
        P = P * np.outer(d, d)
        qt = orc.quat_mul(x[6:10], orc.quat_exp(rng.normal(scale=0.05, size=3)))
        tag = np.concatenate([rng.normal(scale=0.5, size=3) + [0, 0, 2], orc.quat_mul(qt, qvc) * np.array([-1, -1, -1, 1.0])])
        _, Pc = f.correction_step(x, P, tag[:3], tag[3:])
        assert np.linalg.eigvalsh(Pc.astype(np.float32).astype(np.float64)).min() > 0
        _, Ph, _ = hc.correction_step(p, x, P, tag, prec=32)
        assert_spd(Ph[:, :, None])
        errs.append(norm_rel(Ph, Pc))
    assert max(errs) < 3e-6 and np.median(errs) < 2e-7


# every FP32 run configuration: (est_bias, direct) x {single rate, fixed delay, dynamic delay}, and per-filter sweeps
# in single rate and with dynamic delay
REPLAY_CASES = ([(b, d, m, 0) for b in (1, 0) for d in (1, 0) for m in ("single", "fixed", "dynamic")] +
                [(1, 1, "single", 1), (1, 0, "dynamic", 1)])
CUTS = ((0, 1003), (1003, 998), (2001, 999))


def replay_setup(est_bias, direct, mode, sweep, N, seed):
    mr, dyn = mode != "single", mode == "dynamic"
    p = rotors_params(q.default_params(), est_bias=est_bias, direct=direct, multirate=mr, dynamic_delay=dyn)
    scn = delayed_scenario(p, {"single": 0.0, "fixed": 0.030, "dynamic": 0.042}[mode])
    st = noisy_streams(scn, N, seed=seed, T=3000, dropout=(1000, 1400), random_dropout_ticks=200)
    sv = sweep_values(np.random.default_rng(9), p, N, mr) if sweep else {}
    return p, st, sv


@pytest.mark.parametrize("est_bias,direct,mode,sweep", REPLAY_CASES)
def test_fp32_replay_matches_oracle(est_bias, direct, mode, sweep):
    """3,000 ticks with a common and private dropouts, three launches with odd cut points, checked after each."""
    N = 24
    p, st, sv = replay_setup(est_bias, direct, mode, sweep, N, seed=31)
    args = (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    ob = orc.Batch(orc.params_from(p), N)
    hb = hc.HostBatch(p, N, prec=32)
    for field, v in sv.items():
        ob.set_filter_params(field, v)
        hb.set_filter_params(field, v)
    for k0, n in CUTS:
        ob.run(k0, n, *args)
        hb.run(k0, n, *args)
        assert_decisions_equal(host_flags(hb), ob.flags(), p.multirate_ekf)
        assert_fp32_close(hb.state(), hb.cov(), ob.state(), ob.cov())
    assert ob.counts()[1] > 150 * N


# ---- corner-margin gate at its boundary --------------------------------------------------------------------------

CORNER_OFFSETS = 10.0 ** np.arange(-6.0, -1.5, 0.5)     # pixels, 1e-6 .. 1e-2


def _extreme(p, r, q_ct, side):
    """min_u / max_u / min_v / max_v (side 0..3) of the tag's corners at pose (r, q_ct), the oracle's projection."""
    R = orc.quat_to_rot(q_ct)
    hw = p.tag_widths[0] / 2
    K = np.array(list(p.camera_K)).reshape(3, 3)
    uv = []
    for cx, cy in ((hw, hw), (-hw, hw), (-hw, -hw), (hw, -hw)):
        pc = R @ np.array([cx, cy, 0.0]) + r
        uv.append((K @ (pc / pc[2]))[0:2])
    uv = np.array(uv)
    return (uv[:, 0].min(), uv[:, 0].max(), uv[:, 1].min(), uv[:, 1].max())[side]


def corner_gate_poses(p, rng):
    """One tag pose per (side, +-offset): the extreme corner on side u_lo / u_hi / v_lo / v_hi projects at `offset`
    pixels inside (+) or outside (-) the margin line.  Found by bisection in double on the lateral tag position (the
    projection is monotonic in it); the other three extremes stay far inside."""
    w, h, m = p.camera_width, p.camera_height, p.tag_in_view_margin
    bounds = (w * m, w * (1 - m), h * m, h * (1 - m))
    poses, inside = [], []
    for side in range(4):
        for off in CORNER_OFFSETS:
            for sgn in (1, -1):
                q_ct = orc.quat_exp(rng.normal(scale=0.15, size=3))
                r = np.array([0.0, 0.0, rng.uniform(1.5, 3.0)])
                ax = side // 2                        # shift x to move u, y to move v: every extreme grows with it
                target = bounds[side] + (sgn if side % 2 == 0 else -sgn) * off
                lo, hi = -3 * r[2], 3 * r[2]
                for _ in range(100):
                    r[ax] = 0.5 * (lo + hi)
                    if _extreme(p, r, q_ct, side) < target:
                        lo = r[ax]
                    else:
                        hi = r[ax]
                assert abs(_extreme(p, r, q_ct, side) - target) < 1e-9
                poses.append(np.concatenate([r, q_ct]))
                inside.append(sgn > 0)
    return np.array(poses).T, np.array(inside)


def corner_gate_setup(direct, seed=3):
    p = rotors_params(q.default_params(), direct=direct)
    p.limit_measurement_freq = 0          # every arrival reaches the gate
    poses, inside = corner_gate_poses(p, np.random.default_rng(seed))
    N = poses.shape[1]
    T, steps = 40, np.array([0, 9, 18, 27], dtype=np.int32)
    imu = np.zeros((T, 6, N)); imu[:, 2] = 9.81
    imu[:, 3:6] = 0.01
    tag = np.ascontiguousarray(np.repeat(poses[None], len(steps), axis=0))
    return p, (imu, steps, tag, np.zeros(len(steps))), inside


def run_corner_gate_case(make_fp32, direct):
    """The same boundary poses arrive four times; after each arrival tick the decisions and the state must equal the
    oracle's.  Returns the per-arrival decisions of the oracle."""
    p, args, inside = corner_gate_setup(direct)
    N = args[2].shape[2]
    ob = orc.Batch(orc.params_from(p), N)
    b = make_fp32(p, N)
    decided = []
    for k0, n in ((0, 1), (1, 9), (10, 9), (19, 21)):
        ob.run(k0, n, *args)
        b.run(k0, n, *args)
        fl = ob.flags()
        assert_decisions_equal(b.flags_(), fl, False)
        assert_fp32_close(b.state(), b.cov(), ob.state(), ob.cov())
        decided.append(fl[4] == 0)
    # the oracle's decisions are the geometric ones: accepted exactly when the extreme corner is inside the margin
    assert np.array_equal(decided[0], inside)
    return decided


class _HostFP32:
    def __init__(self, p, N):
        self.hb = hc.HostBatch(p, N, prec=32)

    def run(self, *a):
        self.hb.run(*a)

    def flags_(self):
        return host_flags(self.hb)

    def state(self):
        return self.hb.state()

    def cov(self):
        return self.hb.cov()


@pytest.mark.parametrize("direct", [1, 0])
def test_fp32_corner_gate_at_the_boundary_matches_oracle(direct):
    """Tag poses whose extreme corner projects 1e-6 .. 1e-2 px inside or outside u_lo / u_hi / v_lo / v_hi.  Float
    rounding of the projection is ~1e-4 px at 752 px, so a gate evaluated in float flips the smallest offsets; the
    gate is evaluated in double on the double tag pose, whatever the filter's arithmetic type."""
    run_corner_gate_case(_HostFP32, direct)


# ---- Monte-Carlo statistics -------------------------------------------------------------------------------------

def mc_noise(first=0):
    n = q.default_noise()
    n.first_global_id = first
    n.dropout_k0, n.dropout_k1 = 600, 800
    n.rand_dropout_len, n.rand_dropout_lo, n.rand_dropout_hi = 150, 100, 1200
    return n


def nees_tolerance(P):
    """Per-sample bound on the relative error of the FP32 NEES (P [n][n][N] in float64).  The NEES is a block
    elimination in float whose relative error grows with the condition number kappa of the correlation matrix
    (the diagonal scaling costs nothing); 4 n (kappa + 1) u is the first-order bound of a backward-stable solve
    plus the float error vector.  Returns (per-sample relative bound, max kappa)."""
    d = np.sqrt(np.einsum("iin->in", P))
    kappa = np.linalg.cond(np.moveaxis(P / (d[:, None] * d[None]), 2, 0))
    return 4 * P.shape[0] * (kappa + 1) * U32, float(kappa.max())


def square_sum_tolerance(e, truth_row, bias, n):
    """Bound on the error of the float64 sums of e_c^2 when e is computed in float: e_c = (float)truth_c - x_c errs
    by u (|truth_c| + |e_c|) (rounding of the truth or the true bias, then of the difference); the attitude error (float quaternion
    product, normalisation, log) by 8 u.  |d(e^2)| <= 2 |e| delta + delta^2, summed over the samples, times 2."""
    t = np.zeros_like(e)
    t[0:6] = np.abs(truth_row[0:6, None])
    t[9:15] = np.abs(bias[:, :]) if n == 15 else 0.0
    delta = U32 * (t + np.abs(e))
    delta[6:9] = 8 * U32
    return 2 * (2 * np.abs(e) * delta + delta ** 2).sum(axis=1)


def stats_reference(x, P, truth_row, bias, n, est_bias):
    """float64 statistics of one bin from the given states [20], the tolerance of each entry [20] (entry 17: the
    number of samples whose chi-square decision the FP32 NEES error can flip) and the NEES bound's max kappa."""
    e, nees = noise_np.error_stats(x, P, truth_row, bias, n)
    lo, hi = CHI2[est_bias]
    rel, kappa = nees_tolerance(P)
    rel = np.minimum(rel, NEES_REL)
    ref = np.zeros(20)
    ref[0:n] = (e ** 2).sum(axis=1)
    ref[15], ref[16] = nees.sum(), x.shape[1]
    ref[17] = np.sum((nees >= lo) & (nees <= hi))
    ref[19] = (e[0:3] ** 2).sum()
    tol = np.zeros(20)
    tol[0:n] = square_sum_tolerance(e, truth_row, bias, n)
    tol[19] = tol[0:3].sum()
    tol[15] = (rel * nees).sum()
    tol[17] = np.sum((np.abs(nees - lo) <= rel * nees) | (np.abs(nees - hi) <= rel * nees))
    return ref, tol, kappa


def assert_stats_close(stats, ref, tol):
    """[16] samples and [18] failures exact; [17] equal but for the samples within the NEES error of a chi-square
    bound; the sums [0:16] and [19] within their derived bounds."""
    assert np.array_equal(stats[:, 16], ref[:, 16])
    assert np.all(stats[:, 18] == 0)
    assert np.all(np.abs(stats - ref) <= tol), np.argwhere(np.abs(stats - ref) > tol)


@pytest.mark.parametrize("est_bias,direct", [(1, 1), (0, 0)])
def test_fp32_monte_carlo_statistics_match_float64_evaluation(est_bias, direct):
    """Single-rate Monte-Carlo launches in `stride`-tick chunks; after each chunk the float64 statistics of the
    handle's OWN FP32 states (noise_np.error_stats) against the sums the FP32 code accumulated: this isolates the
    FP32 NEES and error arithmetic from the trajectory's drift."""
    p = rotors_params(q.default_params(), est_bias=est_bias, direct=direct)
    spec = scenario.default_spec()
    spec.duration_s, spec.hover_s = 8.0, 2.0
    scn = scenario.generate(p, spec)
    noise = mc_noise(first=1000)
    N, stride = 32, 400
    nb = scn.T // stride
    n = 15 if est_bias else 9
    hb = hc.HostBatch(p, N, prec=32)
    acc = np.zeros((32, nb, 20))
    bias = hc.synthesize(scn, noise, 0, N)["bias"]
    ref, tol = np.zeros((nb, 20)), np.zeros((nb, 20))
    for k in range(nb):
        hb.run_mc(scn, noise, k * stride, stride, acc, stride)
        ref[k], tol[k], _ = stats_reference(hb.state(), hb.cov(), scn.truth[(k + 1) * stride], bias, n, est_bias)
    assert_stats_close(acc.sum(axis=0), ref, tol)
    assert ref[:, 16].sum() > 0
