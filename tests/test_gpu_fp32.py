"""GPU tier of the FP32 mode: every FP32 kernel variant the library ships against the FP64 oracle, through the C ABI,
with the bars of test_fp32_host.py (per-filter norm-relative state and covariance 1e-4, scale-aware covariance
TOL_COV_SCALED, every covariance SPD, the discrete decisions equal to the oracle's).

Which test reaches which FP32 instantiation (inst_run.cu: float x est_bias x direct x multirate; inst_misc.cu: step
kernels; launch_tick<float, ...>: per-tick interface):
  test_fp32_step_kernels_match_oracle          prediction / correction step kernels, all four (est_bias, direct)
  test_fp32_joseph_form_on_the_device           correction step kernel, both measurement models, stiff updates
  test_fp32_replay_matches_oracle               run_kernel<float, B, D, SYNTH=0, PF=0> single rate and delayed fusion
                                                (fixed, dynamic) for all four (B, D); PF=1 in single rate (1, 1) and
                                                delayed-dynamic (1, 0): rebuild_pf_t<float>
  test_fp32_monte_carlo_matches_explicit_path_and_statistics
                                                SYNTH=1 kernels (single rate and delayed fusion with re-synthesised
                                                history) for all four (B, D), without and with per-filter tables
                                                (PF=0 and PF=1), bit for bit against the SYNTH=0 kernels of the same
                                                PF, and against the oracle; the FP32 NEES / RMSE accumulation against
                                                a float64 evaluation
  test_fp32_per_tick_interface_matches_golden   launch_tick<float, ...>, single rate (1, 1), delayed (1, 1), (0, 1)
  test_fp32_per_tick_conventional_model_matches_oracle
                                                launch_tick<float, ...>, single rate (1, 0), delayed (1, 0)
  test_fp32_handles_ignore_the_mapping          explicit and SYNTH launches under set_mapping(2) / set_mapping(3)
  test_fp32_corner_gate_at_the_boundary_matches_oracle
                                                the corner-margin gate of the FP32 replay kernels

Measured on one B200 (NVIDIA B200, 1000 W power limit), worst per filter over the whole file: state 7.4e-6,
covariance norm-relative 4.9e-5, scale-aware 7.3e-5 (both in the per-filter sweeps), FP32 NEES within 1.0e-6 of the
float64 evaluation of the same states (per-sample allowance NEES_REL = 2e-5; correlation condition numbers up to 651).
The file runs in about 25 s.
"""
import os

import numpy as np
import pytest

import quadrotor_landing_b200 as q
from oracle import ekf_oracle as orc
from oracle import noise_np
from streams_np import norm_rel, rotors_params
from test_core_host import rand_case
from test_fp32_host import (CUTS, REPLAY_CASES, assert_decisions_equal, assert_fp32_close, assert_spd,
                            mc_noise, replay_setup, run_corner_gate_case, stats_reference)
from test_gpu_parity import rand_batch
from test_multirate_host import delayed_scenario, sweep_values

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "prototype_vectors.npz"))
FP32 = q.QEKF_FP32


def _per_case(a, b):
    """Norm-relative error of each column (filter) of a against b."""
    a, b = a.reshape(-1, a.shape[-1]), b.reshape(-1, b.shape[-1])
    return np.max(np.abs(a - b), axis=0) / np.max(np.abs(b), axis=0)


@pytest.mark.parametrize("est_bias,direct", [(1, 1), (1, 0), (0, 1), (0, 0)])
def test_fp32_step_kernels_match_oracle(est_bias, direct):
    """300 random cases (ragged last warp and CTA), the first with zero rate (small-angle branch): prediction within
    1e-5 and correction within 1e-4 of the oracle per case, on state, covariance and aux."""
    rng = np.random.default_rng(17)
    N = 300
    p = q.default_params()
    p.est_bias, p.direct_orien_method = est_bias, direct
    p.ab_static[0], p.wb_static[1] = 0.2, -0.01
    b = q.BatchEKF(p, N, precision=FP32)
    f = orc.Filter(orc.params_from(p))
    qvc = orc.quat_norm(np.array(list(p.q_vc)))
    x, P, u = rand_batch(rng, N, b.n, est_bias)
    u[3:6, 0] = x[13:16, 0] + np.array(list(p.wb_static))
    b.set_state(x, P)
    b.prediction_step(u)
    xg, Pg, ag = b.state(), b.cov(), b.aux()
    xo, Po, acc = np.zeros_like(xg), np.zeros_like(Pg), np.zeros((3, N))
    for i in range(N):
        xo[:, i], Po[:, :, i], acc[:, i] = f.prediction_step(x[:, i], P[:, :, i], u[:, i])
    assert _per_case(xg, xo).max() < 1e-5 and _per_case(Pg, Po).max() < 1e-5 and _per_case(ag[0:3], acc).max() < 1e-5
    assert_spd(Pg)
    tag = np.zeros((7, N))
    for i in range(N):
        qt = orc.quat_mul(x[6:10, i], orc.quat_exp(rng.normal(scale=0.05 if i % 2 else 1.0, size=3)))
        tag[3:7, i] = orc.quat_mul(qt, qvc) * np.array([-1, -1, -1, 1.0])
        tag[0:3, i] = rng.normal(scale=0.5, size=3) + [0, 0, 2]
    b.set_state(x, P)
    b.correction_step(tag)
    xg, Pg, ag = b.state(), b.cov(), b.aux()
    obs = np.zeros((7, N))
    for i in range(N):
        xo[:, i], Po[:, :, i] = f.correction_step(x[:, i], P[:, :, i], tag[0:3, i], tag[3:7, i])
        a = f.aux()
        obs[0:3, i], obs[3:7, i] = a["r_t_vt_obs"], a["q_tv_obs"]
    assert _per_case(xg, xo).max() < 1e-4 and _per_case(Pg, Po).max() < 1e-4
    assert _per_case(ag[3:6], obs[0:3]).max() < 1e-4 and _per_case(ag[6:10], obs[3:7]).max() < 1e-4
    assert_spd(Pg)
    b.close()


@pytest.mark.parametrize("direct", [1, 0])
def test_fp32_joseph_form_on_the_device(direct):
    """test_core_host's stress case on the device (rsqrtf / sincosf / FMA contraction): measurements 1000x sharper
    than the preset, priors spread over three decades, 300 cases.  Every updated covariance SPD and within the host
    test's bars of the oracle (max 3e-6, median 2e-7).  Measured on one B200: direct model max 1.1e-6, median 8.1e-8;
    conventional model max 3.95e-6, median 1.1e-7 (host: 2.0e-6, 1.1e-7), so its max bar is 5e-6 on the device: its
    gain comes from double, and what remains is the float subtraction P - K B^T, whose terms |K| |B| are larger than the
    direct model's (G mixes position and attitude through Gam) and which FMA contraction rounds differently from the
    host.  (With the conventional model's refined gain evaluated in float, one of its 300 covariances came out
    indefinite, min eigenvalue -4.9e-7.)"""
    rng = np.random.default_rng(3)
    N = 300
    p = q.default_params()
    p.direct_orien_method = direct
    for i in range(3):
        p.R_r[i] *= 1e-3
        p.R_ang[i] *= 1e-3
    f = orc.Filter(orc.params_from(p))
    qvc = orc.quat_norm(np.array(list(p.q_vc)))
    x, P, tag = np.zeros((16, N)), np.zeros((15, 15, N)), np.zeros((7, N))
    for t in range(N):
        x[:, t], Pt, _ = rand_case(rng, 15, 1)
        d = 10.0 ** (rng.uniform(-1.5, 1.5, 15) / 2)
        P[:, :, t] = Pt * np.outer(d, d)
        qt = orc.quat_mul(x[6:10, t], orc.quat_exp(rng.normal(scale=0.05, size=3)))
        tag[3:7, t] = orc.quat_mul(qt, qvc) * np.array([-1, -1, -1, 1.0])
        tag[0:3, t] = rng.normal(scale=0.5, size=3) + [0, 0, 2]
    b = q.BatchEKF(p, N, precision=FP32)
    b.set_state(x, P)
    b.correction_step(tag)
    Pg = b.cov()
    Pc = np.stack([f.correction_step(x[:, t], P[:, :, t], tag[0:3, t], tag[3:7, t])[1] for t in range(N)], axis=2)
    assert_spd(Pg)
    errs = _per_case(Pg, Pc)
    print("joseph direct=%d: max %.2e median %.2e" % (direct, errs.max(), np.median(errs)))
    assert errs.max() < (3e-6 if direct else 5e-6) and np.median(errs) < 2e-7
    b.close()


@pytest.mark.parametrize("est_bias,direct,mode,sweep", REPLAY_CASES)
def test_fp32_replay_matches_oracle(est_bias, direct, mode, sweep):
    """N = 400 (a ragged last CTA at the FP32 block of 384), 3,000 ticks with a common and private dropouts, three
    launches with odd cut points, checked after each."""
    N = 400
    p, st, sv = replay_setup(est_bias, direct, mode, sweep, N, seed=41)
    args = (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    ob = orc.Batch(orc.params_from(p), N)
    b = q.BatchEKF(p, N, precision=FP32)
    for field, v in sv.items():
        ob.set_filter_params(field, v)
        b.set_filter_params(field, v)
    worst = np.zeros(3)
    for k0, n in CUTS:
        ob.run(k0, n, *args)
        b.run(k0, n, *args)
        assert_decisions_equal(b.flags(), ob.flags(), p.multirate_ekf)
        worst = np.maximum(worst, assert_fp32_close(b.state(), b.cov(), ob.state(), ob.cov()))
    print("replay %s: state %.2e cov %.2e scaled %.2e" % ((est_bias, direct, mode, sweep), *worst))
    assert ob.counts()[1] > 150 * N
    b.close()


def _mc_scenario(p, multirate):
    return delayed_scenario(p, 0.030 if multirate else 0.0, seconds=8.0)


def _drift_tolerance(e, dx, n):
    """Bound on the change of the sums of e_c^2 when the states move by dx = |x32 - x64| [16][N] (e [n][N] of the
    oracle's states): |d(e^2)| <= 2 |e| de + de^2 with de = dx on r, v and the biases and 2 max|dq| on the attitude."""
    de = np.zeros_like(e)
    de[0:6] = dx[0:6]
    de[6:9] = 2 * dx[6:10].max(axis=0)
    if n == 15:
        de[9:15] = dx[10:16]
    t = 2 * (2 * np.abs(e) * de + de ** 2).sum(axis=1)
    return np.concatenate([t, [t[0:3].sum()]])


@pytest.mark.parametrize("sweep", [0, 1])
@pytest.mark.parametrize("multirate", [0, 1])
@pytest.mark.parametrize("est_bias,direct", [(1, 1), (1, 0), (0, 1), (0, 0)])
def test_fp32_monte_carlo_matches_explicit_path_and_statistics(est_bias, direct, multirate, sweep):
    """In-kernel noise in FP32: (a) equal, bit for bit, to the FP32 explicit-stream replay of the dumped realisation;
    (b) the statistics against a float64 evaluation of the handle's OWN FP32 states, launched in `stride`-tick
    chunks (isolates the FP32 NEES from trajectory drift; tolerances derived in test_fp32_host.stats_reference from
    the condition number of the sampled correlation matrices, capped at NEES_REL); (c) the states within the FP32 bars
    of the oracle replaying the realisation; the squared-error sums, column by column, within the change that the
    measured state difference can make (_drift_tolerance); the NEES sums within 1e-3 relative per bin (measured:
    3.9e-6) and the chi-square counts within 1 % of the samples.  sweep: per-filter parameter tables (PF=1 kernels,
    explicit and SYNTH)."""
    p = rotors_params(q.default_params(), est_bias=est_bias, direct=direct, multirate=bool(multirate))
    scn = _mc_scenario(p, multirate)
    noise = mc_noise(first=3000)
    N, stride = 400, 400
    nb = scn.T // stride
    n = 15 if est_bias else 9
    b = q.BatchEKF(p, N, precision=FP32)
    b.stats_configure(nb, stride)
    st = b.synthesize_streams(scn, noise, 0, N)
    args = (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    ob = orc.Batch(orc.params_from(p), N)
    sv = sweep_values(np.random.default_rng(5), p, N, bool(multirate)) if sweep else {}
    for field, v in sv.items():
        ob.set_filter_params(field, v)
        b.set_filter_params(field, v)
    own, own_tol, orac = np.zeros((nb, 20)), np.zeros((nb, 20)), np.zeros((nb, 20))
    drift = np.zeros((nb, n + 1))
    kmax = 0.0
    for k in range(nb):
        b.run_monte_carlo(scn, noise, k * stride, stride)
        own[k], own_tol[k], kap = stats_reference(b.state(), b.cov(), scn.truth[(k + 1) * stride], st["bias"], n, est_bias)
        kmax = max(kmax, kap)
        ob.run(k * stride, stride, *args)
        orac[k], _, _ = stats_reference(ob.state(), ob.cov(), scn.truth[(k + 1) * stride], st["bias"], n, est_bias)
        e, _ = noise_np.error_stats(ob.state(), ob.cov(), scn.truth[(k + 1) * stride], st["bias"], n)
        drift[k] = _drift_tolerance(e, np.abs(b.state() - ob.state()), n)
    stats = b.stats()
    # (a)
    b2 = q.BatchEKF(p, N, precision=FP32)
    for field, v in sv.items():
        b2.set_filter_params(field, v)
    b2.run(0, scn.T, *args)
    for x, y in ((b.state(), b2.state()), (b.cov(), b2.cov()), (b.aux(), b2.aux()), (b.flags(), b2.flags())):
        assert np.array_equal(x, y, equal_nan=True)
    # (b)
    assert np.array_equal(stats[:, 16], own[:, 16]) and np.all(stats[:, 18] == 0)
    assert np.all(np.abs(stats - own) <= own_tol), np.argwhere(np.abs(stats - own) > own_tol)
    nees_err = np.max(np.abs(stats[:, 15] - own[:, 15]) / own[:, 15])
    # (c)
    assert_decisions_equal(b.flags(), ob.flags(), multirate)
    worst = assert_fp32_close(b.state(), b.cov(), ob.state(), ob.cov())
    assert np.array_equal(stats[:, 16], orac[:, 16])
    assert np.all(np.abs(stats[:, 17] - orac[:, 17]) <= 0.01 * N)
    cols = list(range(n)) + [19]
    assert np.all(np.abs(stats[:, cols] - orac[:, cols]) <= drift + own_tol[:, cols]), \
        np.argwhere(np.abs(stats[:, cols] - orac[:, cols]) > drift + own_tol[:, cols])
    assert np.all(np.abs(stats[:, 15] - orac[:, 15]) <= 1e-3 * orac[:, 15])
    print("monte carlo %s: kappa %.0f, NEES rel err vs own states %.2e (bound %.2e), vs oracle %.2e; state %.2e cov %.2e "
          "scaled %.2e" % ((est_bias, direct, multirate, sweep), kmax, nees_err, np.max(own_tol[:, 15] / own[:, 15]),
                            norm_rel(stats[:, 15], orac[:, 15]), *worst))
    assert orac[:, 16].sum() > 0
    b.close(); b2.close()


@pytest.mark.parametrize("name,multirate,est_bias", [("seq_sr", 0, 1), ("seq_mr", 1, 1), ("seq_mr_nb", 1, 0)])
def test_fp32_per_tick_interface_matches_golden(name, multirate, est_bias):
    """RelativePoseEKF(precision=QEKF_FP32) on the reference prototype's golden sequences: state and covariance
    within the FP32 bars, state_initialized and upds_since_correction exactly as recorded."""
    ekf = q.RelativePoseEKF(precision=FP32)
    ekf.update_freq, ekf.measurement_freq = 100.0, float(G["seq_measurement_freq"])
    ekf.limit_measurement_freq = ekf.corner_margin_enbl = ekf.direct_orien_method = 1
    ekf.multirate_ekf, ekf.dynamic_meas_delay, ekf.est_bias = multirate, 0, est_bias
    ekf.measurement_delay = 0.050
    ekf.initialize_params()
    imu, steps, poses = G[name + "_imu"], G[name + "_tag_step"], G[name + "_tag_pose"]
    arrivals = {int(s): m for m, s in enumerate(steps)}
    worst = np.zeros(3)
    n_checked = 0
    for k in range(imu.shape[0]):
        if k in arrivals:
            m = arrivals[k]
            ekf.set_tag(poses[m, 0:3], poses[m, 3:7], 0.0)
        ekf.set_imu(imu[k, 0:3], imu[k, 3:6])
        ekf.filter_update(k * 0.01)
        assert ekf.state_initialized == bool(G[name + "_active"][k])
        if not G[name + "_active"][k]:
            continue
        assert ekf.upds_since_correction == G[name + "_upds"][k]
        x = np.concatenate([ekf.r_nom, ekf.v_nom, ekf.q_nom, ekf.ab_nom, ekf.wb_nom])
        if k % 10 == 0:
            e = assert_fp32_close(x[:, None], ekf.cov_pert[:, :, None], G[name + "_x"][k][:, None],
                                  G[name + "_P"][k // 10][:, :, None])
            worst = np.maximum(worst, e)
            n_checked += 1
        else:
            assert norm_rel(x, G[name + "_x"][k]) < 1e-4
    print("per-tick %s: state %.2e cov %.2e scaled %.2e" % (name, *worst))
    assert n_checked > 10


@pytest.mark.parametrize("name,multirate", [("seq_sr", 0), ("seq_mr", 1)])
def test_fp32_per_tick_conventional_model_matches_oracle(name, multirate):
    """launch_tick<float, ..., DIRECT=0, ...>: the golden sequences' inputs with the conventional measurement model
    (which the golden file does not cover), fed tick by tick to RelativePoseEKF(precision=QEKF_FP32) and to the oracle's
    per-tick interface: FP32 bars every 10 ticks, state_initialized and upds_since_correction equal on every tick."""
    ekf = q.RelativePoseEKF(precision=FP32)
    ekf.update_freq, ekf.measurement_freq = 100.0, float(G["seq_measurement_freq"])
    ekf.limit_measurement_freq = ekf.corner_margin_enbl = 1
    ekf.direct_orien_method = 0
    ekf.multirate_ekf, ekf.dynamic_meas_delay, ekf.est_bias = multirate, 0, 1
    ekf.measurement_delay = 0.050
    ekf.initialize_params()
    f = orc.Filter(orc.params_from(ekf._params))
    imu, steps, poses = G[name + "_imu"], G[name + "_tag_step"], G[name + "_tag_pose"]
    arrivals = {int(s): m for m, s in enumerate(steps)}
    n_checked = 0
    for k in range(imu.shape[0]):
        if k in arrivals:
            m = arrivals[k]
            ekf.set_tag(poses[m, 0:3], poses[m, 3:7], 0.0)
            f.set_tag(poses[m, 0:3], poses[m, 3:7], 0.0)
        ekf.set_imu(imu[k, 0:3], imu[k, 3:6])
        f.set_imu(imu[k, 0:3], imu[k, 3:6])
        ekf.filter_update(k * 0.01)
        f.filter_update(k * 0.01)
        fl = f.flags()
        assert ekf.state_initialized == bool(fl["state_initialized"])
        if not fl["state_initialized"]:
            continue
        assert ekf.upds_since_correction == fl["upds_since_correction"]
        if k % 10 == 0:
            x = np.concatenate([ekf.r_nom, ekf.v_nom, ekf.q_nom, ekf.ab_nom, ekf.wb_nom])
            assert_fp32_close(x[:, None], ekf.cov_pert[:, :, None], f.state()[:, None], f.cov()[:, :, None])
            n_checked += 1
    assert n_checked > 10


def test_fp32_handles_ignore_the_mapping():
    """qekf.h: the cooperative mappings exist for FP64 single-rate handles; other handles keep one thread per filter.
    An FP32 handle under set_mapping(2) or set_mapping(3) must give what mapping 1 gives, bit for bit, for explicit
    and Monte-Carlo launches."""
    p = rotors_params(q.default_params())
    scn = _mc_scenario(p, 0)
    noise = mc_noise(first=11)
    N = 160
    b = q.BatchEKF(p, N)
    st = b.synthesize_streams(scn, noise, 0, N)
    b.close()
    args = (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    out = []
    for lanes in (1, 2, 3):
        res = []
        for mc in (False, True):
            h = q.BatchEKF(p, N, precision=FP32)
            h.set_mapping(lanes)
            h.stats_configure(4, 400)
            if mc:
                h.run_monte_carlo(scn, noise, 0, 999)
                h.run_monte_carlo(scn, noise, 999, scn.T - 999)
                res.append(h.stats())
            else:
                h.run(0, 999, *args)
                h.run(999, scn.T - 999, *args)
            res += [h.state(), h.cov(), h.aux(), h.flags()]
            h.close()
        out.append(res)
    for other in out[1:]:
        for x, y in zip(out[0], other):
            assert np.array_equal(x, y, equal_nan=True)


class _DeviceFP32:
    def __init__(self, p, N):
        self.b = q.BatchEKF(p, N, precision=FP32)

    def run(self, *a):
        self.b.run(*a)

    def flags_(self):
        return self.b.flags()

    def state(self):
        return self.b.state()

    def cov(self):
        return self.b.cov()


@pytest.mark.parametrize("direct", [1, 0])
def test_fp32_corner_gate_at_the_boundary_matches_oracle(direct):
    """Tag poses whose extreme corner projects 1e-6 .. 1e-2 px inside or outside each margin line: the FP32 kernels'
    accept / reject decisions, counters and states after every arrival equal the oracle's."""
    run_corner_gate_case(_DeviceFP32, direct)
