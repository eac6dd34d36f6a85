"""CPU tier of qekf_step, the per-tick step with per-filter device inputs and outputs: the product's step code
(deliver_one + step_filter + step_outputs, ekf_kernels.cuh) instantiated for the host (tests/host_core/host_step.cu).

- Stepping tick by tick through explicit streams reproduces the replay (run_filter / run_filter_mr) on the same streams
  bit for bit: state, covariance, aux, flags and x_hist.size(), for every est_bias x direct x {single rate, fixed delay,
  dynamic delay}, with and without per-filter parameters.
- It agrees with the reference-semantics oracle driven per tick with per-filter stamps.
- In delayed-fusion mode it keeps the head current: ~2 + d / upd_per_meas predictions per filter-tick instead of
  materialising the head from the lagged checkpoint on every tick."""
import numpy as np
import pytest

import host_core as hc
import quadrotor_landing_b200 as q
from host_core import step as hs
from oracle import ekf_oracle as orc
from quadrotor_landing_b200 import scenario
from streams_np import noisy_streams, norm_rel, rotors_params

MODES = {"single": (False, False), "fixed": (True, False), "dynamic": (True, True)}


def make_params(est_bias, direct, mode):
    mr, dyn = MODES[mode]
    return rotors_params(q.default_params(), est_bias=est_bias, direct=direct, multirate=mr, dynamic_delay=dyn)


def make_streams(p, N, T, seed, latency=0.030):
    spec = scenario.default_spec()
    spec.duration_s, spec.hover_s = 8.0, 2.0
    spec.tag_latency_s = latency
    scn = scenario.generate(p, spec)
    return scn, noisy_streams(scn, N, seed=seed, T=T, dropout=(500, 640), random_dropout_ticks=120)


def per_filter_params(hb, N, seed, mode):
    rng = np.random.default_rng(seed)
    p = hb.p
    qv = np.array(list(p.Q_a) + list(p.Q_w) + list(p.Q_ab) + list(p.Q_wb))[:, None] * rng.uniform(0.5, 2.0, (1, N))
    rv = np.array(list(p.R_r) + list(p.R_ang))[:, None] * rng.uniform(0.7, 1.5, (1, N))
    hb.set_filter_params(q.PF_Q, qv)
    hb.set_filter_params(q.PF_R, rv)
    if mode != "single":
        d = np.stack([rng.uniform(0.015, 0.045, N), rng.uniform(0.0, 0.01, N)])
        hb.set_filter_params(q.PF_DELAY, d)


def tick_inputs(st, k, m, N):
    """The arrival of tick k (if any) as qekf_step inputs: arrived = its tag_valid row, the stamp broadcast."""
    if m < len(st["tag_step"]) and st["tag_step"][m] == k:
        tag = np.concatenate([st["tag_pose"][m], np.full((1, N), st["tag_stamp"][m])])
        return st["tag_valid"][m].copy(), tag, m + 1
    return None, None, m


def step_through(hb, st, k0, n, update_freq, t_start=0.0, counts=None):
    N = hb.N
    m = int(np.searchsorted(st["tag_step"], k0))
    out = None
    for k in range(k0, k0 + n):
        arrived, tag, m = tick_inputs(st, k, m, N)
        out = hs.step(hb, t_start + k / update_freq, st["imu"][k], arrived, tag, counts=counts)
    return out


def assert_same(a, b):
    assert np.array_equal(a.x, b.x)
    assert np.array_equal(a.Ppk, b.Ppk)
    assert np.array_equal(a.aux, b.aux)
    assert np.array_equal(a.flags, b.flags)
    assert np.array_equal(a.upds, b.upds)
    assert np.array_equal(a.history_length(), b.history_length())


@pytest.mark.parametrize("pf", [False, True], ids=["shared", "perfilter"])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("est_bias,direct", [(1, 1), (1, 0), (0, 1), (0, 0)])
def test_step_reproduces_replay_bit_for_bit(est_bias, direct, mode, pf):
    p = make_params(est_bias, direct, mode)
    N, T = 4, 1100
    scn, st = make_streams(p, N, T, seed=11 + est_bias + 2 * direct, latency=0.036)
    ref, hb = hc.HostBatch(p, N), hc.HostBatch(p, N)
    if pf:
        per_filter_params(ref, N, 5, mode)
        per_filter_params(hb, N, 5, mode)
    # the replay in chunks, the step tick by tick; compared at the chunk borders
    for k0, n in ((0, 300), (300, 450), (750, 350)):
        ref.run(k0, n, st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
        out = step_through(hb, st, k0, n, p.update_freq)
        assert_same(hb, ref)
    assert (ref.flags & 1).all()
    # the outputs of the last step are the accessors' values
    x, cov, aux, fl = out
    assert np.array_equal(x, hb.x) and np.array_equal(cov, hb.Ppk) and np.array_equal(aux, hb.aux)
    assert np.array_equal(fl[0], hb.flags & 1) and np.array_equal(fl[1], (hb.flags >> 1) & 1)
    assert np.array_equal(fl[2], (hb.flags >> 2) & 1) and np.array_equal(fl[3], (hb.flags >> 3) & 1)
    assert np.array_equal(fl[4], hb.upds) and np.array_equal(fl[5], hb.history_length())


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("est_bias,direct", [(1, 1), (0, 0)])
def test_step_fp32_reproduces_fp32_replay(est_bias, direct, mode):
    p = make_params(est_bias, direct, mode)
    N, T = 3, 700
    scn, st = make_streams(p, N, T, seed=3)
    ref, hb = hc.HostBatch(p, N, prec=32), hc.HostBatch(p, N, prec=32)
    ref.run(0, T, st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    step_through(hb, st, 0, T, p.update_freq)
    assert_same(hb, ref)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("est_bias,direct", [(1, 1), (1, 0), (0, 1)])
def test_step_matches_oracle_with_per_filter_stamps(est_bias, direct, mode):
    """Every filter sees its detections with its own capture stamp (dynamic delay: its own latency), checked after every
    tick against one oracle filter each."""
    p = make_params(est_bias, direct, mode)
    N, T = 3, 900
    scn, st = make_streams(p, N, T, seed=29)
    lat = np.array([0.0, 0.012, 0.027])          # extra capture-to-arrival latency per filter
    hb = hc.HostBatch(p, N)
    op = orc.params_from(p)
    filters = [orc.Filter(op) for _ in range(N)]
    m = 0
    for k in range(T):
        t = k / p.update_freq
        arrived, tag, m = tick_inputs(st, k, m, N)
        if arrived is not None:
            tag[7] -= lat
            for i in range(N):
                if arrived[i]:
                    filters[i].set_tag(tag[0:3, i], tag[3:7, i], tag[7, i])
        for i in range(N):
            filters[i].set_imu(st["imu"][k, 0:3, i], st["imu"][k, 3:6, i])
            filters[i].filter_update(t)
        x, cov, aux, fl = hs.step(hb, t, st["imu"][k], arrived, tag)
        if k % 50 == 49 or k == T - 1:
            Pd = hb.cov()
            for i in range(N):
                f = filters[i].flags()
                assert fl[0, i] == f["state_initialized"] and fl[1, i] == f["measurement_ready"]
                assert fl[2, i] == f["performed_correction"] and fl[4, i] == f["upds_since_correction"]
                assert fl[5, i] == f["hist_len"]
                if f["state_initialized"]:
                    assert norm_rel(x[:, i], filters[i].state()) < 1e-9
                    assert norm_rel(Pd[:, :, i], filters[i].cov()) < 1e-9
    assert fl[0].all()


def test_delayed_fusion_keeps_the_head_current():
    """30 ms delay at 200 Hz / 30 Hz (d = 6 ticks): about 2 + d / upd_per_meas predictions per filter-tick."""
    p = make_params(1, 1, "fixed")
    N, T = 4, 1600
    spec = scenario.default_spec()
    spec.duration_s, spec.hover_s = 9.0, 2.0
    spec.tag_latency_s = 0.030
    scn = scenario.generate(p, spec)
    st = noisy_streams(scn, N, seed=7, T=T)
    hb = hc.HostBatch(p, N)
    step_through(hb, st, 0, 200, p.update_freq)
    assert (hb.flags & 1).all()
    counts = np.zeros(2, dtype=np.int64)
    n = T - 200
    step_through(hb, st, 200, n, p.update_freq, counts=counts)
    d = round(p.measurement_delay * p.update_freq)
    upm = p.update_freq / p.measurement_freq
    per_tick = counts[0] / (N * n)
    assert counts[1] > 0.9 * N * n / upm
    assert per_tick <= 2 + d / upm + 0.05, per_tick
    # what materialising the head on every tick would cost: one replay launch per tick
    ref = hc.HostBatch(p, N)
    ref.run(0, 200, st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    lazy = 0
    h = ref._history()
    for k in range(200, 260):
        lazy += int(h["nh"].sum()) + N        # the head materialised from the checkpoint: nh + this tick's entry
        ref.run(k, 1, st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    assert lazy / (N * 60) > 1.5 * per_tick
