"""CPU tier of the parameter-space sets (param_sets.py): the product's code instantiated for the host (tests/host_core)
against the reference-semantics oracle on parameter sets other than the rotors preset -- anisotropic constants, non-zero
static biases, a tilted g, other camera intrinsics and extrinsics, gate ratios upd_per_meas = 1, 2, 4, 5, 10 and 16,
detections faster and slower than the gate, the delay clamp and the 13-tag bundle.

Same bars as the rotors tests: FP64 1e-9 norm-relative on state and covariance with the discrete decisions, counters and
x_hist.size() exactly equal; FP32 through the per-filter helpers of test_fp32_host.py.  Every test also asserts that its
set exercised what it is for (param_sets.assert_exercised)."""
import numpy as np
import pytest

import host_core as hc
import param_sets as ps
import quadrotor_landing_b200 as q
from host_core import step as hs
from oracle import ekf_oracle as orc
from quadrotor_landing_b200 import _native as nat
from streams_np import norm_rel
from test_fp32_host import assert_decisions_equal, assert_fp32_close, host_flags
from test_multirate_host import compare, sweep_values
from test_step_host import assert_same, step_through

N = 4
T_MAX = 2000
# (est_bias, direct) per case: both models with bias estimation everywhere, the bias-free models on a subset
VARIANTS = [(1, 1), (1, 0)]
CASES64 = ([(s, m, b, d) for s, m in ps.CASES for b, d in VARIANTS] +
           [(s, m, 0, d) for s, m in ps.CASES if m != "fixed" for d in ((1,) if s != "aniso" else (1, 0))])


def ring_len(p):
    return hc.HostBatch(p, 1)._history()["ring_len"] if p.multirate_ekf else 0


def setup(name, mode, est_bias=1, direct=1, n=N, seed=7):
    p, scn = ps.make(name, q.default_params(), mode, est_bias, direct)
    T = min(scn.T, T_MAX)
    L = ring_len(p)
    st = ps.streams(scn, n, seed, T, max(L, 20))
    return p, scn, st, T, L


def args_of(st):
    return st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"]


def exercised(name, p, st, T, ob, L):
    ps.assert_exercised(name, p, st, T, ob.counts()[1], ob.aux(), L if p.multirate_ekf else None)


@pytest.mark.parametrize("name,mode,est_bias,direct", CASES64)
def test_replay_matches_oracle(name, mode, est_bias, direct):
    """Chunked explicit-stream replay (run_filter / run_filter_mr) with borders through pending measurements."""
    p, scn, st, T, L = setup(name, mode, est_bias, direct)
    ob = orc.Batch(orc.params_from(p), N)
    hb = hc.HostBatch(p, N)
    for k0, n in ps.cuts(T):
        ob.run(k0, n, *args_of(st))
        hb.run(k0, n, *args_of(st))
        compare(hb, ob)
    exercised(name, p, st, T, ob, L)
    # tracking (the bundle ends 0.35 m above the tags, where most arrivals are rejected)
    assert np.max(np.abs(ob.state()[0:3] - scn.truth[T][0:3, None])) < (0.25 if name == "bundle" else 0.1)


@pytest.mark.parametrize("name,mode", ps.CASES)
def test_fp32_replay_matches_oracle(name, mode):
    p, scn, st, T, L = setup(name, mode, seed=31)
    ob = orc.Batch(orc.params_from(p), N)
    hb = hc.HostBatch(p, N, prec=32)
    a, b = T // 3 + 1, (2 * T) // 3 - 2
    for k0, n in ((0, a), (a, b - a), (b, T - b)):
        ob.run(k0, n, *args_of(st))
        hb.run(k0, n, *args_of(st))
        assert_decisions_equal(host_flags(hb), ob.flags(), p.multirate_ekf)
        assert_fp32_close(hb.state(), hb.cov(), ob.state(), ob.cov())
    exercised(name, p, st, T, ob, L)


def sweep_all(p, n, seed):
    """Per-filter values of all five overridable fields (the delay field in every mode: a single-rate handle ignores
    it)."""
    return sweep_values(np.random.default_rng(seed), p, n, True)


@pytest.mark.parametrize("prec", [64, 32])
@pytest.mark.parametrize("name,mode", [(s, m) for s, m in ps.CASES if s in ("aniso", "slow_gate")])
def test_per_filter_sweep_matches_oracle(name, mode, prec):
    """Every PF_* field overridden per filter on top of the anisotropic and the 16-ticks-per-gate sets."""
    n = 6
    p, scn, st, T, L = setup(name, mode, n=n, seed=77)
    ob = orc.Batch(orc.params_from(p), n)
    hb = hc.HostBatch(p, n, prec=prec)
    for field, v in sweep_all(p, n, 9).items():
        ob.set_filter_params(field, v)
        hb.set_filter_params(field, v)
    for k0, n_ in ((0, T // 2 + 1), (T // 2 + 1, T - T // 2 - 1)):
        ob.run(k0, n_, *args_of(st))
        hb.run(k0, n_, *args_of(st))
        if prec == 64:
            compare(hb, ob)
        else:
            assert_decisions_equal(host_flags(hb), ob.flags(), p.multirate_ekf)
            assert_fp32_close(hb.state(), hb.cov(), ob.state(), ob.cov())
    assert norm_rel(ob.cov()[:, :, 0], ob.cov()[:, :, 1]) > 1e-2
    ps.assert_exercised(name, p, st, T, ob.counts()[1], ob.aux(), None)


def mc_noise(p, T, L, first=0, edge_loss=0):
    """Monte-Carlo noise with a common dropout and private dropouts longer than the ring (reordering on)."""
    n = nat.default_noise()
    n.seed = 2024
    n.first_global_id = first
    d = 2 * max(L, 20) + 7
    n.dropout_k0, n.dropout_k1 = T // 3, T // 3 + d
    n.rand_dropout_len, n.rand_dropout_lo, n.rand_dropout_hi = d, 20, T - d - 20
    n.edge_loss = edge_loss
    return n


@pytest.mark.parametrize("name,mode", ps.CASES)
def test_monte_carlo_matches_oracle(name, mode):
    """In-kernel noise (run_filter_mc / run_filter_mrs): with delayed fusion the lazy loop equals the ring-based loop bit
    for bit, statistics included; both equal the oracle replaying the dumped realisation.  The bundle runs the
    detection front-end (edge_loss)."""
    p, scn, _, _, L = setup(name, mode)
    T = min(scn.T, T_MAX)
    scn.T = T
    noise = mc_noise(p, T, L, first=1000, edge_loss=int(name == "bundle"))
    stride = T // 4
    runs = []
    for lazy in ((False, True) if p.multirate_ekf else (False,)):
        hb = hc.HostBatch(p, N)
        acc = np.zeros((32, 4, 20))
        for k0, n in ps.cuts(T):
            hb.run_mc(scn, noise, k0, n, acc, stride, lazy=lazy)
        runs.append((hb, acc.sum(axis=0)))
    if len(runs) == 2:
        (ring, rs), (lz, ls) = runs
        assert_same(ring, lz)
        assert np.array_equal(rs[:, 16:19], ls[:, 16:19]) and np.allclose(rs, ls, rtol=1e-12, atol=0)
    hb = runs[-1][0]
    st = hc.synthesize(scn, noise, 0, N, params=p)
    ob = orc.Batch(orc.params_from(p), N)
    ob.run(0, T, *args_of(st))
    compare(hb, ob)
    exercised(name, p, st, T, ob, L)
    if name == "bundle":       # the front-end dropped detections with no tag in the image
        assert st["tag_valid"].mean() < 0.97


@pytest.mark.parametrize("pf", [False, True], ids=["shared", "perfilter"])
@pytest.mark.parametrize("name,mode", ps.CASES)
def test_step_reproduces_replay(name, mode, pf):
    """The per-tick step (step_filter, its own gate and catch-up arithmetic) equals the replay bit for bit."""
    n = 3
    p, scn, st, T, L = setup(name, mode, n=n, seed=13)
    T = min(T, 1200)
    ref, hb = hc.HostBatch(p, n), hc.HostBatch(p, n)
    if pf:
        for field, v in sweep_all(p, n, 5).items():
            ref.set_filter_params(field, v)
            hb.set_filter_params(field, v)
    for k0, n_ in ((0, T // 3), (T // 3, T - T // 3)):
        ref.run(k0, n_, *args_of(st))
        step_through(hb, st, k0, n_, p.update_freq)
        assert_same(hb, ref)
    assert (ref.flags & 1).all()


@pytest.mark.parametrize("kind", ["coop", "duo"])
@pytest.mark.parametrize("name", [s for s in ps.NAMES if "single" in ps.SETS[s]["modes"]])
def test_cooperative_mappings_match_oracle(name, kind):
    """The three-lane (relabelled per-role constants, fill_role_consts) and the two-role replays, single rate."""
    n = 3
    p, scn, st, T, L = setup(name, "single", n=n, seed=11)
    ob = orc.Batch(orc.params_from(p), n)
    hb = (hc.CoopHostBatch if kind == "coop" else hc.DuoHostBatch)(p, n)
    for k0, n_ in ((0, T // 2 + 3), (T // 2 + 3, T - T // 2 - 3)):
        ob.run(k0, n_, *args_of(st))
        hb.run(k0, n_, *args_of(st))
        assert hb.races == 0
        assert norm_rel(hb.state(), ob.state()) < 1e-9
        assert norm_rel(hb.cov(), ob.cov()) < 1e-9
        fl = ob.flags()
        assert np.array_equal(hb.upds, fl[4])
        assert np.array_equal(hb.flags & 1, fl[0]) and np.array_equal((hb.flags >> 1) & 1, fl[1])
        assert norm_rel(hb.aux[0:10], ob.aux()[0:10]) < 1e-9
    ps.assert_exercised(name, p, st, T, ob.counts()[1])
