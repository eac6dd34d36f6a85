"""GPU tier of the parameter-space sets (param_sets.py): every kernel path with its own index or schedule arithmetic, on
parameter sets other than the rotors preset, through the C ABI against the reference-semantics oracle.  The CPU twin is
test_params_space_host.py.

- qekf_run, chunked with borders through pending measurements: every set in every delay mode, FP64 and FP32, with and
  without per-filter tables (aniso, slow_gate), N ragged around the CTA sizes.
- qekf_run_monte_carlo with private dropouts longer than the ring: the lazy and the ring history (QEKF_NO_LAZY_MR) bit for
  bit, both against the oracle replaying qekf_synthesize_streams, statistics against noise_np.error_stats of the
  oracle's states; the bundle with the detection front-end (edge_loss).
- set_mapping(2) and (3) on aniso (the relabelled per-role constants), shared constants and per-filter tables, explicit
  and Monte-Carlo.
- qekf_step open loop equals qekf_run bit for bit on every set (the stepper of test_gpu_step.py).
- qekf_tick through RelativePoseEKF (N = 1) against orc.Filter on aniso and bundle; predict_kernel / correct_kernel on
  aniso at random states, with the zero-rate small-angle branch; one scored replay on aniso."""
import numpy as np
import pytest
import torch

import host_core as hc
import param_sets as ps
import quadrotor_landing_b200 as q
from oracle import ekf_oracle as orc
from oracle import noise_np
from streams_np import norm_rel
from test_fp32_host import assert_decisions_equal, assert_fp32_close
from test_gpu_multirate import compare
from test_gpu_parity import rand_batch
from test_gpu_step import Stepper, device_streams, run_streams, snapshot
from test_multirate_host import sweep_values
from test_params_space_host import args_of, mc_noise, ring_len

pytestmark = pytest.mark.gpu
TOL = 1e-9
T_MAX = 2000
VARIANTS = [(1, 1), (1, 0), (0, 1), (0, 0)]


def variant(i):
    return VARIANTS[i % len(VARIANTS)]


def setup(name, mode, N, est_bias=1, direct=1, seed=7):
    p, scn = ps.make(name, q.default_params(), mode, est_bias, direct)
    T = min(scn.T, T_MAX)
    L = ring_len(p)
    return p, scn, ps.streams(scn, N, seed, T, max(L, 20)), T, L


RUN_CASES = ([(s, m, i, 0) for i, (s, m) in enumerate(ps.CASES)] +
             [(s, m, i, 1) for i, (s, m) in enumerate(ps.CASES) if s in ("aniso", "slow_gate")])


@pytest.mark.parametrize("name,mode,vi,pf", RUN_CASES)
def test_run_matches_oracle(name, mode, vi, pf):
    """FP64 and FP32 handles replay the same streams in the same chunks; each chunk against the oracle."""
    est_bias, direct = variant(vi)
    N = 449 if vi % 2 else 200
    p, scn, st, T, L = setup(name, mode, N, est_bias, direct)
    ob = orc.Batch(orc.params_from(p), N)
    b64, b32 = q.BatchEKF(p, N, 0, 64), q.BatchEKF(p, N, 0, 32)
    if pf:
        for field, v in sweep_values(np.random.default_rng(9), p, N, bool(p.multirate_ekf)).items():
            for h in (ob, b64, b32):
                h.set_filter_params(field, v)
    for k0, n in ps.cuts(T):
        for h in (ob, b64, b32):
            h.run(k0, n, *args_of(st))
        compare(b64, ob)
        if k0 > 1:
            assert_decisions_equal(b32.flags(), ob.flags(), p.multirate_ekf)
            assert_fp32_close(b32.state(), b32.cov(), ob.state(), ob.cov())
    assert b64.step_counts()[1] == ob.counts()[1]
    ps.assert_exercised(name, p, st, T, ob.counts()[1], ob.aux(), L if p.multirate_ekf else None)
    b64.close(); b32.close()


def oracle_stats(ob, st, scn, stride, nb, n):
    """The oracle replaying the realisation bin by bin, and the float64 statistics of its states."""
    ref = np.zeros((nb, 20))
    for k in range(nb):
        ob.run(k * stride, stride, *args_of(st))
        e, nees = noise_np.error_stats(ob.state(), ob.cov(), scn.truth[(k + 1) * stride], st["bias"], n)
        ref[k, 0:n] = (e ** 2).sum(axis=1)
        ref[k, 15], ref[k, 16] = nees.sum(), ob.N
        ref[k, 19] = (e[0:3] ** 2).sum()
    return ref


def assert_stats(stats, ref):
    assert np.array_equal(stats[:, 16], ref[:, 16])
    assert norm_rel(stats[:, 0:16], ref[:, 0:16]) < TOL and norm_rel(stats[:, 19], ref[:, 19]) < TOL


@pytest.mark.parametrize("name,mode", ps.CASES)
def test_monte_carlo_matches_oracle(monkeypatch, name, mode):
    N = 200
    p, scn, _, T, L = setup(name, mode, 4)
    noise = mc_noise(p, T, L, first=3000, edge_loss=int(name == "bundle"))
    stride = T // 5
    nb = 5
    out = []
    for env in (("1",) if p.multirate_ekf else ()) + (None,):
        monkeypatch.delenv("QEKF_NO_LAZY_MR", raising=False)
        if env:
            monkeypatch.setenv("QEKF_NO_LAZY_MR", env)
        b = q.BatchEKF(p, N)
        b.stats_configure(nb, stride)
        for k0, n in ps.cuts(nb * stride):
            b.run_monte_carlo(scn, noise, k0, n)
        out.append((snapshot(b), b.stats(), b.step_counts(), b))
    if len(out) == 2:
        (ring, rs, rc, _), (lazy, ls, lc, _) = out
        for x, y in zip(ring, lazy):
            assert np.array_equal(x, y, equal_nan=True)
        assert rc[1] == lc[1]
        assert np.array_equal(rs[:, 16:19], ls[:, 16:19]) and np.allclose(rs, ls, rtol=1e-11, atol=0)
    b = out[-1][3]
    st = b.synthesize_streams(scn, noise, 0, N)
    ob = orc.Batch(orc.params_from(p), N)
    ref = oracle_stats(ob, st, scn, stride, nb, b.n)
    compare(b, ob)
    assert_stats(b.stats(), ref)
    ps.assert_exercised(name, p, st, nb * stride, ob.counts()[1], ob.aux(), L if p.multirate_ekf else None)
    if name == "bundle":
        assert st["tag_valid"].mean() < 0.97
    for *_, h in out:
        h.close()


@pytest.mark.parametrize("pf", [False, True], ids=["shared", "perfilter"])
@pytest.mark.parametrize("lanes", [2, 3])
def test_mappings_on_aniso(lanes, pf):
    """Explicit replay against the oracle, Monte-Carlo against one thread per filter."""
    N = 200
    p, scn, st, T, L = setup("aniso", "single", N)
    sv = sweep_values(np.random.default_rng(4), p, N, False) if pf else {}
    ob = orc.Batch(orc.params_from(p), N)
    b = q.BatchEKF(p, N)
    for field, v in sv.items():
        ob.set_filter_params(field, v)
        b.set_filter_params(field, v)
    b.set_mapping(lanes)
    for k0, n in ((0, 501), (501, T - 501)):
        ob.run(k0, n, *args_of(st))
        b.run(k0, n, *args_of(st))
        assert norm_rel(b.state(), ob.state()) < TOL and norm_rel(b.cov(), ob.cov()) < TOL
        assert np.array_equal(b.flags()[0:5], ob.flags()[0:5])
        assert norm_rel(b.aux()[0:10], ob.aux()[0:10]) < TOL
    assert b.step_counts() == ob.counts()
    ps.assert_exercised("aniso", p, st, T, ob.counts()[1])
    b.close()
    noise = mc_noise(p, T, L, first=50)
    res = []
    for m in (1, lanes):
        h = q.BatchEKF(p, N)
        for field, v in sv.items():
            h.set_filter_params(field, v)
        h.set_mapping(m)
        h.stats_configure(3, T // 3)
        h.run_monte_carlo(scn, noise, 0, 613)
        h.run_monte_carlo(scn, noise, 613, T - 613)
        res.append((h.state(), h.cov(), h.stats(), h.step_counts(), h.flags()))
        h.close()
    ref, got = res
    assert norm_rel(got[0], ref[0]) < TOL and norm_rel(got[1], ref[1]) < TOL
    assert np.array_equal(got[2][:, 16:19], ref[2][:, 16:19]) and norm_rel(got[2], ref[2]) < TOL
    assert got[3] == ref[3] and np.array_equal(got[4], ref[4])


@pytest.mark.parametrize("name,mode", ps.CASES)
def test_step_open_loop_equals_run(name, mode):
    N = 449
    p, scn = ps.make(name, q.default_params(), mode)
    T = scn.T if name == "bundle" else min(scn.T, 700)     # the bundle's gate rejects late in the descent
    ds = device_streams(scn, N, T, seed=17)
    ref, b = q.BatchEKF(p, N), q.BatchEKF(p, N)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    run_streams(ref, ds, 0, T)
    Stepper(b, ds, p).run(0, T, check_every=350)
    torch.cuda.synchronize()
    for x, y in zip(snapshot(b), snapshot(ref)):
        assert np.array_equal(x, y)
    st = dict(tag_step=ds["steps"], tag_valid=ds["tag_valid"].cpu().numpy(), tag_pose=ds["tag_pose"].cpu().numpy())
    ps.assert_exercised(name, p, st, T, ref.step_counts()[1], ref.aux())
    ref.close(); b.close()


@pytest.mark.parametrize("name,mode", [("aniso", "dynamic"), ("bundle", "dynamic"), ("bundle", "single")])
def test_tick_matches_oracle_filter(name, mode):
    """The N = 1 per-tick interface (set_imu / set_tag / filter_update) against one oracle filter."""
    p, scn, st, T, L = setup(name, mode, 1, seed=3)
    T = min(T, 1200)
    ekf = q.RelativePoseEKF()
    import ctypes as C
    C.memmove(C.addressof(ekf._params), C.addressof(p), C.sizeof(p))
    ekf.initialize_params()
    f = orc.Filter(orc.params_from(p))
    arrivals = {int(s): m for m, s in enumerate(st["tag_step"]) if st["tag_valid"][m, 0]}
    for k in range(T):
        if k in arrivals:
            m = arrivals[k]
            for h in (ekf, f):
                h.set_tag(st["tag_pose"][m, 0:3, 0], st["tag_pose"][m, 3:7, 0], st["tag_stamp"][m])
        for h in (ekf, f):
            h.set_imu(st["imu"][k, 0:3, 0], st["imu"][k, 3:6, 0])
            h.filter_update(k / p.update_freq)
        if k % 100 == 99:
            fl = f.flags()
            assert ekf.upds_since_correction == fl["upds_since_correction"]
            assert ekf.state_initialized == bool(fl["state_initialized"])
            if fl["state_initialized"]:
                x = np.concatenate([ekf.r_nom, ekf.v_nom, ekf.q_nom, ekf.ab_nom, ekf.wb_nom])
                assert norm_rel(x, f.state()) < TOL and norm_rel(ekf.cov_pert, f.cov()) < TOL
    assert f.flags()["state_initialized"]


@pytest.mark.parametrize("est_bias,direct", VARIANTS)
def test_step_kernels_on_aniso(est_bias, direct):
    """predict_kernel / correct_kernel at random states with the anisotropic constants; a third of the filters get an
    angular rate of exactly zero after the bias subtraction (the small-angle branch)."""
    rng = np.random.default_rng(12)
    N = 100
    p, _ = ps.make("aniso", q.default_params(), "single", est_bias, direct)
    b = q.BatchEKF(p, N)
    n = b.n
    f = orc.Filter(orc.params_from(p))
    qvc = orc.quat_norm(np.array(list(p.q_vc)))
    x, P, u = rand_batch(rng, N, n, est_bias)
    zero = np.arange(N) % 3 == 0
    u[3:6, zero] = (x[13:16, zero] if est_bias else 0.0) + np.array(list(p.wb_static))[:, None]
    b.set_state(x, P)
    b.prediction_step(u)
    xg, Pg, ag = b.state(), b.cov(), b.aux()
    tag = np.zeros((7, N))
    for i in range(N):
        xo, Po, acc = f.prediction_step(x[:, i], P[:, :, i], u[:, i])
        assert norm_rel(xg[:, i], xo) < TOL and norm_rel(Pg[:, :, i], Po) < TOL and norm_rel(ag[0:3, i], acc) < TOL
        qt = orc.quat_mul(x[6:10, i], orc.quat_exp(rng.normal(scale=0.05 if i % 2 else 1.0, size=3)))
        tag[3:7, i] = orc.quat_mul(qt, qvc) * np.array([-1, -1, -1, 1.0])
        tag[0:3, i] = rng.normal(scale=0.5, size=3) + [0, 0, 2]
    b.set_state(x, P)
    b.correction_step(tag)
    xg, Pg, ag = b.state(), b.cov(), b.aux()
    for i in range(N):
        xc, Pc = f.correction_step(x[:, i], P[:, :, i], tag[0:3, i], tag[3:7, i])
        assert norm_rel(xg[:, i], xc) < TOL and norm_rel(Pg[:, :, i], Pc) < TOL
        a = f.aux()
        assert norm_rel(ag[3:6, i], a["r_t_vt_obs"]) < TOL and norm_rel(ag[6:10, i], a["q_tv_obs"]) < TOL
    b.close()


def test_scored_replay_on_aniso():
    """run(..., truth=) against the float64 evaluation of the oracle's states at every sampling tick."""
    N = 449
    p, scn, _, T, L = setup("aniso", "dynamic", 4)
    nb, stride = 5, T // 5
    noise = mc_noise(p, T, L, first=77)
    b = q.BatchEKF(p, N)
    st = b.synthesize_streams(scn, noise, 0, N)
    truth = np.zeros((nb, 16, N))
    truth[:, 0:10] = scn.truth[(np.arange(nb) + 1) * stride][:, :, None]
    truth[:, 10:16] = st["bias"][None]
    b.stats_configure(nb, stride)
    b.run(0, 333, *args_of(st), truth=truth)
    b.run(333, nb * stride - 333, *args_of(st), truth=truth)
    ob = orc.Batch(orc.params_from(p), N)
    ref = oracle_stats(ob, st, scn, stride, nb, b.n)
    compare(b, ob)
    assert_stats(b.stats(), ref)
    b.close()
