"""GPU tier of the on-chip statistics of explicit-stream replays (qekf_run_with_truth, BatchEKF.run(truth=...) /
run_device(truth_ptr=...)).

1. Agreement with the Monte-Carlo path: the realisation of qekf_run_monte_carlo (qekf_synthesize_streams) replayed as
   explicit streams and scored against the scenario truth and the dumped true bias gives the states of the unscored
   replay bit for bit, those of the Monte-Carlo run bit for bit or (one variant) to rounding, and the same statistics:
   equal counts, sums within 1e-12 relative (a reordered Monte-Carlo launch groups other filters into warps, which
   changes only the order of the sums).
2. Per-filter indexing: three trajectories interleaved filter by filter, N = 4,096 and 100,003 (not a multiple of the
   warp), host and device truth, against the float64 evaluation of a replay cut at every sampling tick
   (test_explicit_stats_host).
3. Scoring changes nothing: truth = NULL is qekf_run, and a scored replay leaves the filters as an unscored one.
4. Chunked launches and export / import give the statistics of one uninterrupted launch.
5. Interface: truth without statistics configured, bad tick ranges, and the cooperative mapping."""
import ctypes as C

import numpy as np
import pytest

import quadrotor_landing_b200 as q
from quadrotor_landing_b200 import _native as nat
from streams_np import norm_rel, rotors_params
from test_explicit_stats_host import (assert_stats_match, mixed_params, mixed_scenarios, mixed_streams, mixed_truth,
                                      reference_bins)
from test_fp32_host import mc_noise
from test_multirate_host import delayed_scenario, sweep_values

pytestmark = pytest.mark.gpu

SUMS = list(range(16)) + [19]
COUNTS = [16, 17, 18]


def snapshot(b):
    return [b.state(), b.cov(), b.aux(), b.flags()]


def assert_same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)


def assert_same_stats(s, r, rel=1e-12):
    """Equal counts, sums within `rel` relative (atomic accumulation: only the order of the additions may differ)."""
    assert np.array_equal(s[:, COUNTS], r[:, COUNTS]), (s[:, COUNTS], r[:, COUNTS])
    assert np.all(np.abs(s[:, SUMS] - r[:, SUMS]) <= rel * np.abs(r[:, SUMS])), \
        np.max(np.abs(s[:, SUMS] - r[:, SUMS]) / np.maximum(np.abs(r[:, SUMS]), 1e-300))


def args_of(st):
    return (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])


# ---- 1. agreement with the Monte-Carlo path ------------------------------------------------------------------------

MC_CASES = ([(prec, b, d, m, 0) for prec in (64, 32) for b, d in ((1, 1), (1, 0), (0, 1), (0, 0))
             for m in ("single", "fixed", "dynamic")] +
            [(64, 1, 1, "single", 1), (64, 1, 0, "dynamic", 1), (32, 1, 1, "fixed", 1)])


@pytest.mark.parametrize("prec,est_bias,direct,mode,sweep", MC_CASES)
def test_explicit_statistics_equal_monte_carlo_statistics(prec, est_bias, direct, mode, sweep):
    p = rotors_params(q.default_params(), est_bias=est_bias, direct=direct, multirate=mode != "single",
                      dynamic_delay=mode == "dynamic")
    scn = delayed_scenario(p, {"single": 0.0, "fixed": 0.030, "dynamic": 0.042}[mode], seconds=8.0)
    noise = mc_noise(first=500)
    N, stride = 1000, 200
    nb = scn.T // stride
    sv = sweep_values(np.random.default_rng(11), p, N, mode != "single") if sweep else {}
    mc, ex, plain = (q.BatchEKF(p, N, precision=prec) for _ in range(3))
    for b in (mc, ex, plain):
        for field, v in sv.items():
            b.set_filter_params(field, v)
    mc.stats_configure(nb, stride)
    ex.stats_configure(nb, stride)
    st = mc.synthesize_streams(scn, noise, 0, N)
    truth = np.zeros((nb, 16, N))
    truth[:, 0:10] = scn.truth[(np.arange(nb) + 1) * stride][:, :, None]
    truth[:, 10:16] = st["bias"][None]
    mc.run_monte_carlo(scn, noise)
    ex.run(0, scn.T, *args_of(st), truth=truth)
    plain.run(0, scn.T, *args_of(st))
    assert_same(snapshot(ex), snapshot(plain))
    # the Monte-Carlo and explicit kernels agree bit for bit in every variant but FP64 est_bias = 0, direct = 1, where one
    # filter of this batch differs in the last bit (2.8e-17 in the state) without statistics as well: to rounding here
    got, want = snapshot(ex), snapshot(mc)
    assert np.array_equal(got[3], want[3])
    for x, y in zip(got[:3], want[:3]):
        assert norm_rel(x, y) <= 1e-12
    s_mc, s_ex = mc.stats(), ex.stats()
    assert s_mc[:, 16].sum() > 0.9 * N * nb
    assert_same_stats(s_ex, s_mc)
    for h in (mc, ex, plain):
        h.close()


# ---- 2. per-filter indexing ----------------------------------------------------------------------------------------

INDEX_CASES = [(4096, 64, "single"), (4096, 32, "single"), (4096, 64, "fixed"), (4096, 32, "dynamic"),
               (100003, 64, "single"), (100003, 32, "single")]


@pytest.mark.parametrize("N,prec,mode", INDEX_CASES)
def test_explicit_statistics_index_every_filter(N, prec, mode):
    import torch
    T, stride = (1500, 250) if N < 10000 else (300, 60)
    nb = T // stride
    est_bias = 1
    p = mixed_params(est_bias, mode)
    scns = mixed_scenarios(p, mode, seconds=T / p.update_freq + 1.0)
    st = mixed_streams(scns, N, T, seed=23)
    truth = mixed_truth(scns, st["bias"], nb, stride)

    cut = q.BatchEKF(p, N, precision=prec)
    states, covs, inits = [], [], []
    for b in range(nb):
        cut.run(b * stride, stride, *args_of(st))
        states.append(cut.state()); covs.append(cut.cov()); inits.append(cut.flags()[0])
    ref, tol = reference_bins(scns, st["bias"], states, covs, inits, stride, est_bias)
    want = snapshot(cut)
    cut.close()
    del states, covs

    host = q.BatchEKF(p, N, precision=prec)
    host.stats_configure(nb, stride)
    host.run(0, T, *args_of(st), truth=truth)
    assert_same(snapshot(host), want)
    s_host = host.stats()
    assert_stats_match(s_host, ref, tol, prec)
    host.close()

    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in st.items() if k != "bias"}
    d_truth = torch.from_numpy(truth).to(dev)
    devh = q.BatchEKF(p, N, precision=prec)
    devh.stats_configure(nb, stride)
    devh.run_device(0, T, T, d["imu"].data_ptr(), d["tag_step"].shape[0], d["tag_step"].data_ptr(),
                    d["tag_pose"].data_ptr(), d["tag_stamp"].data_ptr(), d["tag_valid"].data_ptr(),
                    truth_ptr=d_truth.data_ptr())
    devh.sync()
    assert_same(snapshot(devh), want)
    s_dev = devh.stats()
    assert_stats_match(s_dev, ref, tol, prec)
    assert_same_stats(s_dev, s_host)
    devh.close()
    del d, d_truth
    torch.cuda.empty_cache()


# ---- 3. scoring changes nothing -------------------------------------------------------------------------------------

def _raw_run(b, st, k0, n, truth_ptr, use_truth_entry):
    """qekf_run / qekf_run_with_truth through the C ABI with host streams."""
    imu = np.ascontiguousarray(st["imu"]); step = np.ascontiguousarray(st["tag_step"], dtype=np.int32)
    pose = np.ascontiguousarray(st["tag_pose"]); stamp = np.ascontiguousarray(st["tag_stamp"])
    valid = np.ascontiguousarray(st["tag_valid"], dtype=np.uint8)
    s = nat.QekfStreams()
    s.T, s.imu, s.M = imu.shape[0], imu.ctypes.data, step.shape[0]
    s.tag_step, s.tag_pose, s.tag_stamp, s.tag_valid = step.ctypes.data, pose.ctypes.data, stamp.ctypes.data, valid.ctypes.data
    s.t_start, s.on_device = 0.0, 0
    L = nat.lib()
    if use_truth_entry:
        rc = L.qekf_run_with_truth(b._h, C.byref(s), truth_ptr, int(k0), int(n))
    else:
        rc = L.qekf_run(b._h, C.byref(s), int(k0), int(n))
    b.sync()
    return rc


@pytest.mark.parametrize("prec,mode", [(64, "single"), (32, "single"), (64, "dynamic")])
def test_scoring_does_not_change_the_filters(prec, mode):
    N, T, stride = 700, 1500, 250
    p = mixed_params(1, mode)
    scns = mixed_scenarios(p, mode)
    st = mixed_streams(scns, N, T, seed=5)
    truth = mixed_truth(scns, st["bias"], T // stride, stride)
    a, b, c = (q.BatchEKF(p, N, precision=prec) for _ in range(3))
    assert _raw_run(a, st, 0, T, None, False) == 0
    assert _raw_run(b, st, 0, T, None, True) == 0
    c.stats_configure(T // stride, stride)
    assert _raw_run(c, st, 0, T, truth.ctypes.data, True) == 0
    want = snapshot(a)
    assert_same(snapshot(b), want)
    assert_same(snapshot(c), want)
    assert a.step_counts() == b.step_counts()
    # delayed fusion scores the head, which it materialises from the lagged checkpoint at every sample on a copy: more
    # predictions are executed, the filters are the same
    (pa, ca), (pc, cc) = a.step_counts(), c.step_counts()
    assert cc == ca and (pc > pa if p.multirate_ekf else pc == pa)
    assert c.stats()[:, 16].sum() > 0
    for h in (a, b, c):
        h.close()


# ---- 4. chunked launches, export / import ---------------------------------------------------------------------------

@pytest.mark.parametrize("prec,mode", [(64, "single"), (64, "fixed"), (32, "dynamic")])
def test_chunked_and_resumed_replays_give_the_same_statistics(prec, mode):
    """Chunks split at ticks that are not multiples of the stride; each chunk gets a host truth in which every bin it
    does not sample is NaN, so a chunk that read any other bin would count diverged samples or NaN sums."""
    N, T, stride = 2000, 1500, 250
    nb = T // stride
    p = mixed_params(1, mode)
    scns = mixed_scenarios(p, mode)
    st = mixed_streams(scns, N, T, seed=9)
    truth = mixed_truth(scns, st["bias"], nb, stride)

    one = q.BatchEKF(p, N, precision=prec)
    one.stats_configure(nb, stride)
    one.run(0, T, *args_of(st), truth=truth)
    want, s_one = snapshot(one), one.stats()
    one.close()

    cuts = [0, 137, 499, 500, 911, 1249, 1377, T]
    ch = q.BatchEKF(p, N, precision=prec)
    ch.stats_configure(nb, stride)
    for k0, k1 in zip(cuts[:-1], cuts[1:]):
        own = np.full_like(truth, np.nan)
        sampled = [b for b in range(nb) if k0 <= (b + 1) * stride - 1 < k1]
        own[sampled] = truth[sampled]
        ch.run(k0, k1 - k0, *args_of(st), truth=own)
    assert_same(snapshot(ch), want)
    assert_same_stats(ch.stats(), s_one)
    ch.close()

    mid = 777
    a = q.BatchEKF(p, N, precision=prec)
    a.stats_configure(nb, stride)
    a.run(0, mid, *args_of(st), truth=truth)
    blob = a.export_state()
    a.close()
    r = q.BatchEKF(p, N, precision=prec)
    r.import_state(blob)
    r.run(mid, T - mid, *args_of(st), truth=truth)
    assert_same(snapshot(r), want)
    assert_same_stats(r.stats(), s_one)
    r.close()


# ---- 5. interface ----------------------------------------------------------------------------------------------------

def test_truth_without_statistics_and_bad_ranges_are_refused():
    N, T, stride = 64, 600, 100
    p = mixed_params(1, "single")
    scns = mixed_scenarios(p, "single")
    st = mixed_streams(scns, N, T, seed=1)
    truth = mixed_truth(scns, st["bias"], T // stride, stride)
    b = q.BatchEKF(p, N)
    with pytest.raises(q.QekfError) as e:
        b.run(0, T, *args_of(st), truth=truth)
    assert e.value.code == 3                                   # QEKF_ERR_NOT_INITIALIZED
    b.stats_configure(T // stride, stride)
    assert _raw_run(b, st, 0, T + 1, truth.ctypes.data, True) == 1      # QEKF_ERR_BAD_ARG
    assert _raw_run(b, st, -1, 10, truth.ctypes.data, True) == 1
    assert np.all(b.stats() == 0) and not b.flags()[0].any()
    b.close()


def test_cooperative_mapping_scores_with_one_thread_per_filter():
    """A handle set to three lanes per filter runs a scored replay one thread per filter: the result of a handle with
    the default mapping, bit for bit (the three-lane kernel agrees only to rounding)."""
    N, T, stride = 1000, 1500, 250
    p = mixed_params(1, "single")
    scns = mixed_scenarios(p, "single")
    st = mixed_streams(scns, N, T, seed=2)
    truth = mixed_truth(scns, st["bias"], T // stride, stride)
    ref = q.BatchEKF(p, N)
    ref.stats_configure(T // stride, stride)
    ref.run(0, T, *args_of(st), truth=truth)
    co = q.BatchEKF(p, N)
    co.set_mapping(3)
    co.stats_configure(T // stride, stride)
    co.run(0, T, *args_of(st), truth=truth)
    assert_same(snapshot(co), snapshot(ref))
    assert_same_stats(co.stats(), ref.stats())
    ref.close(); co.close()
