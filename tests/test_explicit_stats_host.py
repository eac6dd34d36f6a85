"""CPU tier of the on-chip statistics of explicit-stream replays (qekf_run_with_truth): the product's run_filter /
run_filter_mr instantiated for the host (tests/host_core/host_truth.cu, hc_run_truth) score a batch whose filters follow three
different landing trajectories, interleaved filter by filter (i % 3) so that no warp holds one trajectory only, each
against its own truth.  The reference is a float64 evaluation of the same streams: the batch is replayed again cut at
every sampling tick, and the states and covariances read there are scored per trajectory with
oracle/noise_np.error_stats (through test_fp32_host.stats_reference, which defines the sums and the NEES through the
quaternion log as stats_sample does).

Bars: FP64 sums within 1e-9 relative and every count equal; FP32 the per-bin tolerances stats_reference derives
(assert_stats_close).  The GPU twin is test_gpu_explicit_stats.py, which imports the batch builders below."""
import numpy as np
import pytest

import host_core as hc
from host_core.truth import run_truth
import quadrotor_landing_b200 as q
from quadrotor_landing_b200 import scenario
from streams_np import noisy_streams, rotors_params
from test_fp32_host import assert_stats_close, stats_reference
from test_multirate_host import sweep_values

GROUPS = 3
# (sway amplitude, yaw amplitude) multipliers of the default landing, one per trajectory group
SHAPES = ((1.0, 1.0), (2.5, 0.4), (0.3, 2.5))
LATENCY = {"single": 0.0, "fixed": 0.030, "dynamic": 0.042}
FP64_REL = 1e-9
SUMS = list(range(16)) + [19]
COUNTS = [16, 17, 18]


def mixed_params(est_bias, mode):
    mr, dyn = mode != "single", mode == "dynamic"
    return rotors_params(q.default_params(), est_bias=est_bias, direct=est_bias, multirate=mr, dynamic_delay=dyn)


def mixed_scenarios(p, mode, seconds=15.0):
    """Three landings with different lateral sway and yaw; same tick and arrival timing."""
    out = []
    for sway, yaw in SHAPES:
        spec = scenario.default_spec()
        spec.duration_s, spec.hover_s = seconds, 3.0
        spec.tag_latency_s = LATENCY[mode]
        spec.sway_ax *= sway; spec.sway_ay *= sway
        spec.yaw_amp *= yaw
        out.append(scenario.generate(p, spec))
    for s in out[1:]:
        assert np.array_equal(s.tag_step, out[0].tag_step) and np.array_equal(s.tag_stamp, out[0].tag_stamp)
    return out


def group_of(N):
    return np.arange(N) % GROUPS


def mixed_streams(scns, N, T, seed):
    """Explicit streams of N filters, filter i following trajectory i % 3: numpy noise (noisy_streams) with a common
    dropout and private dropouts, and each filter's true bias."""
    g = group_of(N)
    parts = [noisy_streams(scns[k], int(np.sum(g == k)), seed=seed + k, T=T, dropout=(1000, 1300),
                           random_dropout_ticks=150) for k in range(GROUPS)]
    M = parts[0]["tag_step"].shape[0]
    st = dict(imu=np.zeros((T, 6, N)), tag_step=parts[0]["tag_step"], tag_pose=np.zeros((M, 7, N)),
              tag_stamp=parts[0]["tag_stamp"], tag_valid=np.zeros((M, N), dtype=np.uint8), bias=np.zeros((6, N)))
    for k in range(GROUPS):
        sel = g == k
        st["imu"][:, :, sel] = parts[k]["imu"]
        st["tag_pose"][:, :, sel] = parts[k]["tag_pose"]
        st["tag_valid"][:, sel] = parts[k]["tag_valid"]
        st["bias"][:, sel] = parts[k]["bias"]
    return st


def mixed_truth(scns, bias, n_bins, stride):
    """[n_bins][16][N]: row block b = each filter's true state after tick (b+1)*stride - 1 (its trajectory's
    truth[(b+1)*stride]) and its true bias."""
    N = bias.shape[1]
    g = group_of(N)
    truth = np.zeros((n_bins, 16, N))
    for k in range(GROUPS):
        sel = g == k
        truth[:, 0:10, sel] = scns[k].truth[(np.arange(n_bins) + 1) * stride][:, :, None]
    truth[:, 10:16, :] = bias[None]
    return truth


def reference_bins(scns, bias, states, covs, inits, stride, est_bias):
    """float64 statistics per bin from the states / covariances / initialisation flags read after every sampling tick,
    scored trajectory by trajectory.  Returns (ref [n_bins][20], FP32 tolerance [n_bins][20])."""
    n = 15 if est_bias else 9
    nb = len(states)
    g = group_of(bias.shape[1])
    ref, tol = np.zeros((nb, 20)), np.zeros((nb, 20))
    for b in range(nb):
        for k in range(GROUPS):
            sel = (g == k) & (inits[b] != 0)
            if not sel.any():
                continue
            r, t, _ = stats_reference(states[b][:, sel], covs[b][:, :, sel], scns[k].truth[(b + 1) * stride],
                                      bias[:, sel], n, est_bias)
            ref[b] += r
            tol[b] += t
    return ref, tol


def assert_fp64_stats(stats, ref):
    assert np.array_equal(stats[:, COUNTS], ref[:, COUNTS]), (stats[:, COUNTS], ref[:, COUNTS])
    err = np.abs(stats[:, SUMS] - ref[:, SUMS])
    assert np.all(err <= FP64_REL * np.abs(ref[:, SUMS])), np.max(err / np.maximum(np.abs(ref[:, SUMS]), 1e-300))


def assert_stats_match(stats, ref, tol, prec):
    """The bars of this module: FP64 1e-9 relative and exact counts; FP32 the derived per-bin tolerances."""
    assert ref[:, 16].sum() > 0
    if prec == 64:
        assert_fp64_stats(stats, ref)
    else:
        assert_stats_close(stats, ref, tol)


CASES = ([(prec, b, m, 0) for prec in (64, 32) for b in (1, 0) for m in ("single", "fixed", "dynamic")] +
         [(64, 1, "dynamic", 1), (32, 1, "single", 1)])


@pytest.mark.parametrize("prec,est_bias,mode,sweep", CASES)
def test_explicit_statistics_match_float64_evaluation(prec, est_bias, mode, sweep):
    """24 filters on three interleaved trajectories, 3,000 ticks, stride 250 (12 bins), scored in two launches split at
    a tick that is not a multiple of the stride, against the float64 evaluation of a replay cut at every sampling
    tick.  The cut replay runs the same code on the same inputs, so its final state equals the scored one bit for bit:
    scoring does not perturb the filters."""
    N, T, stride = 24, 3000, 250
    nb = T // stride
    p = mixed_params(est_bias, mode)
    scns = mixed_scenarios(p, mode)
    st = mixed_streams(scns, N, T, seed=17)
    truth = mixed_truth(scns, st["bias"], nb, stride)
    args = (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    sv = sweep_values(np.random.default_rng(5), p, N, p.multirate_ekf) if sweep else {}

    hb = hc.HostBatch(p, N, prec=prec)
    cut = hc.HostBatch(p, N, prec=prec)
    for field, v in sv.items():
        hb.set_filter_params(field, v)
        cut.set_filter_params(field, v)
    acc = np.zeros((32, nb, 20))
    run_truth(hb, 0, 1337, st, truth, acc, stride)
    run_truth(hb, 1337, T - 1337, st, truth, acc, stride)

    states, covs, inits = [], [], []
    for b in range(nb):
        cut.run(b * stride, stride, *args)
        states.append(cut.state()); covs.append(cut.cov()); inits.append(cut.flags & 1)
    assert np.array_equal(hb.x, cut.x) and np.array_equal(hb.Ppk, cut.Ppk) and np.array_equal(hb.flags, cut.flags)

    ref, tol = reference_bins(scns, st["bias"], states, covs, inits, stride, est_bias)
    assert_stats_match(acc.sum(axis=0), ref, tol, prec)
    assert ref[-1, 16] == N


def test_explicit_statistics_bins_outside_the_replay_are_untouched():
    """Samples are taken only inside the launch's tick range and only into configured bins: a replay of ticks
    [600, 1400) with 10 bins of stride 250 fills bins 2 (tick 749) .. 4 (tick 1249) and nothing else, and more bins
    than the run reaches stay zero."""
    N, T, stride, nb = 12, 1500, 250, 10
    p = mixed_params(1, "single")
    scns = mixed_scenarios(p, "single")
    st = mixed_streams(scns, N, T, seed=3)
    truth = mixed_truth(scns, st["bias"], nb, stride)
    hb = hc.HostBatch(p, N)
    args = (st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
    hb.run(0, 600, *args)
    acc = np.zeros((32, nb, 20))
    run_truth(hb, 600, 800, st, truth, acc, stride)
    s = acc.sum(axis=0)
    assert np.all(s[[0, 1] + list(range(5, nb))] == 0)
    assert np.all(s[2:5, 16] == N)
