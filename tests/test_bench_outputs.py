"""`bench.py --dump-outputs DIR` writes what its timed path computed, and `--steps` is the number of timed passes: the
dumped statistics and the state / covariance of the sampled filters equal a fresh handle replaying the same workload
once, and the work counted over the timed passes is `--steps` times that handle's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import quadrotor_landing_b200 as q
from streams_np import norm_rel
from test_bench_reference_config import ROOT, _bench


def _run_bench(args, cwd):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=cwd, stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True, timeout=1200)


def test_steps_below_one_are_rejected(tmp_path):
    res = _run_bench(["--steps", "0"], str(tmp_path))
    assert res.returncode == 2 and "--steps" in res.stderr, res.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_steps_computed(tmp_path):
    bench = _bench()
    N, steps = bench.DUMP_FILTERS + 904, 2          # more filters than are dumped: the seeded sample
    out = tmp_path / "out"
    res = _run_bench(["--filters", str(N), "--steps", str(steps), "--warmup", "0", "--no-legs", "--no-parity",
                      "--no-cpu-baseline", "--dump-outputs", str(out)], str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    d = {n: np.load(str(out / (n + ".npy"))) for n in ("stats", "filter_ids", "state", "cov")}
    assert all(a.dtype == np.float64 for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20
    ids = d["filter_ids"].astype(np.int64)
    assert np.array_equal(ids, d["filter_ids"]) and len(np.unique(ids)) == bench.DUMP_FILTERS and ids.max() < N

    p = bench.bench_params(q)
    scn = bench.bench_scenario(q, p)
    b = q.BatchEKF(p, N)
    b.stats_configure(scn.T // 200, 200)
    b.run_monte_carlo(scn, bench.bench_noise(q))
    n_pred, n_corr = b.step_counts()
    work = line["roofline"]["work"]
    assert (work["prediction_steps"], work["correction_steps"]) == (n_pred, n_corr)
    assert norm_rel(d["stats"], b.stats()) < 1e-12
    assert norm_rel(d["state"], np.concatenate([b.state(int(i), 1) for i in ids], axis=1)) < 1e-12
    assert norm_rel(d["cov"], np.concatenate([b.cov(int(i), 1) for i in ids], axis=2)) < 1e-12
    b.close()
