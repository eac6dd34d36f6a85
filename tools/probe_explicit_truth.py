"""Cost of scoring an explicit-stream replay on chip (qekf_run_with_truth) against the same replay unscored.

Device-resident streams as in perf_probe.py, per-filter truth [n_bins][16][N] on the device, statistics sampled every
`stride` ticks.  Scored and unscored launches alternate on the same handle (the filters are reset before each), and
the best of `reps` of each is reported.  Usage: python tools/probe_explicit_truth.py [N] [T] [stride]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import quadrotor_landing_b200 as q
from quadrotor_landing_b200 import scenario
from streams_np import rotors_params


def probe(N, T, stride, precision, reps=4):
    p = rotors_params(q.default_params())
    scn = scenario.generate(p)
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    sel = scn.tag_step < T
    M = int(sel.sum())
    steps = torch.tensor(scn.tag_step[sel], dtype=torch.int32, device=dev)
    imu = torch.tensor(scn.imu_clean[:T], device=dev)[:, :, None] + \
        0.02 * torch.randn((T, 6, N), dtype=torch.float64, device=dev, generator=g)
    pose = torch.tensor(scn.tag_pose_clean[sel], device=dev)[:, :, None].repeat(1, 1, N)
    pose[:, 0:3] += 0.02 * torch.randn((M, 3, N), dtype=torch.float64, device=dev, generator=g)
    stamp = torch.tensor(scn.tag_stamp[sel], device=dev)
    nb = T // stride
    truth = torch.zeros((nb, 16, N), dtype=torch.float64, device=dev)
    truth[:, 0:10] = torch.tensor(scn.truth[(np.arange(nb) + 1) * stride], device=dev)[:, :, None]
    b = q.BatchEKF(p, N, precision=precision)
    b.stats_configure(nb, stride)
    s = torch.cuda.current_stream()
    b.set_stream(s.cuda_stream)
    times = {False: [], True: []}
    for r in range(reps + 1):
        for scored in (False, True):
            b.reset_filters()
            b.stats_reset()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            b.run_device(0, T, T, imu.data_ptr(), M, steps.data_ptr(), pose.data_ptr(), stamp.data_ptr(),
                         truth_ptr=truth.data_ptr() if scored else None)
            e1.record(s)
            torch.cuda.synchronize()
            if r > 0:                                    # the first round warms up
                times[scored].append(e0.elapsed_time(e1))
    t0, t1 = min(times[False]), min(times[True])
    st = b.stats()
    print("N=%d T=%d stride=%d fp%d: unscored %.2f ms, scored %.2f ms -> %+.2f %% (samples %d, diverged %d)" % (
        N, T, stride, precision, t0, t1, 100.0 * (t1 - t0) / t0, int(st[:, 16].sum()), int(st[:, 18].sum())), flush=True)
    b.close()
    del imu, pose, truth
    torch.cuda.empty_cache()
    return t0, t1


if __name__ == "__main__":
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
    T = int(sys.argv[2]) if len(sys.argv) > 2 else 1200
    stride = int(sys.argv[3]) if len(sys.argv) > 3 else 200
    print(torch.cuda.get_device_name(0))
    probe(N, T, stride, q.QEKF_FP64)
    probe(N, T, stride, q.QEKF_FP32)
