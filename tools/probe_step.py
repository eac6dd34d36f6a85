"""Cost of the per-tick step (qekf_step / BatchEKF.step) against the two other ways to advance a batch by one tick.

For N filters (est_bias = 1, direct = 1, the benchmark's model), FP64 / FP32, single rate / fixed delay / dynamic delay:
  step      : step-kernel time from CUDA events over >= --steps steps after warm-up (replays of a captured CUDA
              graph of 120 steps), outputs x and cov requested;
              filter-steps/s; bytes moved per step from the layout and the bandwidth against 7.7 TB/s;
              predictions per filter-tick (qekf_step_counts); CTA size from --blocks (QEKF_STEP_BLOCK)
  today     : qekf_run with n_steps = 1 on device streams plus the state / covariance accessors (host copies)
  replay    : the fused replay's per-tick cost over --replay-ticks ticks of device streams (the open-loop lower reference)
Prints the card and its power limit first, then one JSON line per configuration.

  python tools/probe_step.py [--sizes 65536 262144 1048576] [--steps 1000]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import quadrotor_landing_b200 as q  # noqa: E402
from quadrotor_landing_b200 import scenario  # noqa: E402
from streams_np import rotors_params  # noqa: E402

DEV = torch.device("cuda", 0)
MODES = {"single": (False, False), "fixed": (True, False), "dynamic": (True, True)}
HBM = 7.7e12


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip()
    return out.splitlines()[0] if out else torch.cuda.get_device_name(0)


def inputs(scn, N, pool, g):
    """`pool` distinct IMU samples and tag poses per filter (cycled), drawn around the clean scenario's hover."""
    f64 = dict(dtype=torch.float64, device=DEV)
    imu = torch.as_tensor(scn.imu_clean[100], **f64)[None, :, None] + torch.cat(
        [0.02 * torch.randn((pool, 3, N), generator=g, **f64), 0.007 * torch.randn((pool, 3, N), generator=g, **f64)], 1)
    m = int(np.searchsorted(scn.tag_step, 100))
    tag = torch.zeros((pool, 8, N), **f64)
    tag[:, 0:7] = torch.as_tensor(scn.tag_pose_clean[m], **f64)[None, :, None]
    tag[:, 0:3] += 0.02 * torch.randn((pool, 3, N), generator=g, **f64)
    return imu.contiguous(), tag.contiguous()


def bytes_per_step(N, tsize, nstate, mr, preds, corr_rate, arrive_rate):
    """Bytes a step moves, from the layout: state in and out, inputs, the x / cov outputs (double), and in delayed-fusion
    mode the ring push, the history counters and, per correcting tick, the checkpoint store and the ring replay."""
    npk = nstate * (nstate + 1) // 2
    st = (16 + npk) * tsize
    b = 2 * st + 2 * 8 + 3 * tsize * 2 + 6 * 8         # x / P, flags / upds, accel, imu
    b += (16 + npk) * 8                                    # outputs x and cov
    b += arrive_rate * (1 + 8 * 8 + 8 * 8)                 # arrived, tag, latched pose (bytes per filter per tick)
    if mr:
        b += 6 * tsize + 3 * 4 * 2                         # ring push, nh / hpos / hlen
        b += corr_rate * st + (preds - 1) * 6 * tsize      # checkpoint store, ring reads of the replayed entries
    return N * b


def time_steps(b, p, imu, tag, t0, window, reps, pool, has, stamp, x, cov, stream):
    """Kernel time per step: `window` steps captured into a CUDA graph (so the host's call overhead is not measured),
    replayed `reps` times; each arrival of the window has its own tag with its capture stamp."""
    arr = [k for k in range(t0, t0 + window) if has(k)]
    tags = tag[torch.arange(len(arr), device=DEV) % pool].clone()
    for j, k in enumerate(arr):
        tags[j, 7] = stamp(k)
    ones = torch.ones(b.N, dtype=torch.uint8, device=DEV)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        j = 0
        for k in range(t0, t0 + window):
            h = has(k)
            b.step(k / p.update_freq, imu[k % pool], tags[j] if h else None, ones if h else None, x=x, cov=cov)
            j += 1 if h else 0
    with torch.cuda.stream(stream):
        g.replay()                     # warm-up
        b.step_counts(reset=True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(reps):
            g.replay()
        ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / 1e3 / (window * reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[65536, 262144, 1048576])
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--blocks", type=int, nargs="+", default=[32, 64, 128])
    ap.add_argument("--replay-ticks", type=int, default=200)
    ap.add_argument("--today-ticks", type=int, default=5)
    a = ap.parse_args()
    print("card: %s" % card(), flush=True)
    g = torch.Generator(device=DEV)
    g.manual_seed(1)
    for N in a.sizes:
        for prec in (64, 32):
            for mode in MODES:
                mr, dyn = MODES[mode]
                p = rotors_params(q.default_params(), multirate=mr, dynamic_delay=dyn)
                spec = scenario.default_spec()
                spec.tag_latency_s = 0.030
                scn = scenario.generate(p, spec)
                pool = 16
                imu, tag = inputs(scn, N, pool, g)
                upm = int(p.update_freq / p.measurement_freq)
                has = lambda k: k % upm == 0
                rec = dict(N=N, prec=prec, mode=mode)
                x = torch.zeros((16, N), dtype=torch.float64, device=DEV)
                cov = torch.zeros((120, N), dtype=torch.float64, device=DEV)
                stamp = lambda k: k / p.update_freq - 0.030       # capture stamp: 30 ms before the tick
                side = torch.cuda.Stream()
                for blk in a.blocks:
                    os.environ["QEKF_STEP_BLOCK"] = str(blk)
                    b = q.BatchEKF(p, N, 0, prec)
                    b.set_stream(side.cuda_stream)
                    ones = torch.ones(N, dtype=torch.uint8, device=DEV)
                    with torch.cuda.stream(side):
                        for k in range(200):
                            if has(k):
                                tag[k % pool, 7] = stamp(k)
                            b.step(k / p.update_freq, imu[k % pool], tag[k % pool] if has(k) else None,
                                   ones if has(k) else None)
                    torch.cuda.synchronize()
                    window = 10 * upm * 2
                    reps = -(-a.steps // window)
                    t = time_steps(b, p, imu, tag, 200, window, reps, pool, has, stamp, x, cov, side)
                    npred, ncorr = b.step_counts()
                    rec["step_s_block%d" % blk] = t
                    rec["preds_per_tick"] = npred / (N * window * reps)
                    rec["corr_per_tick"] = ncorr / (N * window * reps)
                    b.close()
                os.environ.pop("QEKF_STEP_BLOCK", None)
                best = min(a.blocks, key=lambda k: rec["step_s_block%d" % k])
                t = rec["step_s_block%d" % best]
                by = bytes_per_step(N, prec // 8, 15, mr, rec["preds_per_tick"], rec["corr_per_tick"], 1.0 / upm)
                rec.update(best_block=best, step_s=t, filter_steps_per_s=N / t, bytes_per_step=by,
                           bandwidth_TBps=by / t / 1e12, share_of_7p7=by / t / HBM)
                # today: one-tick replays on device streams + the host accessors
                b = q.BatchEKF(p, N, 0, prec)
                T = a.replay_ticks
                dimu = imu[torch.arange(T) % pool].contiguous()
                steps = np.arange(0, T, upm, dtype=np.int32)
                M = len(steps)
                dpose = tag[torch.as_tensor(steps) % pool, 0:7].contiguous()
                dstamp = torch.as_tensor(steps / p.update_freq - 0.030, dtype=torch.float64, device=DEV)
                dstep = torch.as_tensor(steps, device=DEV)
                args = (T, dimu.data_ptr(), M, dstep.data_ptr(), dpose.data_ptr(), dstamp.data_ptr())
                b.run_device(0, 50, *args)
                b.sync()
                t1 = time.perf_counter()
                for k in range(50, 50 + a.today_ticks):
                    b.run_device(k, 1, *args)
                    b.state(); b.cov()
                rec["today_s"] = (time.perf_counter() - t1) / a.today_ticks
                # the fused replay of the remaining ticks, per tick
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                b.set_stream(torch.cuda.current_stream().cuda_stream)
                k0 = 50 + a.today_ticks
                ev0.record()
                b.run_device(k0, T - k0, *args)
                ev1.record()
                torch.cuda.synchronize()
                rec["replay_s_per_tick"] = ev0.elapsed_time(ev1) / 1e3 / (T - k0)
                b.close()
                del dimu, dpose
                print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
