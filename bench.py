#!/usr/bin/env python
"""bench.py -- EKF filter-steps/s (propagate + update) on B200, the metric of BASELINE.json.

One "step" = one full pass of the hot path over one batch: every filter of the GPU replays the whole
60 s hover-and-descend landing scenario (12,000 IMU ticks at 200 Hz, 1,800 tag arrivals at 30 Hz, a
common 2 s tag dropout plus a private 1 s dropout per filter), FP64, noise generated in-kernel, RMSE/NEES
statistics accumulated on-chip and -- at N > 1 -- all-reduced over NCCL.  Weak scaling: every GPU owns
`--filters` (default 1,048,576) filters, BASELINE config 3 at N=1 and config 4 (8M filters) at N=8.

  python bench.py --gpus 1 --steps K --warmup W                 (this repo's CUDA path)
  python bench.py --impl reference --gpus N --steps K --warmup W (CPU restatement of the reference on
                                                                 the box's host cores; rank 0 only)

`value` is timed with CUDA events on the launching stream with every input resident in HBM; `e2e` is the
same metric through the C ABI with HOST buffers (pinned), the host->device copies of the scenario and the
device->host read of the statistics inside the timed region.

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (float64): the all-reduced
statistics and the state and covariance of a fixed sample of this rank's filters.  The inputs depend on the
arguments only, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from

# Floating-point operations executed per call by the structured code (FMA = 2), measured with an
# instrumented scalar type (tests/host_core hc_count_flops; tests/test_flop_count.py pins these numbers).
FLOPS = {(1, 1): (1398, 3425), (1, 0): (1398, 3911), (0, 1): (762, 2015), (0, 0): (762, 2231)}
# FP32 mode: K' = K + (B - K S) S^-1 per gain row: 2 x 36 FMA x (15 | 9) rows
JOSEPH_EXTRA_FLOPS = {1: 2 * 2 * 36 * 15, 0: 2 * 2 * 36 * 9}
# Algorithmic HBM bytes per filter-step in Monte-Carlo mode: state + covariance load and store
# (16 + 120 doubles each way) amortised over the ticks of one launch; the shared clean scenario is L2-resident.
STATE_BYTES = (16 + 120) * 8 * 2
# --dump-outputs: filters whose state and covariance are written (a seeded sample when the rank owns more); 7.6 MB in all
DUMP_FILTERS, DUMP_SEED = 4096, 20240


def bench_params(q, multirate=False, dynamic=False):
    """rotors.yaml noises (quad_state_estimation/config/relative_pose_EKF_rotors.yaml:13-19) with the
    benchmark rates of SURVEY.md section 8(d): 200 Hz update, 30 Hz tag, gated, single-rate, direct model."""
    p = q.default_params()
    p.update_freq, p.measurement_freq = 200.0, 30.0
    p.measurement_delay, p.measurement_delay_max, p.dyn_measurement_delay_offset = 0.030, 0.200, 0.005
    for i in range(3):
        p.Q_a[i], p.Q_w[i], p.Q_ab[i], p.Q_wb[i] = 0.0005, 0.00005, 5.0e-5, 5.0e-6
    p.R_r[0], p.R_r[1], p.R_r[2] = 0.015, 0.015, 0.020
    p.R_ang[0], p.R_ang[1], p.R_ang[2] = 0.0015, 0.0015, 0.04
    p.limit_measurement_freq = p.corner_margin_enbl = p.est_bias = p.direct_orien_method = 1
    p.multirate_ekf, p.dynamic_meas_delay = int(multirate), int(dynamic)
    return p


def bench_scenario(q, p):
    """The 60 s hover-and-descend landing; with delayed fusion the tag poses arrive 30 ms after capture."""
    from quadrotor_landing_b200 import scenario
    spec = scenario.default_spec()
    if p.multirate_ekf:
        spec.tag_latency_s = 0.030
    return scenario.generate(p, spec)


def bench_noise(q, first_global_id=0):
    n = q.default_noise()                      # sigma: accel .02, gyro .007, bias .05/.002, tag .02 m/.01 rad
    n.first_global_id = first_global_id
    n.dropout_k0, n.dropout_k1 = 5000, 5400    # t in [25, 27) s
    n.rand_dropout_len, n.rand_dropout_lo, n.rand_dropout_hi = 200, 400, 11600
    return n


def sweep_values(q, p, N, seed):
    """BASELINE config 5: every filter gets its own process / measurement noise and camera extrinsic ({field: [dim][N]})."""
    rng = np.random.default_rng(seed)
    base_q = np.array(list(p.Q_a) + list(p.Q_w) + list(p.Q_ab) + list(p.Q_wb))
    base_r = np.array(list(p.R_r) + list(p.R_ang))
    out = {q.PF_Q: base_q[:, None] * 10 ** rng.uniform(-1, 1, size=(12, N)),
           q.PF_R: base_r[:, None] * 10 ** rng.uniform(-1, 1, size=(6, N)),
           q.PF_R_V_CV: np.array(list(p.r_v_cv))[:, None] + rng.uniform(-0.02, 0.02, size=(3, N))}
    ang = rng.normal(scale=np.deg2rad(1.0) / 2, size=(3, N))                 # small rotation about a random axis
    dq = np.concatenate([ang, np.sqrt(1 - (ang ** 2).sum(axis=0))[None]])   # x, y, z, w
    qv = np.array(list(p.q_vc))
    x1, y1, z1, w1 = qv[:, None] * np.ones((4, N))
    x2, y2, z2, w2 = dq
    out[q.PF_Q_VC] = np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2, w1 * y2 + y1 * w2 + z1 * x2 - x1 * z2,
                               w1 * z2 + z1 * w2 + x1 * y2 - y1 * x2, w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2])
    return out


def apply_sweep(q, b, p, N, seed):
    vals = sweep_values(q, p, N, seed)
    for field, v in vals.items():
        b.set_filter_params(field, v)
    return vals


def facade_latency(seconds=20):
    """N = 1 drop-in: host latency of RelativePoseEKF::filter_update through include/relative_pose_ekf_gpu.hpp (one launch
    + one synchronisation per tick), measured by the C++ replay driver (tools/replay_driver.cpp) on the rotors preset,
    delayed fusion and single rate.  Outside every timed region; None when the driver binary is not built."""
    import subprocess
    import tempfile
    exe = os.path.join(ROOT, "quadrotor_landing_b200", "bin", "qekf_replay")
    preset = os.path.join(ROOT, "quadrotor_landing_b200", "presets", "rotors_sim.yaml")
    if not (os.path.exists(exe) and os.path.exists(preset)):
        return None
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, extra in (("delayed_fusion", []), ("single_rate", ["--single-rate"])):
            try:
                res = subprocess.run([exe, "--preset", preset, "--seconds", str(seconds), "--out", os.path.join(tmp, "t.csv")] + extra,
                                     stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
                ln = [l for l in res.stdout.splitlines() if "tick_latency_us" in l][-1]
                out[name] = json.loads(ln.split("qekf_replay: ", 1)[1])["tick_latency_us"]
            except Exception as e:  # noqa: BLE001 -- a diagnostic leg must not take the bench line down
                out[name] = {"error": str(e)[:120]}
    out["what"] = "per-tick host latency (us) of the C++ facade's filter_update, update_freq from the preset"
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                      "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) >= 7 and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(float(r[2]) for r in self.rows if len(r) >= 7)}


def cpu_streams(noise, scn, n_filters, first=0):
    """Explicit noisy streams for the CPU legs (same noise model and seeds, numpy restatement of the generator)."""
    from oracle import noise_np
    st = noise_np.synthesize(noise, scn.imu_clean, scn.tag_step, scn.tag_pose_clean, np.arange(first, first + n_filters))
    return np.ascontiguousarray(st["imu"]), np.ascontiguousarray(st["tag_pose"]), st["tag_valid"]


def cpu_replay(op, scn, streams, threads):
    """One bounded CPU step: the dense restatement of the reference (oracle/) replays the whole scenario for
    the sample's filters, OpenMP over filters.  `op`: oracle parameter struct.  Returns seconds."""
    from oracle import ekf_oracle as orc
    imu, pose, valid = streams
    ob = orc.Batch(op, imu.shape[2])
    t0 = time.perf_counter()
    ob.run(0, scn.T, imu, scn.tag_step, pose, scn.tag_stamp, valid, n_threads=threads)
    return time.perf_counter() - t0


CPU_NOTE = ("dense C restatement of relative_pose_EKF.cpp (oracle/ekf_oracle.c), gcc -O3, OpenMP over filters; "
            "the reference's own C++ needs Eigen >= 3.4, which is absent, so it cannot be built here")


def cpu_sample_filters(threads):
    return max(32, 32 * threads)


def run_reference(args):
    """--impl reference: the reference's own algorithm on the host cores, same scenario / noise / parameters.
    Rank 0 only; the other ranks exit without work.  Loads oracle/ libraries only -- not the product package."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import bench_ref
    op = bench_ref.params(args.multirate, args.dynamic_delay)
    scn = bench_ref.scenario(op, 0.030 if args.multirate else 0.0)
    threads = os.cpu_count() or 1
    sample = cpu_sample_filters(threads)
    streams = cpu_streams(bench_ref.noise(), scn, sample)
    for _ in range(args.warmup):
        cpu_replay(op, scn, streams, threads)
    times = [cpu_replay(op, scn, streams, threads) for _ in range(args.steps)]
    dt = float(np.mean(times))
    rate = sample * scn.T / dt
    line = {
        "impl": "reference", "metric": "EKF filter-steps/s (propagate+update)", "value": rate, "unit": "filter-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, scn, sample),
        "cpu_baseline": {"value": rate, "unit": "filter-steps/s", "cores": threads, "kind": "port",
                         "sample": "%d filters x %d ticks per step; %s" % (sample, scn.T, CPU_NOTE)},
        "e2e": {"value": rate, "unit": "filter-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def workload_config(args, scn, cpu_sample=None):
    mode = "single-rate"
    if getattr(args, "sweep", False):
        mode = "per-filter Q/R/camera-extrinsic sweep, " + mode
    if args.multirate:
        mode = mode.replace("single-rate", "") + "delayed-fusion (multirate_ekf, %s delay, 30 ms tag latency)" % (
            "dynamic" if args.dynamic_delay else "fixed 30 ms")
    cfg = {"workload": "Monte-Carlo replay of a 60 s hover-and-descend landing: %d filters per GPU x %d ticks "
                       "(200 Hz IMU, 30 Hz tag, 2 s common + 1 s per-filter tag dropout), %s direct-orientation "
                       "EKF, est_bias, rotors.yaml noises" % (args.filters, scn.T, mode),
           "filters_per_gpu": args.filters, "ticks": int(scn.T), "tag_arrivals": int(scn.M),
           "precision": "fp64" if args.precision == 64 else "fp32",
           "l2": "per-filter state (1.1 GB per 1M filters) is far larger than L2 and is re-read every step; the "
                 "shared clean scenario (0.7 MB) is L2-resident by design",
           "parallelism": "filters sharded over %d GPU(s), NCCL all-reduce of the statistics" % args.gpus}
    if cpu_sample is not None:
        # the CPU legs time a bounded SAMPLE of the same workload (same scenario, noise model and parameters)
        cfg["cpu_sample_filters"] = int(cpu_sample)
    return cfg


class Leg:
    """One workload variant on this rank's GPU: a handle, its device-resident inputs and the timed pass."""

    def __init__(self, q, torch, local, rank, world, n_filters, precision=64, multirate=False, dynamic=False, sweep=False,
                 no_stats=False, no_private_dropout=False):
        from quadrotor_landing_b200.sharded import shard_range
        self.q, self.torch, self.local, self.rank, self.world = q, torch, local, rank, world
        self.dev = torch.device("cuda", local)
        self.p = bench_params(q, multirate, dynamic)
        self.scn = bench_scenario(q, self.p)
        self.T, self.M, self.N = self.scn.T, self.scn.M, n_filters
        self.prec = q.QEKF_FP64 if precision == 64 else q.QEKF_FP32
        self.first_id, n_local = shard_range(n_filters * world, rank, world)     # every GPU owns n_filters filters
        assert n_local == n_filters
        self.noise = bench_noise(q, first_global_id=self.first_id)
        if no_private_dropout:
            self.noise.rand_dropout_len = 0
        self.stride = 200                              # one statistics sample per simulated second
        self.nb = self.T // self.stride
        self.b = q.BatchEKF(self.p, n_filters, device=local, precision=self.prec)
        self.stream = torch.cuda.current_stream()
        self.b.set_stream(self.stream.cuda_stream)
        if sweep:
            apply_sweep(q, self.b, self.p, n_filters, seed=1234 + rank)
        self.b.stats_configure(self.nb, self.stride if not no_stats else 10 ** 9)
        self.stats_dev = torch.zeros((self.nb, q.STAT_DIM), dtype=torch.float64, device=self.dev)
        scn, dev = self.scn, self.dev
        # device-resident inputs (the `value` leg)
        self._keep = [torch.tensor(scn.imu_clean, device=dev), torch.tensor(scn.tag_pose_clean, device=dev),
                      torch.tensor(scn.tag_stamp, device=dev), torch.tensor(scn.tag_step, dtype=torch.int32, device=dev),
                      torch.tensor(scn.truth, device=dev)]
        self.sh = self._shared(self._keep, 1)
        self.h_stats = np.zeros((self.nb, q.STAT_DIM))

    def _shared(self, t, on_device):
        sh = self.q.QekfSharedStreams()
        sh.T, sh.imu_clean, sh.M = self.T, t[0].data_ptr(), self.M
        sh.tag_pose_clean, sh.tag_stamp, sh.tag_step = t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr()
        sh.truth, sh.t_start, sh.on_device = t[4].data_ptr(), 0.0, on_device
        return sh

    def host_inputs(self):
        """pinned host copies of the shared scenario (the `e2e` leg); returns (shared view, bytes)"""
        torch, scn = self.torch, self.scn
        t = [torch.tensor(scn.imu_clean).pin_memory(), torch.tensor(scn.tag_pose_clean).pin_memory(),
             torch.tensor(scn.tag_stamp).pin_memory(), torch.tensor(scn.tag_step, dtype=torch.int32).pin_memory(),
             torch.tensor(scn.truth).pin_memory()]
        self._keep_host = t
        nbytes = sum(x.numel() * x.element_size() for x in t)
        return self._shared(t, 0), nbytes

    def one_step(self, shared, host_result):
        """One pass of the hot path: reset -> fused replay of all T ticks -> statistics (all-reduced at N>1)."""
        from quadrotor_landing_b200.sharded import all_reduce_stats
        b = self.b
        b.reset_filters()
        b.stats_reset()
        b.run_monte_carlo_device(shared, self.noise, 0, self.T)
        b.copy_stats_device(self.stats_dev.data_ptr())
        all_reduce_stats(self.stats_dev)                 # NCCL sum over the ranks (no-op at N=1)
        if host_result:
            self.h_stats[:] = self.stats_dev.cpu().numpy()

    def barrier(self, dist):
        if dist is not None:
            dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, shared, host_result, steps, dist):
        torch = self.torch
        self.barrier(dist)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(self.stream)
        for _ in range(steps):
            self.one_step(shared, host_result)
        e1.record(self.stream)
        self.barrier(dist)
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        if host_result:
            ms = max(ms, wall * 1e3)          # the host-visible time is what a caller of the C ABI sees
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def kernel_ms(self, reps=2):
        """The fused kernel alone (for the roofline): events around the launch only, on its stream."""
        torch, b = self.torch, self.b
        out = []
        for _ in range(reps):
            b.reset_filters(); b.stats_reset()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            b.run_monte_carlo_device(self.sh, self.noise, 0, self.T)
            e1.record(self.stream)
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return float(np.mean(out))

    def roofline(self, k_ms, n_pred, n_corr, peak):
        """Executed flops of one launch / kernel time against the self-measured FMA peak of the precision."""
        q, p = self.q, self.p
        fp, fc = FLOPS[(int(p.est_bias), int(p.direct_orien_method))]
        if self.prec == q.QEKF_FP32:
            fc += JOSEPH_EXTRA_FLOPS[int(p.est_bias)]      # the FP32 mode's refined gain (Joseph form), DESIGN.md section 7
        flops = n_pred * fp + n_corr * fc
        achieved = flops / (k_ms * 1e-3) / 1e12
        return {"bound": "fp64" if self.prec == q.QEKF_FP64 else "fp32", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                "peak_source": "self-measured FMA microbenchmark in this run (qekf_measure_fma_peak); "
                               "MEASURED_PEAKS.json has no CUDA-core figure",
                "kernel": "run_kernel", "kernel_ms": k_ms,
                "flops_per_filter_step": flops / (self.N * self.T),
                "work": {"prediction_steps": n_pred, "correction_steps": n_corr,
                         "flops_per_prediction": fp, "flops_per_correction": fc}}

    def parity(self, windows=3, width=64):
        """Max norm-relative deviation of this rank's filters from the oracle, on `windows` id windows (first, middle,
        last) of `width` filters: the device dumps the noise realisation of the window (qekf_synthesize_streams), the
        oracle replays it, and state / covariance after the last tick are compared with what the timed pass left on the
        device.  Outside any timed region."""
        from oracle import ekf_oracle as orc
        b, scn, N = self.b, self.scn, self.N
        op = orc.params_from(self.p)
        starts = sorted({0, max(0, (N - width) // 2), max(0, N - width)})[:windows]
        ex = eP = 0.0
        for f0 in starts:
            w = min(width, N - f0)
            st = b.synthesize_streams(scn, self.noise, f0, w)
            ob = orc.Batch(op, w)
            ob.run(0, self.T, st["imu"], st["tag_step"], st["tag_pose"], st["tag_stamp"], st["tag_valid"])
            xo, Po = ob.state(), ob.cov()
            xg, Pg = b.state(f0, w), b.cov(f0, w)
            ex = max(ex, float(np.max(np.abs(xg - xo)) / np.max(np.abs(xo))))
            eP = max(eP, float(np.max(np.abs(Pg - Po)) / np.max(np.abs(Po))))
        return {"state_norm_rel": ex, "cov_norm_rel": eP, "filters_checked": int(len(starts) * width),
                "windows_first_local_id": [int(x) for x in starts], "first_global_id": int(self.first_id),
                "tolerance": 1e-9 if self.prec == self.q.QEKF_FP64 else 1e-4,
                "against": "oracle/ekf_oracle.c replaying the device's dumped noise realisation (FP64)"}

    def outputs(self):
        """What the last pass left for its caller: the all-reduced statistics and the state / covariance of up to
        DUMP_FILTERS of this rank's filters (local ids drawn with a fixed seed), all float64."""
        b, N = self.b, self.N
        self.torch.cuda.synchronize()
        ids = np.arange(N) if N <= DUMP_FILTERS else np.sort(np.random.default_rng(DUMP_SEED).choice(N, DUMP_FILTERS, replace=False))
        return {"stats": self.stats_dev.cpu().numpy(), "filter_ids": ids.astype(np.float64),
                "state": np.concatenate([b.state(int(i), 1) for i in ids], axis=1),
                "cov": np.concatenate([b.cov(int(i), 1) for i in ids], axis=2)}

    def close(self):
        self.b.close()
        self._keep = None
        self.torch.cuda.empty_cache()


def run_leg(q, torch, nat, local, rank, world, dist, n_filters, steps, **kw):
    """A secondary workload variant, timed the same way as the main line (device-resident inputs), 1 warm-up pass."""
    leg = Leg(q, torch, local, rank, world, n_filters, **kw)
    leg.one_step(leg.sh, False)
    torch.cuda.synchronize()
    leg.b.step_counts(reset=True)
    sampler = ClockSampler(local)
    sampler.start()
    ms = leg.timed(leg.sh, False, steps, dist) / steps
    n_pred, n_corr = leg.b.step_counts(reset=True)
    clocks = sampler.stop()
    k_ms = leg.kernel_ms(1)
    peak = nat.measure_fma_peak(local, leg.prec)
    out = {"value": n_filters * leg.T * world / (ms * 1e-3), "unit": "filter-steps/s", "steps": steps, "ms_per_step": ms,
           "dtype": "f64" if leg.prec == q.QEKF_FP64 else "f32",
           "roofline": leg.roofline(k_ms, n_pred / steps, n_corr / steps, peak), "clocks": clocks}
    if kw.get("precision", 64) == 32:
        out["parity"] = leg.parity(windows=1)
    leg.close()
    return out


def run_ours(args):
    import torch
    import quadrotor_landing_b200 as q
    from quadrotor_landing_b200 import _native as nat

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL's own log (communicator init: "... nranks N ...") is evidence the driver wants, so it is not silenced: it
        # is on at INFO for the INIT subsystem unless the environment already says otherwise, and reaches stderr with
        # everything else that is written to fd 1 (claim_stdout).
        # (the GPU boxes run with NCCL_DEBUG=VERSION, which prints the banner only; INFO is a superset of it)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        dist.init_process_group("nccl", device_id=dev)
        if rank == 0:
            print("[bench] torch.distributed backend nccl: world size %d (one rank per GPU), NCCL %s" % (
                dist.get_world_size(), ".".join(str(v) for v in torch.cuda.nccl.version())), file=sys.stderr, flush=True)

    N = args.filters
    if args.scaling == "strong":
        N = args.filters // world                    # the job's total stays `--filters`
    main = Leg(q, torch, local, rank, world, N, precision=args.precision, multirate=args.multirate, dynamic=args.dynamic_delay,
               sweep=args.sweep, no_stats=args.no_stats, no_private_dropout=args.no_private_dropout)
    b, T, stream = main.b, main.T, main.stream
    hs, h2d = main.host_inputs()

    for _ in range(max(args.warmup, 3)):
        main.one_step(main.sh, False)
    torch.cuda.synchronize()
    b.step_counts(reset=True)
    l0 = b.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    ms_total = main.timed(main.sh, False, args.steps, dist)
    launches = b.launch_count - l0
    n_pred, n_corr = b.step_counts(reset=True)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in main.outputs().items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    k_ms = main.kernel_ms(2)
    clocks = sampler.stop()
    main.one_step(hs, True)                              # warm the host path (staging slab allocation)
    e2e_steps = min(args.steps, 8)
    e2e_ms = main.timed(hs, True, e2e_steps, dist)

    # ---- outside the timed regions: parity of this rank's filters against the oracle (max over ranks) ----
    parity = None
    if not args.no_parity:
        parity = main.parity()
        if dist is not None:
            t = torch.tensor([parity["state_norm_rel"], parity["cov_norm_rel"]], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            parity["state_norm_rel"], parity["cov_norm_rel"] = float(t[0].item()), float(t[1].item())
            parity["ranks_checked"] = world
            parity["filters_checked"] *= world
    h_stats = main.h_stats.copy()
    peak = nat.measure_fma_peak(local, main.prec)
    p, scn, prec = main.p, main.scn, main.prec
    main.close()

    # ---- secondary workloads of BASELINE.json (configs 3 FP32, delayed fusion, config 5), same timing method ----
    legs = None
    default_main = (args.precision == 64 and not args.multirate and not args.sweep and not args.no_stats
                    and not args.no_private_dropout)
    if not args.no_legs and default_main:
        legs = {}
        for name, kw in (("fp32", dict(precision=32)),
                         ("delayed_fusion_fixed", dict(multirate=True)),
                         ("delayed_fusion_dynamic", dict(multirate=True, dynamic=True)),
                         ("config5_sweep_delayed_dynamic", dict(multirate=True, dynamic=True, sweep=True))):
            legs[name] = run_leg(q, torch, nat, local, rank, world, dist, N, args.leg_steps, **kw)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    ms_per_step = ms_total / args.steps
    steps_per_pass = N * T * world
    value = steps_per_pass / (ms_per_step * 1e-3)
    e2e_value = steps_per_pass / (e2e_ms / e2e_steps * 1e-3)
    roof = main.roofline(k_ms, n_pred / args.steps, n_corr / args.steps, peak)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # measured DRAM traffic of this exact launch shape, if an ncu capture of it is on file (profiles/traffic.json)
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "%s|%s|%d|%d" % ("multirate" if args.multirate else "single-rate", "fp64" if prec == q.QEKF_FP64 else "fp32", N, T)
        if key in tj:
            traffic = float(tj[key]["dram_bytes_read"] + tj[key]["dram_bytes_write"])
            traffic_src = tj[key]["source"].split(":")[0]
    except Exception:
        pass
    roof["traffic"], roof["traffic_unit"], roof["traffic_source"] = traffic, "DRAM bytes per launch (ncu)", traffic_src
    k_t = k_ms * 1e-3
    hbm_bytes = N * STATE_BYTES * (1 if prec == q.QEKF_FP64 else 0.5) + h2d
    threads = os.cpu_count() or 1
    sample = cpu_sample_filters(threads)
    line = {
        "metric": "EKF filter-steps/s (propagate+update)", "value": value, "unit": "filter-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64" if prec == q.QEKF_FP64 else "f32", "data": "synthetic",
        "config": workload_config(args, scn, sample if world == 1 and not args.no_cpu_baseline else None),
        "e2e": {"value": e2e_value, "unit": "filter-steps/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(h_stats.nbytes), "steps": e2e_steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "roofline_hbm": {"bound": "hbm", "achieved": hbm_bytes / k_t / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": hbm_bytes / k_t / 1e9 / hbm_peak, "traffic": traffic,
                         "algorithmic_bytes": hbm_bytes,
                         "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
        "stats": {"rmse_pos_m_final": float(np.sqrt(h_stats[-1, 19] / max(h_stats[-1, 16], 1) / 3)),
                  "mean_nees_final": float(h_stats[-1, 15] / max(h_stats[-1, 16], 1)),
                  "samples_final": float(h_stats[-1, 16]), "diverged_total": float(h_stats[:, 18].sum())},
    }
    if args.scaling == "strong":
        line["config"]["filters_per_gpu"] = N
        line["config"]["filters_total"] = N * world
    if parity is not None:
        line["parity"] = parity
    if legs is not None:
        line["legs"] = legs
    if dist is not None:
        line["comm"] = {"backend": "nccl", "nranks": int(dist.get_world_size()),
                        "nccl_version": ".".join(str(v) for v in torch.cuda.nccl.version()),
                        "collective": "all_reduce(sum, f64) of the [%d][%d] statistics, once per pass" % (h_stats.shape[0], h_stats.shape[1])}
    if world == 1 and not args.no_cpu_baseline:
        from oracle import ekf_oracle as orc
        op = orc.params_from(p)
        streams = cpu_streams(bench_noise(q), scn, sample)
        cpu_replay(op, scn, streams, threads)
        reps = [cpu_replay(op, scn, streams, threads) for _ in range(3)]
        dt = float(np.mean(reps))
        one = tuple(np.ascontiguousarray(a[..., :32]) for a in streams)
        dt1 = cpu_replay(op, scn, one, 1)
        line["cpu_baseline"] = {"value": sample * T / dt, "unit": "filter-steps/s", "cores": threads, "kind": "port",
                                "sample": "%d filters x %d ticks of the same workload, %.1f s per replay; %s"
                                          % (sample, T, dt, CPU_NOTE),
                                "single_thread": {"value": 32 * T / dt1, "unit": "filter-steps/s", "cores": 1,
                                                  "sample": "32 filters x %d ticks, %.1f s" % (T, dt1)}}
    if world == 1 and default_main:
        lat = facade_latency()
        if lat:
            line["facade_latency"] = lat
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


_JSON_FD = None


def claim_stdout():
    """stdout carries exactly ONE JSON line.  Everything else any library writes to file descriptor 1 (NCCL's version
    banner and its INFO log, which is evidence the driver wants and is therefore left on) is sent to stderr: fd 1 is
    pointed at fd 2 for the rest of the process and the JSON line is written to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--filters", type=int, default=1 << 20, help="filters per GPU")
    ap.add_argument("--precision", type=int, default=64, choices=[64, 32])
    ap.add_argument("--multirate", action="store_true", help="delayed-measurement fusion (multirate_ekf) workload")
    ap.add_argument("--dynamic-delay", action="store_true", help="with --multirate: stamp-derived measurement delay")
    ap.add_argument("--sweep", action="store_true",
                    help="BASELINE config 5: per-filter Q / R within x[0.1, 10] of the preset (log-uniform), camera extrinsic "
                         "+-2 cm / +-1 deg (use with --multirate --dynamic-delay)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of three id windows after the timed passes")
    ap.add_argument("--no-legs", action="store_true", help="skip the secondary workloads (FP32, delayed fusion, config 5)")
    ap.add_argument("--leg-steps", type=int, default=3)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --filters per GPU (default); strong: --filters in total, split over the ranks")
    ap.add_argument("--no-stats", action="store_true", help="diagnostic: never sample statistics")
    ap.add_argument("--no-private-dropout", action="store_true", help="diagnostic: drop the per-filter dropout window")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy: statistics, filter_ids and the "
                         "state / covariance of those filters (rank 0's)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
