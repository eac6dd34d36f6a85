"""GPU tier of qekf_step / BatchEKF.step, the per-tick step with device-resident per-filter inputs and outputs.

1. Open-loop equivalence: stepping tick by tick through explicit streams equals qekf_run over the same streams, for
   FP64 / FP32 x est_bias x direct x {single rate, fixed delay, dynamic delay} x {with, without} per-filter parameters,
   at N = 4,096 and (a subset) N = 100,003; outputs equal the accessors every 500th step.
2. Closed loop: N = 4,096 simulated vehicles whose PD descent controller acts on the step's state output; 64 of them
   replayed through the oracle tick by tick with the inputs the loop produced; a perturbed tag changes later IMU inputs.
3. Outputs: each pointer optional, cov_out in the accessor's triangle order, FP32 outputs equal the FP32 accessors.
4. CUDA graph: 50 captured steps replayed with inputs refreshed in place equal eager stepping bit for bit.
5. Hand-over: step -> qekf_run -> step, export -> import -> step, Monte-Carlo after steps, qekf_step_counts.
6. Interface: bad arguments, set_mapping(2/3), per-filter parameters."""
import numpy as np
import pytest
import torch

import quadrotor_landing_b200 as q
from oracle import ekf_oracle as orc
from quadrotor_landing_b200 import _native as nat
from quadrotor_landing_b200 import scenario
from streams_np import norm_rel, rotors_params

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
MODES = {"single": (False, False), "fixed": (True, False), "dynamic": (True, True)}
# variants whose step and replay kernels may round differently in the last bit (checked to 1e-12 norm-relative):
# none so far
LAST_BIT = set()


def make_params(est_bias=1, direct=1, mode="single"):
    mr, dyn = MODES[mode]
    return rotors_params(q.default_params(), est_bias=est_bias, direct=direct, multirate=mr, dynamic_delay=dyn)


def scn_of(p, seconds=6.0, latency=0.036):
    spec = scenario.default_spec()
    spec.duration_s, spec.hover_s = seconds, 1.5
    spec.tag_latency_s = latency
    return scenario.generate(p, spec)


def device_streams(scn, N, T, seed):
    """Per-filter explicit streams on the GPU (qekf_streams layout), noise from a seeded torch generator; tag_valid with
    a common dropout and a private dropout per filter."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    sel = scn.tag_step < T
    steps = scn.tag_step[sel]
    M = int(len(steps))
    imu = torch.as_tensor(scn.imu_clean[:T], device=DEV)[:, :, None].repeat(1, 1, N)
    bias = torch.randn((1, 6, N), generator=g, device=DEV, dtype=torch.float64) * torch.tensor(
        [0.05] * 3 + [0.002] * 3, device=DEV, dtype=torch.float64)[None, :, None]
    sig = torch.tensor([0.02] * 3 + [0.007] * 3, device=DEV, dtype=torch.float64)[None, :, None]
    imu = (imu + bias + sig * torch.randn((T, 6, N), generator=g, device=DEV, dtype=torch.float64)).contiguous()
    pose = torch.as_tensor(scn.tag_pose_clean[sel], device=DEV)[:, :, None].repeat(1, 1, N)
    pose[:, 0:3] += 0.02 * torch.randn((M, 3, N), generator=g, device=DEV, dtype=torch.float64)
    pose[:, 3:7] += 0.004 * torch.randn((M, 4, N), generator=g, device=DEV, dtype=torch.float64)
    pose[:, 3:7] /= pose[:, 3:7].norm(dim=1, keepdim=True)
    pose = pose.contiguous()
    st = torch.as_tensor(steps, device=DEV)
    valid = torch.ones((M, N), dtype=torch.uint8, device=DEV)
    valid[(st >= T // 3) & (st < T // 3 + 60)] = 0
    start = torch.randint(0, max(T - 80, 1), (N,), generator=g, device=DEV)
    valid[(st[:, None] >= start[None]) & (st[:, None] < start[None] + 80)] = 0
    return dict(T=T, M=M, imu=imu, tag_step=torch.as_tensor(steps.astype(np.int32), device=DEV), tag_pose=pose,
                tag_stamp=torch.as_tensor(scn.tag_stamp[sel], device=DEV).contiguous(), tag_valid=valid.contiguous(),
                steps=steps)


def run_streams(b, ds, k0, n):
    b.run_device(k0, n, ds["T"], ds["imu"].data_ptr(), ds["M"], ds["tag_step"].data_ptr(), ds["tag_pose"].data_ptr(),
                 ds["tag_stamp"].data_ptr(), ds["tag_valid"].data_ptr())
    b.sync()


class Stepper:
    """Feeds the streams' tick k to BatchEKF.step as a closed-loop caller would: imu row, arrival flags, [8][N] tag."""

    def __init__(self, b, ds, p):
        self.b, self.ds, self.p = b, ds, p
        N = b.N
        self.arrived = torch.zeros(N, dtype=torch.uint8, device=DEV)
        self.tag = torch.zeros((8, N), dtype=torch.float64, device=DEV)
        self.m = 0
        self.x = torch.zeros((16, N), dtype=torch.float64, device=DEV)
        self.cov = torch.zeros((b.n * (b.n + 1) // 2, N), dtype=torch.float64, device=DEV)
        self.aux = torch.zeros((11, N), dtype=torch.float64, device=DEV)
        self.flags = torch.zeros((6, N), dtype=torch.int32, device=DEV)

    def inputs(self, k):
        ds = self.ds
        self.m = int(np.searchsorted(ds["steps"], k))
        if self.m < ds["M"] and ds["steps"][self.m] == k:
            self.arrived.copy_(ds["tag_valid"][self.m])
            self.tag[0:7].copy_(ds["tag_pose"][self.m])
            self.tag[7].fill_(float(ds["tag_stamp"][self.m]))
            return True
        return False

    def step(self, k, outputs=True):
        has = self.inputs(k)
        outs = dict(x=self.x, cov=self.cov, aux=self.aux, flags=self.flags) if outputs else {}
        self.b.step(k / self.p.update_freq, self.ds["imu"][k], self.tag if has else None, self.arrived if has else None,
                    **outs)

    def run(self, k0, n, check_every=500):
        for k in range(k0, k0 + n):
            self.step(k)
            if check_every and (k + 1) % check_every == 0:
                torch.cuda.synchronize()
                self.check_outputs()

    def check_outputs(self):
        b = self.b
        assert np.array_equal(self.x.cpu().numpy(), b.state())
        assert np.array_equal(packed_of(b.cov()), self.cov.cpu().numpy())
        assert np.array_equal(self.aux.cpu().numpy(), b.aux())
        assert np.array_equal(self.flags.cpu().numpy(), b.flags())


def packed_of(P):
    n = P.shape[0]
    return np.stack([P[a, c] for a in range(n) for c in range(a, n)])


def snapshot(b):
    return [b.state(), b.cov(), b.aux(), b.flags()]


def assert_equal_or_last_bit(a, b, variant):
    for k, (u, v) in enumerate(zip(a, b)):
        if k == 3 or variant not in LAST_BIT:
            assert np.array_equal(u, v), (variant, k, norm_rel(u, v))
        else:
            assert norm_rel(u, v) <= 1e-12, (variant, k, norm_rel(u, v))


def sweep(b, p, mode, N, seed):
    rng = np.random.default_rng(seed)
    qv = np.array(list(p.Q_a) + list(p.Q_w) + list(p.Q_ab) + list(p.Q_wb))[:, None] * rng.uniform(0.5, 2.0, (1, N))
    b.set_filter_params(q.PF_Q, qv)
    if mode != "single":
        b.set_filter_params(q.PF_DELAY, np.stack([rng.uniform(0.015, 0.045, N), rng.uniform(0.0, 0.01, N)]))


def open_loop_case(prec, est_bias, direct, mode, pf, N, T):
    p = make_params(est_bias, direct, mode)
    ds = device_streams(scn_of(p), N, T, seed=100 + est_bias + 2 * direct)
    ref, b = q.BatchEKF(p, N, 0, prec), q.BatchEKF(p, N, 0, prec)
    if pf:
        sweep(ref, p, mode, N, 3)
        sweep(b, p, mode, N, 3)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    run_streams(ref, ds, 0, T)
    s = Stepper(b, ds, p)
    s.run(0, T)
    torch.cuda.synchronize()
    variant = (prec, est_bias, direct, mode, pf)
    assert_equal_or_last_bit(snapshot(b), snapshot(ref), variant)
    assert b.flags()[0].mean() > 0.99
    ref.close(); b.close()


@pytest.mark.parametrize("pf", [False, True], ids=["shared", "perfilter"])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("est_bias,direct", [(1, 1), (1, 0), (0, 1), (0, 0)])
@pytest.mark.parametrize("prec", [64, 32], ids=["fp64", "fp32"])
def test_open_loop_equals_replay(prec, est_bias, direct, mode, pf):
    open_loop_case(prec, est_bias, direct, mode, pf, 4096, 1000)


@pytest.mark.parametrize("prec,mode,pf", [(64, "single", False), (64, "dynamic", True), (32, "fixed", False),
                                          (32, "dynamic", True)])
def test_open_loop_equals_replay_ragged(prec, mode, pf):
    open_loop_case(prec, 1, 1, mode, pf, 100003, 520)


# ---- closed loop ----------------------------------------------------------------------------------------------------

def closed_loop(p, N, T, perturb=None, seed=5):
    """N vehicles descending on the tag: the clean scenario is the nominal trajectory, each vehicle deviates from it by
    d (position) / w (velocity) under a PD controller acting on its filter's estimate.  IMU and tag are synthesised from
    the nominal + deviation with seeded noise; per-vehicle detection dropouts and latency.  Returns the recorded inputs
    and outputs of the first 64 vehicles."""
    scn = scn_of(p, seconds=T / p.update_freq + 0.5, latency=0.03)
    dt = 1.0 / p.update_freq
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    f64 = dict(dtype=torch.float64, device=DEV)
    b = q.BatchEKF(p, N, 0)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    d = 0.3 * torch.randn((3, N), generator=g, **f64)
    w = torch.zeros((3, N), **f64)
    bias = torch.cat([0.05 * torch.randn((3, N), generator=g, **f64), 0.002 * torch.randn((3, N), generator=g, **f64)])
    latency = 0.02 * torch.rand(N, generator=g, **f64)
    drop_p = 0.3 * torch.rand(N, generator=g, **f64)
    x = torch.zeros((16, N), **f64)
    flags = torch.zeros((6, N), dtype=torch.int32, device=DEV)
    imu = torch.zeros((6, N), **f64)
    tag = torch.zeros((8, N), **f64)
    arrived = torch.zeros(N, dtype=torch.uint8, device=DEV)
    rec = dict(imu=[], tag=[], arrived=[], x=[], flags=[])
    steps = {int(k): m for m, k in enumerate(scn.tag_step)}
    first = True
    for k in range(T):
        # controller on the estimate (only once the filter is initialised): drive the estimated deviation from the
        # nominal relative position to zero
        r_nom = torch.as_tensor(scn.truth[k][0:3], **f64)[:, None]
        init = flags[0:1].to(torch.float64)
        a_cmd = init * torch.clamp(-0.8 * (x[0:3] - r_nom) - 1.2 * (x[3:6] - torch.as_tensor(scn.truth[k][3:6], **f64)[:, None]),
                                   -0.5, 0.5)
        w += a_cmd * dt
        d += w * dt
        imu.copy_(torch.as_tensor(scn.imu_clean[k], **f64)[:, None] + bias)
        imu[0:3] += a_cmd + 0.02 * torch.randn((3, N), generator=g, **f64)
        imu[3:6] += 0.007 * torch.randn((3, N), generator=g, **f64)
        has = k in steps
        if has:
            m = steps[k]
            tag[0:7] = torch.as_tensor(scn.tag_pose_clean[m], **f64)[:, None]
            tag[0:3] += d + 0.02 * torch.randn((3, N), generator=g, **f64)
            tag[7] = float(scn.tag_stamp[m]) - latency
            arrived.copy_((torch.rand(N, generator=g, **f64) >= drop_p).to(torch.uint8))
            if perturb is not None and first:
                tag[0, perturb] += 0.05
            first = False
        b.step(k * dt, imu, tag if has else None, arrived if has else None, x=x, flags=flags)
        rec["imu"].append(imu[:, :64].cpu().numpy())
        rec["tag"].append(tag[:, :64].cpu().numpy() if has else None)
        rec["arrived"].append(arrived[:64].cpu().numpy() if has else None)
        rec["x"].append(x[:, :64].cpu().numpy())
        rec["flags"].append(flags[:, :64].cpu().numpy())
    cov = b.cov(0, 64)
    b.close()
    return rec, cov


def test_closed_loop_matches_oracle():
    p = make_params(1, 1, "dynamic")
    N, T = 4096, 700
    rec, cov = closed_loop(p, N, T)
    op = orc.params_from(p)
    filters = [orc.Filter(op) for _ in range(64)]
    worst = 0.0
    for k in range(T):
        for i in range(64):
            f = filters[i]
            if rec["tag"][k] is not None and rec["arrived"][k][i]:
                t = rec["tag"][k]
                f.set_tag(t[0:3, i], t[3:7, i], t[7, i])
            f.set_imu(rec["imu"][k][0:3, i], rec["imu"][k][3:6, i])
            f.filter_update(k / p.update_freq)
            fl = f.flags()
            assert rec["flags"][k][0, i] == fl["state_initialized"] and rec["flags"][k][4, i] == fl["upds_since_correction"]
            if fl["state_initialized"]:
                e = norm_rel(rec["x"][k][:, i], f.state())
                worst = max(worst, e)
                assert e < 1e-9, (k, i, e)
    for i in range(64):
        assert norm_rel(cov[:, :, i], filters[i].cov()) < 1e-9
    assert rec["flags"][-1][0].all()
    print("closed loop, 64 vehicles x %d ticks against the oracle: worst state error %.2e" % (T, worst))


def test_closed_loop_is_closed():
    """A different first tag for vehicle 7 changes its estimate, hence its controller's commands and its later IMU
    inputs; the other vehicles see exactly the same inputs."""
    p = make_params(1, 1, "single")
    a, _ = closed_loop(p, 256, 120)
    b, _ = closed_loop(p, 256, 120, perturb=7)
    ia, ib = np.stack(a["imu"]), np.stack(b["imu"])
    assert not np.array_equal(ia[:, :, 7], ib[:, :, 7])
    others = [i for i in range(64) if i != 7]
    assert np.array_equal(ia[:, :, others], ib[:, :, others])


# ---- outputs ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("prec", [64, 32], ids=["fp64", "fp32"])
def test_outputs_optional_and_in_accessor_layout(prec):
    p = make_params(1, 0, "fixed")
    N, T = 1000, 300
    ds = device_streams(scn_of(p), N, T, seed=9)
    b = q.BatchEKF(p, N, 0, prec)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    s = Stepper(b, ds, p)
    for k in range(T):
        s.step(k, outputs=(k % 7 == 0))
    # each output alone
    for name in ("x", "cov", "aux", "flags"):
        s.x.fill_(-1); s.cov.fill_(-1); s.aux.fill_(-1); s.flags.fill_(-1)
        before = [t.clone() for t in (s.x, s.cov, s.aux, s.flags)]
        k = T
        out = dict(x=s.x, cov=s.cov, aux=s.aux, flags=s.flags)
        b.step(k / p.update_freq, ds["imu"][-1], None, None, **{name: out[name]})
        torch.cuda.synchronize()
        T += 1
        for nm, t, t0 in zip(("x", "cov", "aux", "flags"), (s.x, s.cov, s.aux, s.flags), before):
            if nm != name:
                assert torch.equal(t, t0)
        if name == "x":
            assert np.array_equal(s.x.cpu().numpy(), b.state())
        elif name == "cov":
            assert np.array_equal(s.cov.cpu().numpy(), packed_of(b.cov()))
        elif name == "aux":
            assert np.array_equal(s.aux.cpu().numpy(), b.aux())
        else:
            assert np.array_equal(s.flags.cpu().numpy(), b.flags())
    b.close()


# ---- CUDA graph -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", ["single", "dynamic"])
def test_cuda_graph_capture_equals_eager(mode):
    p = make_params(1, 1, mode)
    N, K, T = 4096, 50, 400
    ds = device_streams(scn_of(p), N, T, seed=13)
    eager, graph = q.BatchEKF(p, N, 0), q.BatchEKF(p, N, 0)
    side = torch.cuda.Stream()
    graph.set_stream(side.cuda_stream)
    # warm both up to past the first detections
    for b in (eager, graph):
        run_streams(b, ds, 0, 100)
    eager.set_stream(torch.cuda.current_stream().cuda_stream)
    # the graph's inputs: K ticks of imu / arrived / tag, refreshed in place before every replay
    imu = torch.zeros((K, 6, N), dtype=torch.float64, device=DEV)
    arrived = torch.zeros((K, N), dtype=torch.uint8, device=DEV)
    tag = torch.zeros((K, 8, N), dtype=torch.float64, device=DEV)
    x = torch.zeros((16, N), dtype=torch.float64, device=DEV)
    cov = torch.zeros((120, N), dtype=torch.float64, device=DEV)
    t0 = 100

    def fill(k0):
        imu.copy_(ds["imu"][k0:k0 + K])
        arrived.zero_()
        for j in range(K):
            m = int(np.searchsorted(ds["steps"], k0 + j))
            if m < ds["M"] and ds["steps"][m] == k0 + j:
                arrived[j].copy_(ds["tag_valid"][m])
                tag[j, 0:7].copy_(ds["tag_pose"][m])
                tag[j, 7].fill_(float(ds["tag_stamp"][m]))

    g = torch.cuda.CUDAGraph()
    fill(t0)
    torch.cuda.synchronize()
    # the tick times are baked into the graph: the captured window is replayed over the same ticks on a fresh copy of
    # the state each time (export / import), and eager stepping over those ticks is the reference
    blob = graph.export_state()
    with torch.cuda.graph(g, stream=side):
        for j in range(K):
            graph.step((t0 + j) / p.update_freq, imu[j], tag[j], arrived[j], x=x, cov=cov)
    torch.cuda.synchronize()
    graph.import_state(blob)
    for rep in range(2):
        fill(t0)            # refreshed in place: same values, new writes
        g.replay()
        torch.cuda.synchronize()
        got = snapshot(graph) + [x.cpu().numpy(), cov.cpu().numpy()]
        if rep == 0:
            first = got
            graph.import_state(blob)
    for a, c in zip(first, got):
        assert np.array_equal(a, c)
    for j in range(K):
        m = int(np.searchsorted(ds["steps"], t0 + j))
        has = m < ds["M"] and ds["steps"][m] == t0 + j
        eager.step((t0 + j) / p.update_freq, imu[j], tag[j] if has else None, arrived[j] if has else None)
    torch.cuda.synchronize()
    ref = snapshot(eager)
    for a, c in zip(got[:4], ref):
        assert np.array_equal(a, c)
    assert np.array_equal(got[4], ref[0]) and np.array_equal(got[5], packed_of(ref[1]))
    eager.close(); graph.close()


# ---- hand-over ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", list(MODES))
def test_hand_over_with_run_and_export(mode):
    p = make_params(1, 1, mode)
    N, T = 2048, 900
    ds = device_streams(scn_of(p), N, T, seed=17)
    ref = q.BatchEKF(p, N, 0)
    run_streams(ref, ds, 0, T)
    # step -> qekf_run -> step
    b = q.BatchEKF(p, N, 0)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    s = Stepper(b, ds, p)
    s.run(0, 300, check_every=0)
    torch.cuda.synchronize()
    run_streams(b, ds, 300, 300)
    s.run(600, 300, check_every=0)
    torch.cuda.synchronize()
    assert_equal_or_last_bit(snapshot(b), snapshot(ref), ("handover", mode))
    # export after steps -> import into a fresh handle -> step
    c = q.BatchEKF(p, N, 0)
    c.set_stream(torch.cuda.current_stream().cuda_stream)
    s = Stepper(c, ds, p)
    s.run(0, 450, check_every=0)
    torch.cuda.synchronize()
    blob = c.export_state()
    d = q.BatchEKF(p, N, 0)
    d.set_stream(torch.cuda.current_stream().cuda_stream)
    d.import_state(blob)
    Stepper(d, ds, p).run(450, 450, check_every=0)
    torch.cuda.synchronize()
    assert_equal_or_last_bit(snapshot(d), snapshot(ref), ("export", mode))
    for h in (ref, b, c, d):
        h.close()


def test_monte_carlo_after_steps_uses_the_ring():
    """After steps, qekf_run_monte_carlo continues from the ring-based history: its result equals a qekf_run of its own
    synthesised streams from the same state."""
    p = make_params(1, 1, "fixed")
    scn = scn_of(p, seconds=5.0, latency=0.03)
    N = 1024
    noise = nat.default_noise()
    noise.seed = 77
    syn = q.BatchEKF(p, N, 0)
    st = syn.synthesize_streams(scn, noise)
    syn.close()
    a, b = q.BatchEKF(p, N, 0), q.BatchEKF(p, N, 0)
    ds = dict(T=st["imu"].shape[0], M=len(st["tag_step"]), steps=st["tag_step"],
              imu=torch.as_tensor(st["imu"], device=DEV), tag_step=torch.as_tensor(st["tag_step"], device=DEV),
              tag_pose=torch.as_tensor(st["tag_pose"], device=DEV), tag_stamp=torch.as_tensor(st["tag_stamp"], device=DEV),
              tag_valid=torch.as_tensor(st["tag_valid"], device=DEV))
    for h in (a, b):
        h.set_stream(torch.cuda.current_stream().cuda_stream)
        Stepper(h, ds, p).run(0, 400, check_every=0)
    torch.cuda.synchronize()
    a.run_monte_carlo(scn, noise, k0=400, n_steps=300)
    run_streams(b, ds, 400, 300)
    assert_equal_or_last_bit(snapshot(a), snapshot(b), ("mc", 64, 1, 1))
    a.close(); b.close()


@pytest.mark.parametrize("mode", list(MODES))
def test_step_counts(mode):
    p = make_params(1, 1, mode)
    N, T = 4096, 1200
    ds = device_streams(scn_of(p), N, T, seed=21)
    b = q.BatchEKF(p, N, 0)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    s = Stepper(b, ds, p)
    s.run(0, 300, check_every=0)
    b.step_counts(reset=True)
    s.run(300, 900, check_every=0)
    npred, ncorr = b.step_counts()
    per_tick = npred / (N * 900)
    if mode == "single":
        assert npred == N * 900
    else:
        d = round(p.measurement_delay * p.update_freq) if mode == "fixed" else round(0.036 * p.update_freq)
        upm = int(p.update_freq / p.measurement_freq)
        assert per_tick <= 2 + (d + 2) / upm, per_tick
    assert ncorr > 0.5 * N * 900 / (p.update_freq / p.measurement_freq)
    print("%s: %.3f predictions per filter-tick" % (mode, per_tick))
    b.close()


# ---- interface --------------------------------------------------------------------------------------------------------

def test_bad_arguments():
    import ctypes as C
    BAD_ARG = {v: k for k, v in nat.STATUS.items()}["QEKF_ERR_BAD_ARG"]
    p = make_params()
    N = 64
    b = q.BatchEKF(p, N, 0)
    L = nat.lib()
    imu = torch.zeros((6, N), dtype=torch.float64, device=DEV)
    tag = torch.zeros((8, N), dtype=torch.float64, device=DEV)
    arrived = torch.ones(N, dtype=torch.uint8, device=DEV)
    io = nat.QekfStepIO()
    io.imu = imu.data_ptr()
    assert L.qekf_step(None, 0.0, C.byref(io)) == BAD_ARG
    assert L.qekf_step(b._h, 0.0, None) == BAD_ARG
    io.imu = None
    assert L.qekf_step(b._h, 0.0, C.byref(io)) == BAD_ARG
    io.imu = imu.data_ptr()
    io.arrived = arrived.data_ptr()
    assert L.qekf_step(b._h, 0.0, C.byref(io)) == BAD_ARG          # arrived without tag
    io.tag = tag.data_ptr()
    host = np.zeros((6, N))
    io.x_out = host.ctypes.data                                                   # unregistered host memory
    assert L.qekf_step(b._h, 0.0, C.byref(io)) == BAD_ARG
    io.x_out = None
    io.imu = host.ctypes.data
    assert L.qekf_step(b._h, 0.0, C.byref(io)) == BAD_ARG
    with pytest.raises(ValueError):
        b.step(0.0, imu.cpu())
    with pytest.raises(ValueError):
        b.step(0.0, imu.float())
    with pytest.raises(ValueError):
        b.step(0.0, torch.zeros((N, 6), dtype=torch.float64, device=DEV).t())
    with pytest.raises(ValueError):
        b.step(0.0, imu, x=torch.zeros((15, N), dtype=torch.float64, device=DEV))
    with pytest.raises(ValueError):
        b.step(0.0, imu, arrived=arrived)
    b.step(0.0, imu)                                 # the handle still works
    b.close()


@pytest.mark.parametrize("lanes", [2, 3])
def test_step_ignores_the_mapping(lanes):
    p = make_params(1, 1, "single")
    N, T = 2048, 400
    ds = device_streams(scn_of(p), N, T, seed=31)
    a, b = q.BatchEKF(p, N, 0), q.BatchEKF(p, N, 0)
    b.set_mapping(lanes)
    for h in (a, b):
        h.set_stream(torch.cuda.current_stream().cuda_stream)
        Stepper(h, ds, p).run(0, T, check_every=0)
    torch.cuda.synchronize()
    for u, v in zip(snapshot(a), snapshot(b)):
        assert np.array_equal(u, v)
    a.close(); b.close()


def test_per_filter_parameters_are_accepted():
    """Unlike qekf_tick: a sweep of per-filter parameters steps exactly like the per-filter replay (also covered by the
    open-loop matrix); here, per-filter delays under dynamic delay and a filter-by-filter check against the oracle."""
    p = make_params(1, 1, "fixed")
    N, T = 256, 500
    ds = device_streams(scn_of(p), N, T, seed=41)
    b = q.BatchEKF(p, N, 0)
    sweep(b, p, "fixed", N, 7)
    b.set_stream(torch.cuda.current_stream().cuda_stream)
    Stepper(b, ds, p).run(0, T, check_every=0)
    torch.cuda.synchronize()
    ob = orc.Batch(orc.params_from(p), N)
    rng = np.random.default_rng(7)
    qv = np.array(list(p.Q_a) + list(p.Q_w) + list(p.Q_ab) + list(p.Q_wb))[:, None] * rng.uniform(0.5, 2.0, (1, N))
    ob.set_filter_params(q.PF_Q, qv)
    ob.set_filter_params(q.PF_DELAY, np.stack([rng.uniform(0.015, 0.045, N), rng.uniform(0.0, 0.01, N)]))
    ob.run(0, T, ds["imu"].cpu().numpy(), ds["steps"], ds["tag_pose"].cpu().numpy(), ds["tag_stamp"].cpu().numpy(),
           ds["tag_valid"].cpu().numpy())
    assert norm_rel(b.state(), ob.state()) < 1e-9
    assert norm_rel(b.cov(), ob.cov()) < 1e-9
    b.close()
