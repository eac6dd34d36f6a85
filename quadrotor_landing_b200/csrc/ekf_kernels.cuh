// ekf_kernels.cuh -- sm_100a kernels: one CUDA thread per filter, covariance staged in shared memory
// (element-major, conflict-free), nominal state in registers, many ticks fused per launch.
//
// run_kernel is RelativePoseEKF::filter_update (relative_pose_EKF.cpp:127-303) iterated n_steps times
// with the node's callback sequencing (relative_pose_EKF_node.cpp:144-182) folded in: before tick k
// the tag arrival scheduled for k is latched (and initialises the filter if it is the first one), then
// the IMU sample of tick k is latched, then the tick runs.
#pragma once

#include <type_traits>

#include "ekf_core.cuh"
#include "ekf_synth.cuh"

namespace qekf {

enum : int32_t {
    FLAG_INIT = 1,        // state_initialized
    FLAG_READY = 2,       // measurement_ready
    FLAG_CORRECTED = 4,   // performed_correction
    FLAG_ACTIVE = 8       // filter_active
};

constexpr int AUX_DIM = 11;   // accel_rel(3) r_t_vt_obs(3) q_tv_obs(4) measurement_delay_curr(1)
constexpr int PEND_DIM = 8;   // pending tag pose(7) + capture stamp(1)

// Device-resident state of N filters, structure-of-arrays with leading dimension ld (>= N, multiple
// of 32) so that every per-component access is a coalesced warp transaction.
template <typename T> struct DeviceState {
    T *x;            // [16][ld]   nominal state
    T *P;            // [NP][ld]   packed upper triangle of cov_pert
    T *aux;          // [11][ld]
    double *pend;    // [8][ld]    latched-but-unconsumed tag pose + stamp
    int32_t *flags;  // [ld]
    int32_t *upds;   // [ld]       upds_since_correction
    unsigned long long *counts;   // [2] prediction_step / correction_step calls executed (all launches)
    int64_t ld;
    int64_t n;
    // Delayed-measurement fusion (multirate_ekf, cpp:196-236,251-264): instead of the reference's vectors of
    // (x, u, P) per tick, a lagged checkpoint (the oldest history entry that can still be addressed) plus a
    // ring of the IMU inputs of the entries after it.  Every later entry is a pure function of those
    // (x_hist[i] = prediction_step(x_hist[i-1], u_hist[i])), so it is recomputed when needed.  nullptr when
    // the handle is single-rate.
    T *xc;              // [16][ld]   checkpoint nominal state
    T *Pc;              // [NP][ld]   checkpoint covariance
    T *ring;            // [ring_len][6][ld]  u_hist of entry e at slot e % ring_len
    int32_t *nh;        // [ld] history entries after the checkpoint (the head is entry nh)
    int32_t *hpos;      // [ld] ring slot of the head entry
    int32_t *hlen;      // [ld] x_hist.size() as the reference would report it (grows without bound between corrections)
    int32_t ring_len;   // L >= dmax_m1 + 1 + upd_per_meas
    int32_t dmax_m1;    // D - 1, D = largest step delay any correction of this handle can use
    // Per-filter parameter overrides (BASELINE config 5); nullptr = launch-wide constants only.
    const T *pf;              // [PF_DIM][ld]
    const double *pf_delay;   // [2][ld]
    // Monte-Carlo launches: which filter the thread slot j of the fused replay advances (nullptr = filter j).  The
    // host orders filters by the start of their private tag dropout, so that the filters sharing a CTA lose and
    // regain their measurements together and their correction cadence stays aligned; filters are independent and
    // the noise is keyed by the filter id, so the order changes no result.
    //   perm     : index indirection -- slot j works on row perm[j] of every array (the cooperative mappings, ekf_coop.cuh /
    //              ekf_duo.cuh; uncoalesced loads and stores at the two ends of the launch)
    //   gid_perm : the arrays themselves have been reordered for the launch (the host gathers them into slot order before
    //              and scatters them back after, qekf_capi.cu permute_state), so slot j works on row j, coalesced, and
    //              only the noise identity is perm[j] (the thread-per-filter kernels, single-rate and delayed fusion)
    const int32_t *perm;
    const int32_t *gid_perm;
    // delayed fusion, Monte-Carlo launches: 1 = the entries after every checkpoint are the synthetic IMU samples of this
    // launch's noise model and scenario, so the replay may re-synthesise them instead of reading the ring (run_filter_mrs)
    int32_t hist_synth;
};

// the parameter view of filter i: launch-wide constants, or this filter's column of the override table.
// cold<CSM>: what the out-of-line calls read the constants through -- the same view (CSM = false: host instantiation,
// per-tick kernel) or the view over the CTA's shared-memory copy of the constant block (CSM = true: the fused replay).
template <typename T, bool PF> struct ParSel;
template <typename T> struct ParSel<T, false> {
    using type = ParU<T>;
    static QEKF_FN type make(const Consts<T> &c, const DeviceState<T> &, int64_t) { return type{ c }; }
    static QEKF_FN type make_cold(const type &par, const Consts<T> *, const DeviceState<T> &, int64_t, std::false_type) { return par; }
#ifdef __CUDACC__
    static __device__ __forceinline__ ParUS<T> make_cold(const type &, const Consts<T> *csm, const DeviceState<T> &, int64_t, std::true_type)
    {
        return ParUS<T>{ (uint32_t)__cvta_generic_to_shared(csm) };
    }
#endif
};
template <typename T> struct ParSel<T, true> {
    using type = ParF<T>;
    static QEKF_FN type make(const Consts<T> &c, const DeviceState<T> &st, int64_t i)
    {
        return type{ c, st.pf + i, st.pf_delay + i, st.ld };
    }
    static QEKF_FN type make_cold(const type &par, const Consts<T> *, const DeviceState<T> &, int64_t, std::false_type) { return par; }
#ifdef __CUDACC__
    static __device__ __forceinline__ ParFS<T> make_cold(const type &, const Consts<T> *csm, const DeviceState<T> &st, int64_t i, std::true_type)
    {
        return ParFS<T>{ (uint32_t)__cvta_generic_to_shared(csm), st.pf + i, st.pf_delay + i, st.ld };
    }
#endif
};

// Input streams as seen by the kernel.  Element (k, c) of filter i lives at base[(k*6+c)*cs + i*is]:
// explicit per-filter streams use (cs, is) = (N, 1); one stream shared by all filters uses (1, 0).
struct StreamView {
    const double *imu;
    const int32_t *tag_step;
    const double *tag_pose;
    const double *tag_stamp;
    const uint8_t *tag_valid;
    const double *tag_sigma;  // SYNTH with the detection front-end: per-arrival (sigma_p, sigma_th) [M][2], else nullptr
    int64_t cs, is;
    int64_t M;
    int64_t vs;           // stride of tag_valid rows (N)
    double t_start;
    double update_freq;
};

template <typename T> struct RunArgs {
    DeviceState<T> st;
    StreamView in;
    Consts<T> c;
    int64_t k0, n_steps;
    int32_t m0;           // first arrival with tag_step >= k0
    NoiseSpec ns;         // SYNTH launches only
    StatsView stats;      // acc == nullptr: no statistics
};

#ifdef __CUDA_ARCH__
#define QEKF_COLD __device__ __noinline__
#else
#define QEKF_COLD inline
#endif

// Where a filter's inputs come from.  Explicit: per-filter (or shared) streams in memory.  Synth: one
// clean stream shared by all filters plus this filter's own noise realisation, generated on the fly.
template <typename T, bool SYNTH> struct Inputs {
    const double *imu_i, *tag_i;
    int64_t cs;
    const uint8_t *valid_i;
    int64_t vs;
    int64_t gid;
    double bias[6];
    int32_t priv_start;

    // i: row of this filter in the per-filter arrays; id: its index in the handle's id space (noise identity)
    QEKF_FN void init(const RunArgs<T> &a, int64_t i) { init(a, i, i); }
    QEKF_FN void init(const RunArgs<T> &a, int64_t i, int64_t id)
    {
        imu_i = a.in.imu + i * a.in.is;
        tag_i = a.in.tag_pose + i * a.in.is;
        cs = a.in.cs;
        valid_i = (!SYNTH && a.in.tag_valid) ? a.in.tag_valid + i : nullptr;
        vs = a.in.vs;
        gid = a.ns.gid0 + id;
        if (SYNTH) {
            true_bias(a.ns, gid, bias);
            priv_start = private_dropout_start(a.ns, gid);
        }
    }
    QEKF_FN void raw_imu(int64_t k, double u[6]) const
    {
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) u[cc] = imu_i[(k * 6 + cc) * cs];
    }
    QEKF_FN void raw_imu(const StreamView &sv, int64_t k, double u[6]) const
    {
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) u[cc] = SYNTH ? sv.imu[k * 6 + cc] : imu_i[(k * 6 + cc) * cs];
    }
    // turn the raw sample of tick k into what the filter sees
    QEKF_FN void imu(const NoiseSpec &ns, int64_t k, const double raw[6], T u[6]) const
    {
        if (SYNTH) {
            double un[6];
            synth_imu(ns, gid, k, raw, bias, un);
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) u[cc] = (T)un[cc];
        } else {
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) u[cc] = (T)raw[cc];
        }
    }
    // `sv`, `ns`: the launch's StreamView and NoiseSpec (kernel-parameter resident, passed by the caller as a.in, a.ns):
    // read through the constant bank rather than through per-lane copies of pointers, which would live in local memory
    // and turn every access into a generic load
    QEKF_FN void tag_f64(const StreamView &sv, const NoiseSpec &ns, int32_t m, double tag[7]) const
    {
        double raw[7];
        // SYNTH launches read the one shared clean scenario (element stride 1) straight through the kernel
        // parameters: no per-lane pointer has to stay alive for it
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) raw[cc] = SYNTH ? sv.tag_pose[(int64_t)m * 7 + cc] : tag_i[((int64_t)m * 7 + cc) * cs];
        if (SYNTH) {
            double sp = (double)ns.sig_p, sth = (double)ns.sig_th;
            if (sv.tag_sigma) { sp = sv.tag_sigma[2 * m]; sth = sv.tag_sigma[2 * m + 1]; }
            synth_tag(ns, gid, m, raw, tag, sp, sth);
        }
        else {
#pragma unroll
            for (int cc = 0; cc < 7; ++cc) tag[cc] = raw[cc];
        }
    }
    QEKF_FN void tag(const StreamView &sv, const NoiseSpec &ns, int32_t m, T t[7]) const
    {
        double d[7];
        tag_f64(sv, ns, m, d);
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) t[cc] = (T)d[cc];
    }
    QEKF_FN bool valid(const StreamView &sv, const NoiseSpec &ns, int32_t m, int32_t step) const
    {
        return valid(sv, ns, m, step, priv_start);
    }
    // (pstart: this filter's private_dropout_start, kept by the caller where it pleases)
    QEKF_FN bool valid(const StreamView &sv, const NoiseSpec &ns, int32_t m, int32_t step, int32_t pstart) const
    {
        // SYNTH: sv.tag_valid is the detection front-end's visibility mask [M], shared by all filters (or nullptr)
        if (SYNTH) return arrival_valid(ns, step, pstart) && (sv.tag_valid == nullptr || sv.tag_valid[m] != 0);
        return valid_i ? (valid_i[(int64_t)m * vs] != 0) : true;
    }
};

// One statistics sample after tick k.  Where the truth comes from is decided at compile time: SYNTH (Monte-Carlo)
// launches read the shared scenario truth and get the filter's true bias from the caller; explicit-stream launches
// read row i of the per-filter truth, bin by bin, true bias included (StatsView::truth_pf).  Called by every
// lane of the CTA at the same point (`valid` = this lane holds an initialised filter that is at the sampling
// tick), so that the 20 sums can be reduced over the warp with shuffles and leave as ONE atomic per warp and
// statistic instead of one per lane.  Deliberately NOT inlined on the device: it runs once per `stride` ticks
// and must not take part in the register allocation of the hot loop.
// (SAVE is a leftover of the in-place NEES factorisation, which had to park P in HBM; the covariance is only read now.)
template <typename T, bool BIAS, class PS, bool SAVE = true, bool SYNTH = true>
QEKF_COLD void stats_sample(const RunArgs<T> &a, int64_t i, int64_t k, const Nominal<T> s, PS P, const double *bias,
                            bool valid)
{
    constexpr int N = PS::n;
    constexpr int NP = N * (N + 1) / 2;
    // by value: this function is reached through a generic reference to the kernel parameters, and every store
    // below would otherwise force the compiler to reload these fields (it cannot rule out aliasing)
    const StatsView sv = a.stats;
    int32_t bin = (int32_t)((k + 1) / sv.stride - 1);
    if (bin < 0 || bin >= sv.n_bins) valid = false;
    double sum[STAT_DIM];
#pragma unroll
    for (int c = 0; c < STAT_DIM; ++c) sum[c] = 0.0;
    if (valid) {
        // component c of the true state (r v q_tv ab wb); the bias components only exist per filter
        auto tr = [&](int c) -> double {
            return SYNTH ? sv.truth[(k + 1) * 10 + c] : sv.truth_pf[((int64_t)bin * 16 + c) * sv.ld_t + i];
        };
        T e[N];
#pragma unroll
        for (int c = 0; c < 3; ++c) { e[c] = (T)tr(c) - s.r[c]; e[3 + c] = (T)tr(3 + c) - s.v[c]; }
        {
            T qt[4] = { (T)tr(6), (T)tr(7), (T)tr(8), (T)tr(9) }, dq[4];
            quat_conj_mul(s.q, qt, dq);
            quat_normclip(dq);
            quat_log(dq, e + 6);
        }
        if (BIAS) {
            auto tb = [&](int c) -> double { return SYNTH ? bias[c] : tr(10 + c); };
#pragma unroll
            for (int c = 0; c < 3; ++c) { e[9 + c] = (T)tb(c) - s.ab[c]; e[12 + c] = (T)tb(3 + c) - s.wb[c]; }
        }
        // (the covariance is only read: see nees_readonly)
        T nees;
        bool ok = nees_readonly<T>(P, e, nees);
        bool finite = true;
#pragma unroll
        for (int c = 0; c < N; ++c) { finite = finite && (M<T>::abs_(e[c]) < T(1e30)); }
        ok = ok && finite && (M<T>::abs_(nees) < T(1e30));
        if (ok) {
#pragma unroll
            for (int c = 0; c < N; ++c) sum[c] = (double)e[c] * (double)e[c];
            sum[15] = (double)nees;
            sum[16] = 1.0;
            sum[17] = ((double)nees >= sv.chi2_lo && (double)nees <= sv.chi2_hi) ? 1.0 : 0.0;
            sum[19] = (double)e[0] * (double)e[0] + (double)e[1] * (double)e[1] + (double)e[2] * (double)e[2];
        } else {
            sum[18] = 1.0;
        }
    }
#ifdef __CUDA_ARCH__
    const unsigned full = 0xffffffffu;
    bin = __reduce_max_sync(full, valid ? bin : -1);          // the valid lanes of a CTA all sit at the same tick
    if (bin < 0) return;
#pragma unroll
    for (int c = 0; c < STAT_DIM; ++c) {
        double v = sum[c];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(full, v, off);
        sum[c] = v;
    }
    if ((threadIdx.x & 31) == 0) {
        double *acc = sv.acc + (((i >> 5) % STAT_REPL) * (int64_t)sv.n_bins + bin) * STAT_DIM;
#pragma unroll
        for (int c = 0; c < STAT_DIM; ++c)
            if (sum[c] != 0.0) atomicAdd(acc + c, sum[c]);
    }
#else
    if (!valid) return;
    double *acc = sv.acc + (((i >> 5) % STAT_REPL) * (int64_t)sv.n_bins + bin) * STAT_DIM;
    for (int c = 0; c < STAT_DIM; ++c) acc[c] += sum[c];
#endif
}

template <typename T, class PS>
QEKF_FN void load_filter(const DeviceState<T> &st, int64_t i, Nominal<T> &s, PS &P)
{
    constexpr int N = PS::n;
    constexpr int NP = N * (N + 1) / 2;
    const T *x = st.x + i;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        s.r[k] = x[(0 + k) * st.ld];
        s.v[k] = x[(3 + k) * st.ld];
        s.ab[k] = x[(10 + k) * st.ld];
        s.wb[k] = x[(13 + k) * st.ld];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) s.q[k] = x[(6 + k) * st.ld];
#pragma unroll 8
    for (int e = 0; e < NP; ++e) P.el(e) = st.P[e * st.ld + i];
}

template <typename T, class PS>
QEKF_FN void store_filter(const DeviceState<T> &st, int64_t i, const Nominal<T> &s, const PS &P)
{
    constexpr int N = PS::n;
    constexpr int NP = N * (N + 1) / 2;
    T *x = st.x + i;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x[(0 + k) * st.ld] = s.r[k];
        x[(3 + k) * st.ld] = s.v[k];
        x[(10 + k) * st.ld] = s.ab[k];
        x[(13 + k) * st.ld] = s.wb[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) x[(6 + k) * st.ld] = s.q[k];
#pragma unroll 8
    for (int e = 0; e < NP; ++e) st.P[e * st.ld + i] = P.el(e);
}

// ------------------------------------------------------------------------------------------------
// fused multi-tick replay
// ------------------------------------------------------------------------------------------------
// correction_step behind a real call on the device: it runs on one tick in upd_per_meas, and keeping it out
// of line keeps its ~120 live doubles out of the register allocation of the per-tick prediction loop.
template <typename T, bool BIAS, bool DIRECT, class PS, class PAR>
QEKF_COLD void correction_call(Nominal<T> *sp, PS &P, const T *tag, const PAR par, Observation<T> *obs)
{
    Nominal<T> s = *sp;
    T tg[7];
#pragma unroll
    for (int cc = 0; cc < 7; ++cc) tg[cc] = tag[cc];
    Observation<T> o;
    correction_step<T, BIAS, DIRECT>(s, P, tg, par, o);
    *sp = s;
    *obs = o;
}

// CTA-wide votes, one barrier per loop iteration.  Each warp reduces its lanes with a ballot, lane 0 adds the
// packed counts into a triple-buffered shared-memory slot, one __syncthreads(), everybody reads.  The barrier
// also keeps the warps of the CTA walking through the same stretch of the (large, fully unrolled) instruction
// stream together, so they share its instruction-cache lines.  The host instantiation is a CTA of one lane.
struct CtaVote {
    int active, want, fenced, at_fence, lanes;
    bool out_of_patience;
};
constexpr int VOTE_WORDS = 12;   // 3 buffers x 4 words

QEKF_FN void cta_vote_init(int *vbuf)
{
#ifdef __CUDA_ARCH__
    if (threadIdx.x < VOTE_WORDS) vbuf[threadIdx.x] = 0;
    __syncthreads();
#else
    (void)vbuf;
#endif
}

QEKF_FN CtaVote cta_vote(int *vbuf, uint32_t iter, bool active, bool want, bool oop, bool fenced, bool at_fence)
{
    CtaVote r;
#ifdef __CUDA_ARCH__
    const unsigned full = 0xffffffffu;
    const unsigned ma = __ballot_sync(full, active), mw = __ballot_sync(full, want), mo = __ballot_sync(full, oop);
    const unsigned mf = __ballot_sync(full, fenced), mt = __ballot_sync(full, at_fence);
    int *v = vbuf + (iter % 3u) * 4;
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(v + 0, __popc(ma) | (__popc(mw) << 16));
        atomicAdd(v + 1, __popc(mf) | (__popc(mt) << 16));
        if (mo) atomicOr(v + 2, 1);
    }
    __syncthreads();
    const int x0 = v[0], x1 = v[1], x2 = v[2];
    if (threadIdx.x == 0) {          // recycle the buffer of two iterations ahead (read last in iteration iter-1)
        int *z = vbuf + ((iter + 2u) % 3u) * 4;
        z[0] = 0; z[1] = 0; z[2] = 0;
    }
    r.active = x0 & 0xffff; r.want = x0 >> 16; r.fenced = x1 & 0xffff; r.at_fence = x1 >> 16;
    r.out_of_patience = x2 != 0;
    r.lanes = (int)blockDim.x;
#else
    (void)vbuf; (void)iter;
    r.active = active; r.want = want; r.fenced = fenced; r.at_fence = at_fence; r.out_of_patience = oop; r.lanes = 1;
#endif
    return r;
}

// Warp-level votes (five ballots, no shared memory).  Measured and NOT used by the thread-per-filter loops: when every
// warp decides for itself, the warps of a CTA serve their corrections in different iterations, and since the CTA
// meets once per iteration (lockstep keeps the instruction cache shared) everybody pays for every warp's correction:
// 4.21e9 vs 4.68e9 filter-steps/s with the CTA-wide vote (profiles/r2_04_mappings.md).
struct WarpVote {
    int active, want, fenced, at_fence, lanes;
    bool out_of_patience;
};
QEKF_FN WarpVote warp_vote(bool active, bool want, bool oop, bool fenced, bool at_fence)
{
    WarpVote r;
#ifdef __CUDA_ARCH__
    const unsigned full = 0xffffffffu;
    r.active = __popc(__ballot_sync(full, active));
    r.want = __popc(__ballot_sync(full, want));
    r.fenced = __popc(__ballot_sync(full, fenced));
    r.at_fence = __popc(__ballot_sync(full, at_fence));
    r.out_of_patience = __ballot_sync(full, oop) != 0u;
    r.lanes = 32;
#else
    r.active = active; r.want = want; r.fenced = fenced; r.at_fence = at_fence; r.out_of_patience = oop; r.lanes = 1;
#endif
    return r;
}
QEKF_FN bool cta_any(bool x)
{
#ifdef __CUDA_ARCH__
    return __syncthreads_or(x) != 0;
#else
    return x;
#endif
}

// An int32 that lives in the lane's slot of a shared-memory scratch array.  Whatever the replay loops carry from
// one iteration to the next competes with the ~200 registers of the unrolled tick; what loses ends up in local
// memory, and with 7 warps per SM and an L1 that shared memory has squeezed to a few KB the reloads are L2 round
// trips on the critical path of every tick (profiles/r1_05_sr_vs_multirate.md: 73 local loads per warp-tick in the
// delayed-fusion loop; profiles/r2_06_sr_stalls.md: the tick index, the prediction counter, the prefetched IMU sample and
// the true bias in the single-rate loop).  The sequencer's integer state and the true bias' six normals are therefore
// kept here explicitly: a shared-memory access costs a tenth of that.
struct SmemInt {
    int32_t *p;
    QEKF_FN operator int32_t() const { return *p; }
    QEKF_FN SmemInt &operator=(int32_t v) { *p = v; return *this; }
    QEKF_FN SmemInt &operator=(const SmemInt &o) { *p = *o.p; return *this; }   // assigns the value, not the slot
    QEKF_FN SmemInt &operator+=(int32_t v) { *p += v; return *this; }
    QEKF_FN SmemInt &operator-=(int32_t v) { *p -= v; return *this; }
    QEKF_FN SmemInt &operator|=(int32_t v) { *p |= v; return *this; }
    QEKF_FN SmemInt &operator&=(int32_t v) { *p &= v; return *this; }
    QEKF_FN SmemInt &operator++() { *p += 1; return *this; }
};
// per-lane scratch words of the replay loops:
//   delayed fusion: flags upds nh hpos hlen m next_tag_step pend_m held k | 6 floats: the true bias' normals | n_pred
//                   priv_start
//   single rate   : flags upds n_pred n_corr n_iter m next_tag_step pend_m held k | 6 floats: the true bias' normals
constexpr int MR_SCRATCH_INTS = 18;
constexpr int SR_SCRATCH_INTS = 16;

// The per-filter replay loop, one lane per filter.  Host-callable so that the CPU-side unit tests
// (tests/host_core) can run the very same code against the oracle without a GPU; the product only ever
// calls it from run_kernel.
//
// Event-driven: every lane keeps its OWN tick index k and runs the ticks that need no decision of the CTA -- tag
// callbacks, predictions, bookkeeping -- in an inner loop without calls, votes or barriers (round 2; the loop used to
// iterate over ticks with one CTA-wide vote and barrier per tick, and the ~250 instructions of sequencing per tick plus
// the values ptxas parked in local memory around the call sites were a fifth of the time).  A lane leaves the inner
// loop when the prediction of a tick whose measurement gate is open is done, at a sampling boundary, or at the end of
// the launch; only there the CTA meets.  The correction step (2.5x a prediction, once per upd_per_meas ticks) is then
// executed once for the whole CTA: lanes whose cadence is out of phase with their CTA-mates (a private tag dropout, a
// rejected detection, a late initialisation) arrive after different numbers of ticks and are corrected together, at
// their own tick indices.  Filters are independent, so when a filter's tick is executed changes nothing in its
// arithmetic: results are bit-identical to a loop that walks all filters tick by tick.
// Statistics fence: a lane that has finished a sampling tick waits until every lane of the CTA has, then all
// sample together (one execution of the sampling code per stride; the time skew is back to zero).
// `live` = false marks the padding lanes of a ragged last CTA (they only take part in the votes).
// STATS: the fence and the sampling are compiled in (Monte-Carlo launches, and explicit-stream launches scored against
// per-filter truth).  The unscored explicit kernels leave them out: compiled in, with the statistics switched off at
// run time, they cost those kernels 1.0 % (FP64, N = 65,536) and 2.4 % (FP64 conventional model, N = 1M) in
// tools/perf_probe.py on a B200.
template <typename T, bool BIAS, bool DIRECT, bool SYNTH, bool PF, class PS, bool CSM = false, bool STATS = SYNTH>
QEKF_FN void run_filter(const RunArgs<T> &a, const int64_t i_in, PS &P, int32_t *scr, const int scr_stride,
                        const bool live = true, int *vbuf = nullptr, const Consts<T> *c_cold = nullptr)
{
    const Consts<T> &c = a.c;
    const int64_t i = live ? i_in : 0;
    const typename ParSel<T, PF>::type par = ParSel<T, PF>::make(a.c, a.st, i);
    // what the out-of-line calls read the launch-wide constants through (ParSel::make_cold)
    const auto par_cold = ParSel<T, PF>::make_cold(par, c_cold, a.st, i, std::integral_constant<bool, CSM>());
    const int32_t k_end = (int32_t)(a.k0 + a.n_steps);       // (qekf_run bounds tick indices to 31 bits)
    Nominal<T> s;
    SmemInt flags{ scr + 0 * scr_stride }, upds{ scr + 1 * scr_stride }, n_pred{ scr + 2 * scr_stride };
    SmemInt n_corr{ scr + 3 * scr_stride }, n_iter{ scr + 4 * scr_stride }, m{ scr + 5 * scr_stride };
    SmemInt next_tag_step{ scr + 6 * scr_stride }, pend_m{ scr + 7 * scr_stride }, held{ scr + 8 * scr_stride };
    SmemInt k{ scr + 9 * scr_stride };
    flags = 0; upds = 0; n_pred = 0; n_corr = 0; n_iter = 0;
    T accel[3] = { T(0), T(0), T(0) };
    Inputs<T, SYNTH> in;
    double un[6] = { 0, 0, 0, 0, 0, 0 };
    k = k_end;                         // padding lanes are born finished
    if (live) {
        load_filter<T>(a.st, i, s, P);
        flags = a.st.flags[i];
        upds = a.st.upds[i];
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) accel[cc] = a.st.aux[cc * a.st.ld + i];
        in.init(a, i, a.st.gid_perm ? (int64_t)a.st.gid_perm[i] : i);
        k = (int32_t)a.k0;
        if (SYNTH) {                   // the true bias as its six normals, in the scratch
            float z[6];
            normals6(a.ns, in.gid, STREAM_BIAS, 0u, z);
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) reinterpret_cast<float *>(scr)[(10 + cc) * scr_stride] = z[cc];
        } else {
            in.raw_imu(k, un);         // software prefetch (explicit streams live in HBM): un holds the raw sample of tick k
        }
    }
    auto true_bias_now = [&](double b[6]) {
#pragma unroll
        for (int cc = 0; cc < 6; ++cc)
            b[cc] = (double)(cc < 3 ? a.ns.sig_ba : a.ns.sig_bw) * (double)reinterpret_cast<const float *>(scr)[(10 + cc) * scr_stride];
    };

    uint32_t n_sexec = 0, n_cev = 0;
    m = a.m0;
    next_tag_step = (m < a.in.M) ? a.in.tag_step[m] : INT32_MAX;
    pend_m = -1;                       // index of the latched arrival; -1 = latched pose lives in st.pend
    held = 0;                          // iterations this lane has held its correction back
    bool at_fence = false;             // finished a sampling tick; waiting for the CTA to catch up
    const bool do_stats = STATS && a.stats.acc != nullptr;
    const int32_t patience = c.limit_measurement_freq ? (c.upd_per_meas - 1) : 0;
    // the next sampling boundary (a multiple of the stride): every lane of the CTA stops there until all have arrived, so
    // it is the same for all of them and moves on when the sample is taken -- no k % stride on the per-tick path
    int32_t next_fence = do_stats ? (int32_t)((a.k0 / a.stats.stride + 1) * a.stats.stride) : INT32_MAX;
    bool predicted = false;            // the prediction of tick k has run; the tick waits for its correction

    cta_vote_init(vbuf);
    for (uint32_t iter = 0;; ++iter) {
        // ---- The ticks that need no decision of the CTA: tag callback (node.cpp:153-176), prediction (cpp:240-249),
        //      bookkeeping -- a loop of its own, without calls, votes or barriers, whose state lives in registers.  A lane
        //      leaves it with the prediction of a tick whose measurement gate is open (cpp:147) done and its correction
        //      pending, at a sampling boundary, or at the end of the launch; the CTA meets (one vote, one barrier) only
        //      there.  Lanes whose tick indices differ (private dropouts, late initialisation) leave after different
        //      numbers of ticks and are corrected together, at their own ticks: filters are independent, so when a
        //      filter's tick is executed changes nothing in its arithmetic. ----
        bool want = predicted;
        if (k < k_end && !at_fence && !predicted) {
            int32_t kk = k, up = upds, fl = flags, nts = next_tag_step, np_run = 0;
            for (;;) {
                if (kk == nts) {
                    const int32_t mm = m;
                    if (in.valid(a.in, a.ns, mm, kk)) {
                        pend_m = mm;
                        fl |= FLAG_READY;
                        if (!(fl & FLAG_INIT)) {
                            T tag0[7];
                            in.tag(a.in, a.ns, mm, tag0);
                            initialize_state<T, BIAS>(s, P, tag0, par, false);
                            fl |= FLAG_INIT;
                        }
                    }
                    m = mm + 1;
                    nts = (mm + 1 < a.in.M) ? a.in.tag_step[mm + 1] : INT32_MAX;
                }
                const bool init = (fl & FLAG_INIT) != 0;
                const bool gate = init && (fl & FLAG_READY) && (!c.limit_measurement_freq || (up + 1) >= c.upd_per_meas);
                if (init) {
                    T u[6];
                    if (SYNTH) {
                        // the clean sample is shared by all filters (L1 / L2 resident) and is fetched here, at its use: the
                        // Philox rounds of the noise cover the load
                        double raw[6], tb[6], ud[6];
                        in.raw_imu(a.in, kk, raw);
                        true_bias_now(tb);
                        synth_imu(a.ns, in.gid, kk, raw, tb, ud);
#pragma unroll
                        for (int cc = 0; cc < 6; ++cc) u[cc] = (T)ud[cc];
                    } else {
                        in.imu(a.ns, kk, un, u);
                    }
                    prediction_step<T, BIAS>(s, P, u, par, accel);
                    ++np_run;
                }
                if (gate) { want = true; break; }        // tick kk: predicted, correction pending
                if (init) {
                    up += 1;
                    fl = (fl & ~FLAG_CORRECTED) | FLAG_ACTIVE;
                }
                ++kk;
                if (!SYNTH && kk < k_end) in.raw_imu(kk, un);
                if (kk == next_fence) { at_fence = true; break; }          // tick kk-1 was a sampling tick
                if (kk >= k_end) break;
            }
            k = kk; upds = up; flags = fl; next_tag_step = nts;
            n_pred += np_run;
            predicted = want;
        }
        const bool active = (k < k_end) && !at_fence;
        const int32_t fl0 = flags;
        const CtaVote v = cta_vote(vbuf, iter, active, want, want && held >= patience, at_fence || k >= k_end, at_fence);
        if (v.active == 0 && v.at_fence == 0) break;     // every lane of the CTA has finished
        ++n_iter;
        if (do_stats && v.fenced == v.lanes && v.at_fence != 0) {
            // every lane is at the fence (or finished): sample together, then resume on the next iteration
            const bool mine = live && at_fence && (fl0 & FLAG_INIT);
            double tb[6] = { 0, 0, 0, 0, 0, 0 };
            if (SYNTH) true_bias_now(tb);
            stats_sample<T, BIAS, PS, true, SYNTH>(a, i, (int64_t)k - 1, s, P, tb, mine);
            if (mine) ++n_sexec;
            at_fence = false;
            next_fence += a.stats.stride;
        }
        // (every active lane is waiting for a correction here, so the wanting lanes are always a majority of the active
        //  ones; the hold logic stays for CTAs of the per-tick interface, where it is a no-op too)
        bool serve = true;
        if (v.want != 0) serve = (2 * v.want > v.active) || v.out_of_patience;
        if (want && !serve) ++held;

#if defined(__CUDA_ARCH__) && defined(QEKF_DIAG_EVENTS)
        if (__ballot_sync(0xffffffffu, want && serve) != 0u) ++n_cev;    // diagnostics: iterations in which this warp runs the correction
#endif
        if (want && serve) {
            // ---- consume the measurement, corner-margin gate (cpp:150-186), single-rate correction (cpp:265-279) ----
            T tag[7];
            double tg[7];       // the gate decides on the double pose
            if (pend_m >= 0) {
                in.tag_f64(a.in, a.ns, pend_m, tg);
            } else {
#pragma unroll
                for (int cc = 0; cc < 7; ++cc) tg[cc] = a.st.pend[cc * a.st.ld + i];
            }
#pragma unroll
            for (int cc = 0; cc < 7; ++cc) tag[cc] = (T)tg[cc];
            flags &= ~FLAG_READY;
            const bool perform = c.corner_margin_enbl ? corner_gate<T>(tg, c) : true;
            held = 0;
            if (perform) {
                ++n_corr;
                Observation<T> obs;
                // inlined: behind a call (as it was while the loop iterated over ticks, to keep its ~120 live doubles out of
                // the per-tick register allocation) everything the inner loop carries was spilled around it: 6.66e9 -> 7.09e9
                correction_step<T, BIAS, DIRECT>(s, P, tag, par, obs);
#pragma unroll
                for (int cc = 0; cc < 3; ++cc) a.st.aux[(3 + cc) * a.st.ld + i] = obs.r_t_vt_obs[cc];
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) a.st.aux[(6 + cc) * a.st.ld + i] = obs.q_tv_obs[cc];
                upds = 0;
                flags |= FLAG_CORRECTED;
            } else {
                upds += 1;
                flags &= ~FLAG_CORRECTED;
            }
            flags |= FLAG_ACTIVE;
            predicted = false;
            ++k;
            if (!SYNTH && k < k_end) in.raw_imu(k, un);
            if (k == next_fence) at_fence = true;        // tick k-1 was a sampling tick
        }
    }
    if (!live) return;

    // a latched, still unconsumed measurement survives the launch in st.pend
    if ((flags & FLAG_READY) && pend_m >= 0) {
        double tg[7];
        in.tag_f64(a.in, a.ns, pend_m, tg);
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) a.st.pend[cc * a.st.ld + i] = tg[cc];
        a.st.pend[7 * a.st.ld + i] = a.in.tag_stamp[pend_m];
    }
    store_filter<T>(a.st, i, s, P);
    a.st.flags[i] = flags;
    a.st.upds[i] = upds;
    if (a.st.counts) {
#ifdef __CUDA_ARCH__
        atomicAdd(a.st.counts + 0, (unsigned long long)(uint32_t)(int32_t)n_pred);
        atomicAdd(a.st.counts + 1, (unsigned long long)(uint32_t)(int32_t)n_corr);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(a.st.counts + 2, (unsigned long long)(uint32_t)(int32_t)n_iter);   // loop iterations per warp
            atomicAdd(a.st.counts + 3, (unsigned long long)n_cev);    // ... of which the warp ran the correction
        }
        atomicAdd(a.st.counts + 4, (unsigned long long)n_sexec);
#else
        a.st.counts[0] += (uint32_t)(int32_t)n_pred;
        a.st.counts[1] += (uint32_t)(int32_t)n_corr;
#endif
    }
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) a.st.aux[cc * a.st.ld + i] = accel[cc];
}

// ------------------------------------------------------------------------------------------------
// delayed-measurement fusion (multirate_ekf = true), evaluated lazily
// ------------------------------------------------------------------------------------------------
template <typename T, class PS>
QEKF_FN void load_checkpoint(const DeviceState<T> &st, int64_t i, Nominal<T> &s, PS &P)
{
    DeviceState<T> v = st;
    v.x = st.xc; v.P = st.Pc;
    load_filter<T>(v, i, s, P);
}
template <typename T, class PS>
QEKF_FN void store_checkpoint(const DeviceState<T> &st, int64_t i, const Nominal<T> &s, const PS &P)
{
    DeviceState<T> v = st;
    v.x = st.xc; v.P = st.Pc;
    store_filter<T>(v, i, s, P);
}

template <typename T> QEKF_FN void prefetch_l2(const T *p)
{
#ifdef __CUDA_ARCH__
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

// n consecutive prediction_steps through the stored IMU inputs of ring slots first, first+1, ... (mod L).
// (Streaming loads / stores, __ldcs / __stcs, for the ring were measured and cost 8 %: 4.17e9 -> 3.86e9 filter-steps/s.)
// One out-of-line copy of the prediction code serves the replay before a delayed correction, the checkpoint
// catch-up and the materialisation of the head, so the whole multirate tick loop stays small.
template <typename T, bool BIAS, class PS, class PAR>
QEKF_COLD void advance_call(Nominal<T> *sp, PS &P, const PAR par, const T *ring_i, int64_t ld, int32_t L, int32_t first,
                            int32_t n, T *accel_out)
{
    if (n <= 0) return;
    Nominal<T> s = *sp;
    T acc[3] = { accel_out[0], accel_out[1], accel_out[2] };
    int32_t slot = first;
    T u[6];
#pragma unroll
    for (int cc = 0; cc < 6; ++cc) u[cc] = ring_i[((int64_t)slot * 6 + cc) * ld];
    for (int32_t j = 0; j < n; ++j) {
        slot = (slot + 1 == L) ? 0 : slot + 1;
        // the next entry's input: asked for now (an L2 prefetch holds no registers through the prediction, where a
        // register prefetch cost 12 and pushed as many values of the covariance code into local memory), loaded after
        if (j + 1 < n) {
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) prefetch_l2(ring_i + ((int64_t)slot * 6 + cc) * ld);
        }
        prediction_step<T, BIAS>(s, P, u, par, acc);
        if (j + 1 < n) {
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) u[cc] = ring_i[((int64_t)slot * 6 + cc) * ld];
        }
    }
    *sp = s;
    accel_out[0] = acc[0]; accel_out[1] = acc[1]; accel_out[2] = acc[2];
}

// The multirate replay loop of one filter.  Semantics: filter_update with multirate_ekf = true
// (cpp:196-264).  Mechanics: the registers / shared memory hold the CHECKPOINT (oldest retained history
// entry), not the head.  A tick only appends its IMU sample to the ring (the head prediction of cpp:240-257 is
// implied, not executed).  A correction with step delay d lands on history entry size-d: the checkpoint is
// advanced to that entry (ind_rel prediction_steps), corrected there, and becomes the new oldest entry
// (cpp:206-218); the re-propagation of cpp:222-226 is again implied.  The head is materialised (nh
// prediction_steps on a copy) only where somebody looks at it: at the end of the launch and at statistics
// samples.  Every history entry is the same pure function of (checkpoint, ring) the reference evaluates, so
// the results are bit-identical to the eager evaluation, for ~1 prediction per tick instead of ~2.
// Ring invariant: nh <= L - 1 before a push and the checkpoint never passes entry size-D (D = largest possible
// step delay), so every index a future correction can address is still reachable.  Lanes that do not correct
// (tag dropout, rejected detection) catch their checkpoint up to size-D inside their CTA-mates' correction
// events, where the warp executes prediction code anyway.
template <typename T, bool BIAS, bool DIRECT, bool SYNTH, bool PF, class PS, bool CSM = false, bool STATS = SYNTH>
QEKF_FN void run_filter_mr(const RunArgs<T> &a, const int64_t i_in, PS &P, int32_t *scr, const int scr_stride,
                           const bool live = true, int *vbuf = nullptr, const Consts<T> *c_cold = nullptr)
{
    const Consts<T> &c = a.c;
    const int64_t i = live ? i_in : 0;
    const typename ParSel<T, PF>::type par = ParSel<T, PF>::make(a.c, a.st, i);
    const auto par_cold = ParSel<T, PF>::make_cold(par, c_cold, a.st, i, std::integral_constant<bool, CSM>());   // see run_filter
    const int64_t k_end = a.k0 + a.n_steps;
    const int32_t L = a.st.ring_len, Dm1 = a.st.dmax_m1;
    T *ring_i = a.st.ring + i;
    Nominal<T> s;                      // the checkpoint
    SmemInt flags{ scr + 0 * scr_stride }, upds{ scr + 1 * scr_stride }, nh{ scr + 2 * scr_stride };
    SmemInt hpos{ scr + 3 * scr_stride }, hlen{ scr + 4 * scr_stride }, m{ scr + 5 * scr_stride };
    SmemInt next_tag_step{ scr + 6 * scr_stride }, pend_m{ scr + 7 * scr_stride }, held{ scr + 8 * scr_stride };
    SmemInt k{ scr + 9 * scr_stride };       // tick index (qekf_run bounds it to int32)
    SmemInt n_pred{ scr + 16 * scr_stride }, pstart{ scr + 17 * scr_stride };
    flags = 0; upds = 0; nh = 0; hpos = 0; hlen = 0; n_pred = 0; pstart = INT32_MAX;
    T accel[3] = { T(0), T(0), T(0) };
    Inputs<T, SYNTH> in;
    k = (int32_t)k_end;
    if (live) {
        load_checkpoint<T>(a.st, i, s, P);
        flags = a.st.flags[i];
        upds = a.st.upds[i];
        nh = a.st.nh[i]; hpos = a.st.hpos[i]; hlen = a.st.hlen[i];
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) accel[cc] = a.st.aux[cc * a.st.ld + i];
        in.init(a, i, a.st.gid_perm ? (int64_t)a.st.gid_perm[i] : i);
        k = (int32_t)a.k0;
        if (SYNTH) pstart = in.priv_start;
        if (SYNTH) {                   // the true bias as its six normals, in the scratch (12 registers less across calls)
            float z[6];
            normals6(a.ns, in.gid, STREAM_BIAS, 0u, z);
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) reinterpret_cast<float *>(scr)[(10 + cc) * scr_stride] = z[cc];
        }
    }
    auto true_bias_now = [&](double b[6]) {
#pragma unroll
        for (int cc = 0; cc < 6; ++cc)
            b[cc] = (double)(cc < 3 ? a.ns.sig_ba : a.ns.sig_bw) * (double)reinterpret_cast<const float *>(scr)[(10 + cc) * scr_stride];
    };

    uint32_t n_corr = 0, n_iter = 0, n_sexec = 0;
    m = a.m0;
    next_tag_step = (m < a.in.M) ? a.in.tag_step[m] : INT32_MAX;
    pend_m = -1;
    held = 0;
    bool at_fence = false;
    const bool do_stats = STATS && a.stats.acc != nullptr;          // see run_filter
    const int32_t patience = c.limit_measurement_freq ? (c.upd_per_meas - 1) : 0;
    int32_t next_fence = do_stats ? (int32_t)((a.k0 / a.stats.stride + 1) * a.stats.stride) : INT32_MAX;   // see run_filter

    cta_vote_init(vbuf);
    for (uint32_t iter = 0;; ++iter) {
        const bool active = (k < k_end) && !at_fence;

        // ---- AprilTagSubCallback for the arrival scheduled at tick k (node.cpp:153-176) ----
        if (active && k == next_tag_step) {
            if (in.valid(a.in, a.ns, m, (int32_t)k, pstart)) {
                pend_m = m;
                flags |= FLAG_READY;
                if (!(flags & FLAG_INIT)) {
                    T tag0[7];
                    in.tag(a.in, a.ns, m, tag0);
                    initialize_state<T, BIAS>(s, P, tag0, par, false);
                    flags |= FLAG_INIT;
                    nh = 0; hlen = 1;                    // history <- single entry (cpp:326-339)
                }
            }
            ++m;
            next_tag_step = (m < a.in.M) ? a.in.tag_step[m] : INT32_MAX;
        }

        const bool want = active && (flags & FLAG_INIT) && (flags & FLAG_READY) &&
                          (!c.limit_measurement_freq || (upds + 1) >= c.upd_per_meas);
        const CtaVote v = cta_vote(vbuf, iter, active, want, want && held >= patience, at_fence || k >= k_end, at_fence);
        if (v.active == 0 && v.at_fence == 0) break;
        ++n_iter;
        if (do_stats && v.fenced == v.lanes && v.at_fence != 0) {
            // look at the head: park the checkpoint, replay the nh implied predictions, sample, come back
            const bool mine = live && at_fence && (flags & FLAG_INIT);
            Nominal<T> head = s;
            if (mine) {
                store_checkpoint<T>(a.st, i, s, P);
                int32_t first = hpos - nh + 1;
                if (first < 0) first += L;
                advance_call<T, BIAS>(&head, P, par_cold, ring_i, a.st.ld, L, first, nh, accel);
                n_pred += nh;
            }
            double tb[6] = { 0, 0, 0, 0, 0, 0 };
            if (SYNTH) true_bias_now(tb);
            stats_sample<T, BIAS, PS, true, SYNTH>(a, i, k - 1, head, P, tb, mine);
            if (mine) {
                load_checkpoint<T>(a.st, i, s, P);
                ++n_sexec;
            }
            at_fence = false;
            next_fence += a.stats.stride;
        }
        bool serve = true;
        if (v.want != 0) serve = (2 * v.want > v.active) || v.out_of_patience;
        const bool event = (v.want != 0) && serve;       // CTA-uniform: corrections are being served now
        if (want && !serve) ++held;
        const bool exec = active && !(want && !serve) && (flags & FLAG_INIT);

        // ---- consume the measurement, corner-margin gate (cpp:150-186) ----
        bool perform = false;
        T tag[7];
        double stamp = 0;
        if (exec && want) {
            double tg[7];       // the gate decides on the double pose
            if (pend_m >= 0) {
                in.tag_f64(a.in, a.ns, pend_m, tg);
                stamp = a.in.tag_stamp[pend_m];
            } else {
#pragma unroll
                for (int cc = 0; cc < 7; ++cc) tg[cc] = a.st.pend[cc * a.st.ld + i];
                stamp = a.st.pend[7 * a.st.ld + i];
            }
#pragma unroll
            for (int cc = 0; cc < 7; ++cc) tag[cc] = (T)tg[cc];
            flags &= ~FLAG_READY;
            perform = c.corner_margin_enbl ? corner_gate<T>(tg, c) : true;
            held = 0;
        }

        // ---- how far this lane moves its checkpoint now ----
        int32_t n_adv = 0;
        if (perform) {
            // cpp:199-201
            const double t_curr = a.in.t_start + (double)k / a.in.update_freq;
            const double delay = c.dynamic_meas_delay ? fmin(t_curr - stamp + par.dyn_offset(), c.meas_delay_max)
                                                      : par.meas_delay();
            int32_t step = (int32_t)(delay / c.dT_nom + 0.5);
            if (step < 1) step = 1;
            int32_t ind = hlen - step;
            if (ind < 0) ind = 0;
            n_adv = ind - (hlen - 1 - nh);               // >= 0 by the ring invariant
            if (n_adv < 0) n_adv = 0;
            a.st.aux[10 * a.st.ld + i] = (T)delay;       // measurement_delay_curr
        } else if ((flags & FLAG_INIT) && active && (event || (exec && nh >= L - 1))) {
            n_adv = (nh > Dm1) ? nh - Dm1 : 0;           // catch-up (never past entry size-D)
        }
        if (event || n_adv > 0) {
            int32_t first = hpos - nh + 1;
            if (first < 0) first += L;
            T scratch[3] = { T(0), T(0), T(0) };
            advance_call<T, BIAS>(&s, P, par_cold, ring_i, a.st.ld, L, first, n_adv, scratch);
            nh -= n_adv;
            n_pred += n_adv;
        }
        if (perform) {
            ++n_corr;
            Observation<T> obs;
            correction_call<T, BIAS, DIRECT>(&s, P, tag, par_cold, &obs);
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) a.st.aux[(3 + cc) * a.st.ld + i] = obs.r_t_vt_obs[cc];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) a.st.aux[(6 + cc) * a.st.ld + i] = obs.q_tv_obs[cc];
            hlen = nh + 1;                               // history before the corrected entry is erased (cpp:214-219)
        }
        if (exec) {
            // cpp:240-257: the head prediction is implied; its input joins the history
            // (the raw sample is fetched here rather than prefetched across iterations: whatever is carried across the
            // out-of-line calls of this loop lives in local memory, and nothing on the control path waits for this load)
            T u[6];
            {
                double un[6];
                in.raw_imu(a.in, k, un);
                if (SYNTH) {
                    double tb[6], ud[6];
                    true_bias_now(tb);
                    synth_imu(a.ns, in.gid, k, un, tb, ud);
#pragma unroll
                    for (int cc = 0; cc < 6; ++cc) u[cc] = (T)ud[cc];
                } else {
                    in.imu(a.ns, k, un, u);
                }
            }
            hpos = (hpos + 1 == L) ? 0 : hpos + 1;
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) ring_i[((int64_t)hpos * 6 + cc) * a.st.ld] = u[cc];
            ++nh; ++hlen;
            if (perform) { upds = 0; flags |= FLAG_CORRECTED; }
            else { upds += 1; flags &= ~FLAG_CORRECTED; }
            flags |= FLAG_ACTIVE;
        }
        if (active && !(want && !serve)) {
            ++k;
            if (k == next_fence) at_fence = true;
        }
    }
    if (!live) return;

    if ((flags & FLAG_READY) && pend_m >= 0) {
        double tg[7];
        in.tag_f64(a.in, a.ns, pend_m, tg);
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) a.st.pend[cc * a.st.ld + i] = tg[cc];
        a.st.pend[7 * a.st.ld + i] = a.in.tag_stamp[pend_m];
    }
    // checkpoint home, then the head (what the accessors read: r_nom ... cov_pert, accel_rel)
    // (an uninitialised filter keeps the constructor's state: cpp:129-130 returns before touching anything)
    if (flags & FLAG_INIT) {
        store_checkpoint<T>(a.st, i, s, P);
        int32_t first = hpos - nh + 1;
        if (first < 0) first += L;
        advance_call<T, BIAS>(&s, P, par_cold, ring_i, a.st.ld, L, first, nh, accel);
        n_pred += nh;
        store_filter<T>(a.st, i, s, P);
    }
    a.st.flags[i] = flags;
    a.st.upds[i] = upds;
    a.st.nh[i] = nh; a.st.hpos[i] = hpos; a.st.hlen[i] = hlen;
    if (a.st.counts) {
#ifdef __CUDA_ARCH__
        atomicAdd(a.st.counts + 0, (unsigned long long)(uint32_t)(int32_t)n_pred);
        atomicAdd(a.st.counts + 1, (unsigned long long)n_corr);
        if ((i & 31) == 0) atomicAdd(a.st.counts + 2, (unsigned long long)n_iter);
        atomicAdd(a.st.counts + 4, (unsigned long long)n_sexec);
#else
        a.st.counts[0] += (uint32_t)(int32_t)n_pred;
        a.st.counts[1] += n_corr;
#endif
    }
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) a.st.aux[cc * a.st.ld + i] = accel[cc];
}

// ------------------------------------------------------------------------------------------------
// delayed-measurement fusion of a Monte-Carlo launch: no ring, no light ticks
// ------------------------------------------------------------------------------------------------
// In a Monte-Carlo launch u_hist[k] is a pure function of (seed, filter id, k): the entries after the checkpoint need
// no storage, they are re-synthesised where the replay consumes them.  A tick that fuses nothing then has no work left
// at all (the head prediction is implied, its input is implied), so the loop below does not iterate over ticks: every
// lane jumps straight to its next decision point -- the tick whose measurement gate opens, a sampling boundary, the end
// of the launch -- handling tag arrivals on the way, and the CTA only meets (one vote, one barrier) where lanes fuse
// measurements or sample statistics.  Lanes whose tick indices differ (private dropouts) reach their correction ticks
// in the same iteration, so the time skew costs nothing here.  Same arithmetic on the same inputs as run_filter_mr
// with SYNTH = true: the results are bit-identical (tests/test_gpu_multirate.py, test_gpu_reorder.py).

// n consecutive prediction_steps whose inputs are the synthesised IMU samples of ticks tick0, tick0+1, ...
// bz: the true bias' six normals (shared-memory scratch, stride bz_stride).  ring_out != nullptr: the samples are also
// written to ring slots 0, 1, ... of this filter (the launch epilogue leaves a valid ring behind for the entry points
// that read it: per-tick interface, explicit streams).
template <typename T, bool BIAS, class PS, class PAR>
QEKF_COLD void advance_synth_call(Nominal<T> *sp, PS &P, const PAR par, const double *imu_clean, const ImuSynth nz, int64_t gid,
                                  const float *bz, int bz_stride, int32_t tick0, int32_t n, T *accel_out, T *ring_out, int64_t ld)
{
    if (n <= 0) return;
    Nominal<T> s = *sp;
    T acc[3] = { accel_out[0], accel_out[1], accel_out[2] };
    for (int32_t j = 0; j < n; ++j) {
        const int64_t k = (int64_t)tick0 + j;
        T u[6];
        {
            double raw[6], tb[6], ud[6];
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) raw[cc] = imu_clean[k * 6 + cc];
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) tb[cc] = (double)(cc < 3 ? nz.sig_ba : nz.sig_bw) * (double)bz[cc * bz_stride];
            synth_imu(nz, gid, k, raw, tb, ud);
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) u[cc] = (T)ud[cc];
        }
        if (ring_out) {
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) ring_out[((int64_t)j * 6 + cc) * ld] = u[cc];
        }
        prediction_step<T, BIAS>(s, P, u, par, acc);
    }
    *sp = s;
    accel_out[0] = acc[0]; accel_out[1] = acc[1]; accel_out[2] = acc[2];
}

template <typename T, bool BIAS, bool DIRECT, bool PF, class PS, bool CSM = false>
QEKF_FN void run_filter_mrs(const RunArgs<T> &a, const int64_t i_in, PS &P, int32_t *scr, const int scr_stride,
                            const bool live = true, int *vbuf = nullptr, const Consts<T> *c_cold = nullptr)
{
    const Consts<T> &c = a.c;
    const int64_t i = live ? i_in : 0;
    const typename ParSel<T, PF>::type par = ParSel<T, PF>::make(a.c, a.st, i);
    const auto par_cold = ParSel<T, PF>::make_cold(par, c_cold, a.st, i, std::integral_constant<bool, CSM>());
    const int32_t k_end = (int32_t)(a.k0 + a.n_steps);
    const int32_t Dm1 = a.st.dmax_m1;
    Nominal<T> s;                      // the checkpoint
    SmemInt flags{ scr + 0 * scr_stride }, upds{ scr + 1 * scr_stride }, nh{ scr + 2 * scr_stride };
    SmemInt hlen{ scr + 4 * scr_stride }, m{ scr + 5 * scr_stride };
    SmemInt next_tag_step{ scr + 6 * scr_stride }, pend_m{ scr + 7 * scr_stride }, held{ scr + 8 * scr_stride };
    SmemInt k{ scr + 9 * scr_stride };
    SmemInt n_pred{ scr + 16 * scr_stride }, pstart{ scr + 17 * scr_stride };
    const float *bz = reinterpret_cast<const float *>(scr) + 10 * scr_stride;
    flags = 0; upds = 0; nh = 0; hlen = 0; n_pred = 0; pstart = INT32_MAX;
    T accel[3] = { T(0), T(0), T(0) };
    Inputs<T, true> in;
    k = k_end;
    if (live) {
        load_checkpoint<T>(a.st, i, s, P);
        flags = a.st.flags[i];
        upds = a.st.upds[i];
        nh = a.st.nh[i]; hlen = a.st.hlen[i];
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) accel[cc] = a.st.aux[cc * a.st.ld + i];
        in.init(a, i, a.st.gid_perm ? (int64_t)a.st.gid_perm[i] : i);
        k = (int32_t)a.k0;
        pstart = in.priv_start;
        float z[6];
        normals6(a.ns, in.gid, STREAM_BIAS, 0u, z);
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) reinterpret_cast<float *>(scr)[(10 + cc) * scr_stride] = z[cc];
    }
    const ImuSynth nz{ a.ns.seed, a.ns.sig_a, a.ns.sig_w, a.ns.sig_ba, a.ns.sig_bw };
    // advance *sp by n entries starting with the input of tick t0
    auto advance = [&](Nominal<T> *sp, int32_t t0, int32_t n, T *acc, T *ring_out) {
        advance_synth_call<T, BIAS>(sp, P, par_cold, a.in.imu, nz, in.gid, bz, scr_stride, t0, n, acc, ring_out, a.st.ld);
        if (n > 0) n_pred += n;
    };

    uint32_t n_corr = 0, n_iter = 0, n_sexec = 0;
    m = a.m0;
    next_tag_step = (m < a.in.M) ? a.in.tag_step[m] : INT32_MAX;
    pend_m = -1;
    held = 0;
    bool at_fence = false;
    const bool do_stats = a.stats.acc != nullptr;
    const int32_t patience = c.limit_measurement_freq ? (c.upd_per_meas - 1) : 0;
    int32_t next_fence = do_stats ? (int32_t)((a.k0 / a.stats.stride + 1) * a.stats.stride) : INT32_MAX;

    cta_vote_init(vbuf);
    for (uint32_t iter = 0;; ++iter) {
        // ---- to this lane's next decision point: the tag callbacks on the way (node.cpp:153-176), and every tick that
        //      fuses nothing as counters only (its entry joins the history: cpp:240-257) ----
        bool want = false;
        if (k < k_end && !at_fence) {
            for (;;) {
                if (k == next_tag_step) {
                    if (in.valid(a.in, a.ns, m, (int32_t)k, pstart)) {
                        pend_m = m;
                        flags |= FLAG_READY;
                        if (!(flags & FLAG_INIT)) {
                            T tag0[7];
                            in.tag(a.in, a.ns, m, tag0);
                            initialize_state<T, BIAS>(s, P, tag0, par, false);
                            flags |= FLAG_INIT;
                            nh = 0; hlen = 1;                    // history <- single entry (cpp:326-339)
                        }
                    }
                    ++m;
                    next_tag_step = (m < a.in.M) ? a.in.tag_step[m] : INT32_MAX;
                }
                const int32_t fl = flags, up = upds, kk = k;
                const bool init = (fl & FLAG_INIT) != 0, armed = init && (fl & FLAG_READY);
                // ticks until the gate of cpp:147 opens (0: this tick fuses)
                const int32_t t_gate = !armed ? INT32_MAX : (c.limit_measurement_freq ? max(0, c.upd_per_meas - 1 - up) : 0);
                if (t_gate == 0) { want = true; break; }
                int32_t q = min(min(t_gate, next_tag_step - kk), min(next_fence - kk, k_end - kk));   // >= 1
                if (init) {
                    nh += q; hlen += q; upds = up + q;
                    flags = (fl & ~FLAG_CORRECTED) | FLAG_ACTIVE;
                }
                k = kk + q;
                if (kk + q == next_fence) { at_fence = true; break; }     // tick k-1 was a sampling tick
                if (kk + q >= k_end) break;
            }
        }
        const bool active = (k < k_end) && !at_fence;
        const CtaVote v = cta_vote(vbuf, iter, active, want, want && held >= patience, at_fence || k >= k_end, at_fence);
        if (v.active == 0 && v.at_fence == 0) break;
        ++n_iter;
        if (do_stats && v.fenced == v.lanes && v.at_fence != 0) {
            // look at the head: bring the checkpoint as far as any future correction allows, park it, replay the rest on
            // a copy, sample, come back
            const bool mine = live && at_fence && (flags & FLAG_INIT);
            Nominal<T> head = s;
            if (mine) {
                const int32_t n_c = (nh > Dm1) ? nh - Dm1 : 0;
                T scratch[3] = { T(0), T(0), T(0) };
                advance(&s, k - nh, n_c, scratch, nullptr);
                nh -= n_c;
                head = s;
                store_checkpoint<T>(a.st, i, s, P);
                advance(&head, k - nh, nh, accel, nullptr);
            }
            double tb[6] = { 0, 0, 0, 0, 0, 0 };
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) tb[cc] = (double)(cc < 3 ? nz.sig_ba : nz.sig_bw) * (double)bz[cc * scr_stride];
            stats_sample<T, BIAS>(a, i, (int64_t)k - 1, head, P, tb, mine);
            if (mine) {
                load_checkpoint<T>(a.st, i, s, P);
                ++n_sexec;
            }
            at_fence = false;
            next_fence += a.stats.stride;
        }
        bool serve = true;
        if (v.want != 0) serve = (2 * v.want > v.active) || v.out_of_patience;
        const bool event = (v.want != 0) && serve;       // CTA-uniform: corrections are being served now
        if (want && !serve) ++held;
        const bool exec = want && serve;                 // (a lane that wants is active and initialised)

        // ---- consume the measurement, corner-margin gate (cpp:150-186) ----
        bool perform = false;
        T tag[7];
        double stamp = 0;
        if (exec) {
            double tg[7];       // the gate decides on the double pose
            if (pend_m >= 0) {
                in.tag_f64(a.in, a.ns, pend_m, tg);
                stamp = a.in.tag_stamp[pend_m];
            } else {
#pragma unroll
                for (int cc = 0; cc < 7; ++cc) tg[cc] = a.st.pend[cc * a.st.ld + i];
                stamp = a.st.pend[7 * a.st.ld + i];
            }
#pragma unroll
            for (int cc = 0; cc < 7; ++cc) tag[cc] = (T)tg[cc];
            flags &= ~FLAG_READY;
            perform = c.corner_margin_enbl ? corner_gate<T>(tg, c) : true;
            held = 0;
        }
        // ---- how far this lane moves its checkpoint now ----
        int32_t n_adv = 0;
        if (perform) {
            // cpp:199-201
            const double t_curr = a.in.t_start + (double)k / a.in.update_freq;
            const double delay = c.dynamic_meas_delay ? fmin(t_curr - stamp + par.dyn_offset(), c.meas_delay_max)
                                                      : par.meas_delay();
            int32_t step = (int32_t)(delay / c.dT_nom + 0.5);
            if (step < 1) step = 1;
            int32_t ind = hlen - step;
            if (ind < 0) ind = 0;
            n_adv = ind - (hlen - 1 - nh);               // >= 0: the checkpoint never passes entry size-D
            if (n_adv < 0) n_adv = 0;
            a.st.aux[10 * a.st.ld + i] = (T)delay;       // measurement_delay_curr
        } else if (event && want && (flags & FLAG_INIT)) {
            n_adv = (nh > Dm1) ? nh - Dm1 : 0;           // held or rejected: catch up inside the CTA-mates' event
        }
        if (event) {
            // the replay before a delayed correction, inlined: the one place where predictions run in bulk (the calls of
            // `advance` serve the sampling and the epilogue).  A loop without calls on a copy that never leaves registers.
            if (n_adv > 0) {
                Nominal<T> sl = s;
                T scratch[3] = { T(0), T(0), T(0) };
                const int32_t t0 = k - nh;
                for (int32_t j = 0; j < n_adv; ++j) {
                    T u[6];
                    {
                        double raw[6], tb[6], ud[6];
                        in.raw_imu(a.in, (int64_t)(t0 + j), raw);
#pragma unroll
                        for (int cc = 0; cc < 6; ++cc) tb[cc] = (double)(cc < 3 ? nz.sig_ba : nz.sig_bw) * (double)bz[cc * scr_stride];
                        synth_imu(nz, in.gid, (int64_t)(t0 + j), raw, tb, ud);
#pragma unroll
                        for (int cc = 0; cc < 6; ++cc) u[cc] = (T)ud[cc];
                    }
                    prediction_step<T, BIAS>(sl, P, u, par, scratch);
                }
                s = sl;
                n_pred += n_adv;
                nh -= n_adv;
            }
        }
        if (perform) {
            ++n_corr;
            Observation<T> obs;
            {
                Nominal<T> sl = s;                       // (inlined on a copy that never leaves registers, like the replay)
                correction_step<T, BIAS, DIRECT>(sl, P, tag, par, obs);
                s = sl;
            }
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) a.st.aux[(3 + cc) * a.st.ld + i] = obs.r_t_vt_obs[cc];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) a.st.aux[(6 + cc) * a.st.ld + i] = obs.q_tv_obs[cc];
            hlen = nh + 1;                               // history before the corrected entry is erased (cpp:214-219)
        }
        if (exec) {
            // cpp:240-257: the head prediction of tick k is implied; its (implied) input joins the history
            ++nh; ++hlen;
            if (perform) { upds = 0; flags |= FLAG_CORRECTED; }
            else { upds += 1; flags &= ~FLAG_CORRECTED; }
            flags |= FLAG_ACTIVE;
            ++k;
            if (k == next_fence) at_fence = true;
        }
    }
    if (!live) return;

    if ((flags & FLAG_READY) && pend_m >= 0) {
        double tg[7];
        in.tag_f64(a.in, a.ns, pend_m, tg);
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) a.st.pend[cc * a.st.ld + i] = tg[cc];
        a.st.pend[7 * a.st.ld + i] = a.in.tag_stamp[pend_m];
    }
    // checkpoint home (as far forward as any future correction allows), then the head (what the accessors read); the
    // inputs of the entries in between go to ring slots 0 .. nh-1 for whoever continues from this state
    int32_t hp = 0;
    if (flags & FLAG_INIT) {
        const int32_t n_c = (nh > Dm1) ? nh - Dm1 : 0;
        T scratch[3] = { T(0), T(0), T(0) };
        advance(&s, k - nh, n_c, scratch, nullptr);
        nh -= n_c;
        store_checkpoint<T>(a.st, i, s, P);
        advance(&s, k - nh, nh, accel, a.st.ring + i);
        store_filter<T>(a.st, i, s, P);
        hp = (nh > 0) ? nh - 1 : 0;
    }
    a.st.flags[i] = flags;
    a.st.upds[i] = upds;
    a.st.nh[i] = nh; a.st.hpos[i] = hp; a.st.hlen[i] = hlen;
    if (a.st.counts) {
#ifdef __CUDA_ARCH__
        atomicAdd(a.st.counts + 0, (unsigned long long)(uint32_t)(int32_t)n_pred);
        atomicAdd(a.st.counts + 1, (unsigned long long)n_corr);
        if ((i & 31) == 0) atomicAdd(a.st.counts + 2, (unsigned long long)n_iter);
        atomicAdd(a.st.counts + 4, (unsigned long long)n_sexec);
#else
        a.st.counts[0] += (uint32_t)(int32_t)n_pred;
        a.st.counts[1] += n_corr;
#endif
    }
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) a.st.aux[cc * a.st.ld + i] = accel[cc];
}

// CTA-cooperative copy of the launch-wide constants into shared memory (whole 8-byte words; VOTE_WORDS and the
// scratch sizes keep the destination 8-byte aligned)
template <typename T> __device__ __forceinline__ void copy_consts(Consts<T> *dst, const Consts<T> &src)
{
#ifdef __CUDA_ARCH__
    static_assert(sizeof(Consts<T>) % 8 == 0, "Consts is copied in 8-byte words");
    const unsigned long long *s = reinterpret_cast<const unsigned long long *>(&src);
    unsigned long long *d = reinterpret_cast<unsigned long long *>(dst);
    for (unsigned w = threadIdx.x; w < sizeof(Consts<T>) / 8; w += blockDim.x) d[w] = s[w];
#endif
}
constexpr size_t consts_smem_bytes(size_t consts_size) { return (consts_size + 15) / 16 * 16; }

// fused multi-tick replay: MR = false single-rate filter, MR = true delayed-measurement fusion; STATS: see run_filter
template <typename T, bool BIAS, bool DIRECT, bool SYNTH, bool MR, bool PF, int BLOCK, bool STATS = SYNTH>
__global__ void __launch_bounds__(BLOCK, 1) run_kernel(const __grid_constant__ RunArgs<T> a)
{
    constexpr int N = BIAS ? 15 : 9;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sm = reinterpret_cast<T *>(smem_raw);
    const int64_t slot = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    const bool live = slot < a.st.n;
    const int64_t i = slot;      // (a reordered launch has its arrays in slot order: DeviceState::gid_perm)
    PShared<T, N, BLOCK> P{ sm + threadIdx.x };
#ifdef QEKF_EXP8
    int *vbuf = reinterpret_cast<int *>(sm + (size_t)BLOCK * ((sizeof(T) == 8 && N == 15) ? 105 : N * (N + 1) / 2));
#else
    int *vbuf = reinterpret_cast<int *>(sm + (size_t)BLOCK * (N * (N + 1) / 2));
#endif
    // behind the vote words: the sequencer's integers, then a copy of the launch-wide constants for the out-of-line calls
    int32_t *scr = vbuf + VOTE_WORDS;
    Consts<T> *csm = reinterpret_cast<Consts<T> *>(scr + (size_t)BLOCK * (MR ? MR_SCRATCH_INTS : SR_SCRATCH_INTS));
#ifndef QEKF_EXP8
    copy_consts(csm, a.c);             // (published by the barrier of cta_vote_init)
#else
    csm = nullptr;
#endif
    // padding lanes still take part in the votes
#ifndef QEKF_EXP8
    if constexpr (MR && SYNTH) {
        if (a.st.hist_synth) run_filter_mrs<T, BIAS, DIRECT, PF, PShared<T, N, BLOCK>, true>(a, i, P, scr + threadIdx.x, BLOCK, live, vbuf, csm);
        else run_filter_mr<T, BIAS, DIRECT, SYNTH, PF, PShared<T, N, BLOCK>, true, STATS>(a, i, P, scr + threadIdx.x, BLOCK, live, vbuf, csm);
    } else if constexpr (MR) {
        run_filter_mr<T, BIAS, DIRECT, SYNTH, PF, PShared<T, N, BLOCK>, true, STATS>(a, i, P, scr + threadIdx.x, BLOCK, live, vbuf, csm);
    } else {
        run_filter<T, BIAS, DIRECT, SYNTH, PF, PShared<T, N, BLOCK>, true, STATS>(a, i, P, scr + threadIdx.x, BLOCK, live, vbuf, csm);
    }
#else
    if (MR) run_filter_mr<T, BIAS, DIRECT, SYNTH, PF>(a, i, P, scr + threadIdx.x, BLOCK, live, vbuf, csm);
    else run_filter<T, BIAS, DIRECT, SYNTH, PF>(a, i, P, scr + threadIdx.x, BLOCK, live, vbuf, csm);
#endif
}

// ------------------------------------------------------------------------------------------------
// single-step kernels (stateless step functions and the tag callback)
// ------------------------------------------------------------------------------------------------
// "history <- this single entry" for filter i (cpp:326-339): checkpoint = current state, nothing after it
template <typename T, class PS>
QEKF_FN void rebase_history(const DeviceState<T> &st, int64_t i, const Nominal<T> &s, const PS &P)
{
    if (!st.xc) return;
    store_checkpoint<T>(st, i, s, P);
    st.nh[i] = 0;
    st.hlen[i] = 1;
}

// AprilTagSubCallback for filter i with pose8 = (position, orientation xyzw, stamp)  (node.cpp:153-176):
// latch the pose, raise measurement_ready (unless raise_ready = 0: the latch only, what a forced initialize_state
// of the facade needs), initialise on the first detection; force_init: initialize_state from the latched members.
template <typename T, bool BIAS, bool PF, class PS>
QEKF_FN void deliver_one(const DeviceState<T> &st, const Consts<T> &c, const double *pose8, int force_init, int reinit_bias,
                         int raise_ready, PS &P, int64_t i)
{
    int32_t flags = st.flags[i];
    if (!force_init) {
#pragma unroll
        for (int cc = 0; cc < PEND_DIM; ++cc) st.pend[cc * st.ld + i] = pose8[cc];
        if (raise_ready) flags |= FLAG_READY;
    }
    if (force_init || (raise_ready && !(flags & FLAG_INIT))) {
        Nominal<T> s;
        load_filter<T>(st, i, s, P);
        T tag[7];
        // initialize_state reads the latched apriltag_pos/orien members (cpp:310-313)
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) tag[cc] = (T)st.pend[cc * st.ld + i];
        const typename ParSel<T, PF>::type par = ParSel<T, PF>::make(c, st, i);
        initialize_state<T, BIAS>(s, P, tag, par, reinit_bias != 0);
        store_filter<T>(st, i, s, P);
        rebase_history<T>(st, i, s, P);
        flags |= FLAG_INIT;
    }
    st.flags[i] = flags;
}

// AprilTagSubCallback with one pose shared by all filters (node.cpp:153-176)
template <typename T, bool BIAS, bool PF, int BLOCK>
__global__ void __launch_bounds__(BLOCK) deliver_tag_kernel(DeviceState<T> st, Consts<T> c, const double *pose8,
                                                            int force_init, int reinit_bias, int raise_ready)
{
    constexpr int N = BIAS ? 15 : 9;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sm = reinterpret_cast<T *>(smem_raw);
    const int64_t i = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (i >= st.n) return;
    PShared<T, N, BLOCK> P{ sm + threadIdx.x };
    deliver_one<T, BIAS, PF>(st, c, pose8, force_init, reinit_bias, raise_ready, P, i);
}

// One timer tick of the node for a small batch (the N = 1 drop-in): the tag callback (if a detection arrived since
// the last tick), filter_update, and the members the node reads afterwards -- one launch of 32-thread CTAs.  Inputs
// (a.in.imu, pose8) and the output record live in mapped pinned host memory, so a tick costs the host one launch and
// one stream synchronisation.  Record of filter j, TICK_REC doubles at out + j*TICK_REC:
//   x[16] | cov_pert[n*n] row-major | aux[11] | state_initialized measurement_ready performed_correction
//   filter_active upds_since_correction x_hist.size()
constexpr int TICK_REC = 16 + 225 + AUX_DIM + 6;
constexpr int TICK_BLOCK = 32;
template <typename T, bool BIAS, bool DIRECT, bool MR>
__global__ void __launch_bounds__(TICK_BLOCK) tick_kernel(const __grid_constant__ RunArgs<T> a, const double *pose8,
                                                          int tag_mode, double *out, int n_out)
{
    constexpr int N = BIAS ? 15 : 9;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sm = reinterpret_cast<T *>(smem_raw);
    const int64_t i = (int64_t)blockIdx.x * TICK_BLOCK + threadIdx.x;
    const bool live = i < a.st.n;
    PShared<T, N, TICK_BLOCK> P{ sm + threadIdx.x };
    int *vbuf = reinterpret_cast<int *>(sm + (size_t)TICK_BLOCK * (N * (N + 1) / 2));
    if (live && tag_mode != 0) deliver_one<T, BIAS, false>(a.st, a.c, pose8, 0, 0, tag_mode == 1, P, i);
    if (MR) run_filter_mr<T, BIAS, DIRECT, false, false>(a, i, P, vbuf + VOTE_WORDS + threadIdx.x, TICK_BLOCK, live, vbuf);
    else run_filter<T, BIAS, DIRECT, false, false>(a, i, P, vbuf + VOTE_WORDS + threadIdx.x, TICK_BLOCK, live, vbuf);
    // the records of this CTA's filters, written by all 32 lanes together (element e of a record by lane e % 32): the
    // output lives in mapped host memory, and 258 single-lane stores would cross PCIe as 258 transactions
    __syncwarp();
    __threadfence_block();
    const DeviceState<T> &st = a.st;
    const int64_t f0 = (int64_t)blockIdx.x * TICK_BLOCK;
    for (int64_t f = f0; f < f0 + TICK_BLOCK && f < st.n && f < n_out; ++f) {
        double *r = out + f * TICK_REC;
        const int32_t fl = st.flags[f];
        for (int e = threadIdx.x; e < TICK_REC; e += TICK_BLOCK) {
            double v = 0.0;
            if (e < 16) v = (double)st.x[e * st.ld + f];
            else if (e < 16 + 225) {
                const int idx = e - 16, p = idx / N, q2 = idx - p * N;
                if (p < N) v = (double)st.P[sym_idx<N>(p, q2) * st.ld + f];
            } else if (e < 16 + 225 + AUX_DIM) v = (double)st.aux[(e - 16 - 225) * st.ld + f];
            else {
                const int w = e - (16 + 225 + AUX_DIM);
                if (w == 0) v = (fl & FLAG_INIT) ? 1 : 0;
                else if (w == 1) v = (fl & FLAG_READY) ? 1 : 0;
                else if (w == 2) v = (fl & FLAG_CORRECTED) ? 1 : 0;
                else if (w == 3) v = (fl & FLAG_ACTIVE) ? 1 : 0;
                else if (w == 4) v = st.upds[f];
                else v = (fl & FLAG_INIT) ? (st.hlen ? st.hlen[f] : 1) : 0;
            }
            r[e] = v;
        }
    }
}

// prediction_step applied once to every filter with per-filter inputs u [6][ld] (cpp:346-415)
template <typename T, bool BIAS, bool PF, int BLOCK>
__global__ void __launch_bounds__(BLOCK) predict_kernel(DeviceState<T> st, Consts<T> c, const double *u_in)
{
    constexpr int N = BIAS ? 15 : 9;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sm = reinterpret_cast<T *>(smem_raw);
    const int64_t i = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (i >= st.n) return;
    PShared<T, N, BLOCK> P{ sm + threadIdx.x };
    Nominal<T> s;
    load_filter<T>(st, i, s, P);
    T u[6], accel[3];
#pragma unroll
    for (int cc = 0; cc < 6; ++cc) u[cc] = (T)u_in[cc * st.ld + i];
    const typename ParSel<T, PF>::type par = ParSel<T, PF>::make(c, st, i);
    prediction_step<T, BIAS>(s, P, u, par, accel);
    store_filter<T>(st, i, s, P);
    rebase_history<T>(st, i, s, P);
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) st.aux[cc * st.ld + i] = accel[cc];
}

// correction_step applied once to every filter with per-filter tag poses [7][ld] (cpp:417-502)
template <typename T, bool BIAS, bool DIRECT, bool PF, int BLOCK>
__global__ void __launch_bounds__(BLOCK) correct_kernel(DeviceState<T> st, Consts<T> c, const double *tag_in)
{
    constexpr int N = BIAS ? 15 : 9;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sm = reinterpret_cast<T *>(smem_raw);
    const int64_t i = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (i >= st.n) return;
    PShared<T, N, BLOCK> P{ sm + threadIdx.x };
    Nominal<T> s;
    load_filter<T>(st, i, s, P);
    T tag[7];
#pragma unroll
    for (int cc = 0; cc < 7; ++cc) tag[cc] = (T)tag_in[cc * st.ld + i];
    Observation<T> obs;
    const typename ParSel<T, PF>::type par = ParSel<T, PF>::make(c, st, i);
    correction_step<T, BIAS, DIRECT>(s, P, tag, par, obs);
    store_filter<T>(st, i, s, P);
    rebase_history<T>(st, i, s, P);
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) st.aux[(3 + cc) * st.ld + i] = obs.r_t_vt_obs[cc];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) st.aux[(6 + cc) * st.ld + i] = obs.q_tv_obs[cc];
}

// The noise realisation of filters [first, first+count) written out as explicit streams in the C-ABI
// layout (the checker replays exactly these through the oracle): imu [T][6][count], tag [M][7][count],
// valid [M][count], bias [6][count].
template <typename T>
__global__ void synth_dump_kernel(RunArgs<T> a, int64_t first, int64_t count, int64_t T_ticks, double *imu_out,
                                  double *tag_out, uint8_t *valid_out, double *bias_out)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    Inputs<T, true> in;
    in.init(a, first + j);
    for (int c = 0; c < 6; ++c) bias_out[c * count + j] = in.bias[c];
    for (int64_t k = 0; k < T_ticks; ++k) {
        double raw[6], u[6];
        in.raw_imu(k, raw);
        synth_imu(a.ns, in.gid, k, raw, in.bias, u);
        for (int c = 0; c < 6; ++c) imu_out[(k * 6 + c) * count + j] = u[c];
    }
    for (int32_t m = 0; m < a.in.M; ++m) {
        double tg[7];
        in.tag_f64(a.in, a.ns, m, tg);
        for (int c = 0; c < 7; ++c) tag_out[((int64_t)m * 7 + c) * count + j] = tg[c];
        valid_out[(int64_t)m * count + j] = in.valid(a.in, a.ns, m, a.in.tag_step[m]) ? 1 : 0;
    }
}

}  // namespace qekf
