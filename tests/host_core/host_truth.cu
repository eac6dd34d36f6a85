// host_truth.cu -- TEST HARNESS (not product): the product's explicit-stream replay (run_filter / run_filter_mr in
// ekf_kernels.cuh) instantiated for the HOST with the statistics fence compiled in and scored against per-filter
// truth, as qekf_run_with_truth runs it on the device, so that the CPU-only test tier can check the on-chip
// statistics of explicit streams.  Same array layouts as host_core.cu's hc_run_ext.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../quadrotor_landing_b200/csrc/ekf_kernels.cuh"
#include "../../quadrotor_landing_b200/csrc/ekf_params.hpp"

using namespace qekf;

namespace {

template <typename T, bool BIAS, bool DIRECT>
void run_truth_t(const qekf_params *p, int64_t N, int64_t k0, int64_t n_steps, const double *imu, int64_t M,
                 const int32_t *tag_step, const double *tag_pose, const double *tag_stamp, const uint8_t *tag_valid,
                 double t_start, double *x, double *Ppk, double *aux, double *pend, int32_t *flags, int32_t *upds,
                 double *xc, double *Pc, double *ring, int32_t *nh, int32_t *hpos, int32_t *hlen, int32_t ring_len,
                 int32_t dmax, const double *const pf_in[5], const double *truth, double *stats_acc, int32_t n_bins,
                 int32_t stride)
{
    constexpr int NS = BIAS ? 15 : 9;
    constexpr int NP = NS * (NS + 1) / 2;
    std::vector<T> xs(16 * N), Ps((size_t)NP * N), as(AUX_DIM * N);
    for (size_t k = 0; k < xs.size(); ++k) xs[k] = (T)x[k];
    for (size_t k = 0; k < Ps.size(); ++k) Ps[k] = (T)Ppk[k];
    for (size_t k = 0; k < as.size(); ++k) as[k] = (T)aux[k];
    RunArgs<T> a;
    std::memset(&a, 0, sizeof a);
    a.st.x = xs.data(); a.st.P = Ps.data(); a.st.aux = as.data(); a.st.pend = pend;
    a.st.flags = flags; a.st.upds = upds; a.st.counts = nullptr; a.st.ld = N; a.st.n = N;
    a.in.imu = imu; a.in.tag_step = tag_step; a.in.tag_pose = tag_pose; a.in.tag_stamp = tag_stamp;
    a.in.tag_valid = tag_valid; a.in.cs = N; a.in.is = 1; a.in.M = M; a.in.vs = N;
    a.in.t_start = t_start; a.in.update_freq = p->update_freq;
    a.c = make_consts<T>(*p);
    a.k0 = k0; a.n_steps = n_steps;
    int32_t m0 = 0;
    while (m0 < M && tag_step[m0] < k0) ++m0;
    a.m0 = m0;
    // the statistics of qekf_run_with_truth (run_typed in qekf_capi.cu)
    a.stats.acc = stats_acc; a.stats.truth_pf = truth; a.stats.ld_t = N;
    a.stats.n_bins = n_bins; a.stats.stride = stride;
    a.stats.chi2_lo = BIAS ? 6.262137795043251 : 2.7003894999803584;
    a.stats.chi2_hi = BIAS ? 27.488392863442982 : 19.02276779864163;
    const bool mr = p->multirate_ekf != 0;
    const bool pf = pf_in[0] != nullptr;
    std::vector<T> xcs, Pcs, rings, pft;
    std::vector<double> pfd;
    if (mr) {
        xcs.resize(16 * N); Pcs.resize((size_t)NP * N); rings.resize((size_t)ring_len * 6 * N);
        for (size_t k = 0; k < xcs.size(); ++k) xcs[k] = (T)xc[k];
        for (size_t k = 0; k < Pcs.size(); ++k) Pcs[k] = (T)Pc[k];
        for (size_t k = 0; k < rings.size(); ++k) rings[k] = (T)ring[k];
        a.st.xc = xcs.data(); a.st.Pc = Pcs.data(); a.st.ring = rings.data();
        a.st.nh = nh; a.st.hpos = hpos; a.st.hlen = hlen;
        a.st.ring_len = ring_len; a.st.dmax_m1 = dmax - 1;
    }
    if (pf) {
        pft.assign((size_t)PF_DIM * N, T(0));
        pfd.assign(2 * (size_t)N, 0.0);
        qekf_params q = *p;
        for (int64_t i = 0; i < N; ++i) {
            for (int k = 0; k < 3; ++k) {
                q.Q_a[k] = pf_in[0][(0 + k) * N + i]; q.Q_w[k] = pf_in[0][(3 + k) * N + i];
                q.Q_ab[k] = pf_in[0][(6 + k) * N + i]; q.Q_wb[k] = pf_in[0][(9 + k) * N + i];
                q.R_r[k] = pf_in[1][(0 + k) * N + i]; q.R_ang[k] = pf_in[1][(3 + k) * N + i];
                q.r_v_cv[k] = pf_in[2][k * N + i];
            }
            for (int k = 0; k < 4; ++k) q.q_vc[k] = pf_in[3][k * N + i];
            fill_pf_column<T>(q, pft.data() + i, N);
            pfd[i] = pf_in[4][i]; pfd[N + i] = pf_in[4][N + i];
        }
        a.st.pf = pft.data(); a.st.pf_delay = pfd.data();
    }
    for (int64_t i = 0; i < N; ++i) {
        PLocal<T, NS> P;
        int32_t ints[MR_SCRATCH_INTS > SR_SCRATCH_INTS ? MR_SCRATCH_INTS : SR_SCRATCH_INTS];
#define RUN_(F)                                                                                              \
        do {                                                                                                 \
            if (mr) run_filter_mr<T, BIAS, DIRECT, false, F, PLocal<T, NS>, false, true>(a, i, P, ints, 1); \
            else run_filter<T, BIAS, DIRECT, false, F, PLocal<T, NS>, false, true>(a, i, P, ints, 1);       \
        } while (0)
        if (pf) RUN_(true);
        else RUN_(false);
#undef RUN_
    }
    for (size_t k = 0; k < xs.size(); ++k) x[k] = xs[k];
    for (size_t k = 0; k < Ps.size(); ++k) Ppk[k] = Ps[k];
    for (size_t k = 0; k < as.size(); ++k) aux[k] = as[k];
    if (mr) {
        for (size_t k = 0; k < xcs.size(); ++k) xc[k] = xcs[k];
        for (size_t k = 0; k < Pcs.size(); ++k) Pc[k] = Pcs[k];
        for (size_t k = 0; k < rings.size(); ++k) ring[k] = rings[k];
    }
}

}  // namespace

// Built twice, like host_core.cu: -DHT_ONLY_PREC=64 -> libhost_truth64.so, -DHT_ONLY_PREC=32 -> libhost_truth32.so.
#ifndef HT_ONLY_PREC
#define HT_ONLY_PREC 64
#endif
#if HT_ONLY_PREC == 64
typedef double ht_real;
#else
typedef float ht_real;
#endif

extern "C" {

// hc_run_ext of host_core.cu, scored against per-filter truth (qekf_run_with_truth): truth [n_bins][16][N] (r v q_tv
// ab wb after the sampling tick of each bin), stats_acc [STAT_REPL][n_bins][STAT_DIM]
void hc_run_truth(const qekf_params *p, int prec, int64_t N, int64_t k0, int64_t n_steps, const double *imu, int64_t M,
                  const int32_t *tag_step, const double *tag_pose, const double *tag_stamp, const uint8_t *tag_valid,
                  double t_start, double *x, double *Ppk, double *aux, double *pend, int32_t *flags, int32_t *upds,
                  double *xc, double *Pc, double *ring, int32_t *nh, int32_t *hpos, int32_t *hlen, int32_t ring_len,
                  int32_t dmax, const double *pf_q, const double *pf_r, const double *pf_rvcv, const double *pf_qvc,
                  const double *pf_delay, const double *truth, double *stats_acc, int32_t n_bins, int32_t stride)
{
    if (prec != HT_ONLY_PREC) std::abort();
    const double *pf[5] = { pf_q, pf_r, pf_rvcv, pf_qvc, pf_delay };
#define C_(B, D) run_truth_t<ht_real, B, D>(p, N, k0, n_steps, imu, M, tag_step, tag_pose, tag_stamp, tag_valid, t_start, x, \
                                            Ppk, aux, pend, flags, upds, xc, Pc, ring, nh, hpos, hlen, ring_len, dmax, pf,  \
                                            truth, stats_acc, n_bins, stride)
    const bool b = p->est_bias != 0, d = p->direct_orien_method != 0;
    if (b && d) C_(true, true);
    else if (b) C_(true, false);
    else if (d) C_(false, true);
    else C_(false, false);
#undef C_
}

}  // extern "C"
