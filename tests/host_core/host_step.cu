// host_step.cu -- TEST HARNESS (not product): the product's per-tick step (deliver_one + step_filter + step_outputs in
// ekf_kernels.cuh, what step_kernel runs per lane) instantiated for the HOST, so that the CPU-only test tier can check
// qekf_step -- the head-keeping delayed-fusion path included -- against the replay and the oracle.  Same state layouts
// as host_truth.cu's hc_run_truth.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../quadrotor_landing_b200/csrc/ekf_kernels.cuh"
#include "../../quadrotor_landing_b200/csrc/ekf_params.hpp"

using namespace qekf;

namespace {

template <typename T, bool BIAS, bool DIRECT>
void step_t(const qekf_params *p, int64_t N, double t_curr, const double *imu, const uint8_t *arrived, const double *tag,
            double *x, double *Ppk, double *aux, double *pend, int32_t *flags, int32_t *upds, double *xc, double *Pc,
            double *ring, int32_t *nh, int32_t *hpos, int32_t *hlen, int32_t ring_len, int32_t dmax,
            const double *const pf_in[5], int64_t *counts, double *x_out, double *cov_out, double *aux_out,
            int32_t *flags_out)
{
    constexpr int NS = BIAS ? 15 : 9;
    constexpr int NP = NS * (NS + 1) / 2;
    std::vector<T> xs(16 * N), Ps((size_t)NP * N), as(AUX_DIM * N);
    for (size_t k = 0; k < xs.size(); ++k) xs[k] = (T)x[k];
    for (size_t k = 0; k < Ps.size(); ++k) Ps[k] = (T)Ppk[k];
    for (size_t k = 0; k < as.size(); ++k) as[k] = (T)aux[k];
    StepArgs<T> a;
    std::memset(&a, 0, sizeof a);
    a.st.x = xs.data(); a.st.P = Ps.data(); a.st.aux = as.data(); a.st.pend = pend;
    a.st.flags = flags; a.st.upds = upds; a.st.counts = nullptr; a.st.ld = N; a.st.n = N;
    a.c = make_consts<T>(*p);
    a.t_curr = t_curr;
    a.imu = imu; a.arrived = arrived; a.tag = tag;
    a.x_out = x_out; a.cov_out = cov_out; a.aux_out = aux_out; a.flags_out = flags_out;
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
        StepOut<T> o;
        // what step_kernel runs for lane i
#define STEP_(MR_, PF_)                                                                                         \
        do {                                                                                                    \
            if (a.arrived && a.arrived[i]) deliver_one<T, BIAS, PF_>(a.st, a.c, a.tag + i, 0, 0, 1, P, i, N);   \
            step_filter<T, BIAS, DIRECT, MR_, PF_>(a.st, a.c, i, a.t_curr, a.imu + i, N, P, o);                 \
        } while (0)
        if (mr && pf) STEP_(true, true);
        else if (mr) STEP_(true, false);
        else if (pf) STEP_(false, true);
        else STEP_(false, false);
#undef STEP_
        step_outputs<T>(a, i, o, P);
        counts[0] += o.n_pred;
        counts[1] += o.n_corr;
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

// Built twice, like host_core.cu: -DHS_ONLY_PREC=64 -> libhost_step64.so, -DHS_ONLY_PREC=32 -> libhost_step32.so.
#ifndef HS_ONLY_PREC
#define HS_ONLY_PREC 64
#endif
#if HS_ONLY_PREC == 64
typedef double hs_real;
#else
typedef float hs_real;
#endif

extern "C" {

// one qekf_step of N filters held in host arrays (host_core.HostBatch layout); counts[2] += (predictions, corrections);
// outputs as qekf_step_io (NULL = not written)
void hc_step(const qekf_params *p, int prec, int64_t N, double t_curr, const double *imu, const uint8_t *arrived,
             const double *tag, double *x, double *Ppk, double *aux, double *pend, int32_t *flags, int32_t *upds, double *xc,
             double *Pc, double *ring, int32_t *nh, int32_t *hpos, int32_t *hlen, int32_t ring_len, int32_t dmax,
             const double *pf_q, const double *pf_r, const double *pf_rvcv, const double *pf_qvc, const double *pf_delay,
             int64_t *counts, double *x_out, double *cov_out, double *aux_out, int32_t *flags_out)
{
    if (prec != HS_ONLY_PREC) std::abort();
    const double *pf[5] = { pf_q, pf_r, pf_rvcv, pf_qvc, pf_delay };
#define C_(B, D) step_t<hs_real, B, D>(p, N, t_curr, imu, arrived, tag, x, Ppk, aux, pend, flags, upds, xc, Pc, ring, nh, hpos, \
                                       hlen, ring_len, dmax, pf, counts, x_out, cov_out, aux_out, flags_out)
    const bool b = p->est_bias != 0, d = p->direct_orien_method != 0;
    if (b && d) C_(true, true);
    else if (b) C_(true, false);
    else if (d) C_(false, true);
    else C_(false, false);
#undef C_
}

}  // extern "C"
