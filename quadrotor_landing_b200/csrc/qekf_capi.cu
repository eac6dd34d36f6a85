// qekf_capi.cu -- host side of libqekf: handle, parameter derivation, launches, and the C ABI declared
// in include/qekf.h.  Host code is C++ over the CUDA runtime; nothing here falls back to the CPU.
#include "../../include/qekf.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "ekf_params.hpp"
#include "launch.hpp"
#include "launch_coop.hpp"
#include "preset.hpp"
#include "scenario.hpp"

using namespace qekf;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return fail(QEKF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));        \
    } while (0)

}  // namespace

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
struct qekf_handle {
    qekf_params p;
    int precision = QEKF_FP64;
    int device = 0;
    int64_t n = 0, ld = 0;
    int nstates = 15, np = 120;
    size_t tsize = 8;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    void *x = nullptr, *P = nullptr, *aux = nullptr;
    double *pend = nullptr;
    int32_t *flags = nullptr, *upds = nullptr;
    unsigned long long *counts = nullptr;
    // delayed-measurement fusion (multirate_ekf): lagged checkpoint + IMU ring, see ekf_kernels.cuh
    void *xc = nullptr, *Pc = nullptr, *ring = nullptr;
    int32_t *nh = nullptr, *hpos = nullptr, *hlen = nullptr;
    int ring_len = 0, dmax = 1;
    // per-filter parameter overrides: host copies [dim][N] per field, derived device tables
    std::vector<double> pf_host[5];
    bool pf_overridden[5] = { false, false, false, false, false };   // which fields the caller has set (the others follow p)
    bool pf_on = false;
    void *pf = nullptr;
    double *pf_delay = nullptr;
    // per-tick interface staging
    double *d_tick = nullptr;        // [6 imu][8 tag]
    double *h_tick = nullptr;        // pinned mirror
    // fused per-tick path (qekf_tick): inputs [6 imu][8 tag] and the output records in MAPPED pinned memory
    double *tick_in = nullptr, *tick_in_dev = nullptr;
    double *tick_out = nullptr, *tick_out_dev = nullptr;
    int tick_out_cap = 0;
    int32_t *d_no_steps = nullptr;
    double imu_latched[6] = { 0, 0, 0, 0, 0, 0 };
    // cached device copies of host streams (qekf_run with on_device = 0)
    void *d_in = nullptr;
    size_t d_in_bytes = 0;
    // Monte-Carlo statistics (device): acc [STAT_REPL][n_bins][STAT_DIM], reduced [n_bins][STAT_DIM]
    double *stats_acc = nullptr, *stats_red = nullptr;
    int32_t stats_bins = 0, stats_stride = 0;
    // cached device copy of the shared clean scenario (qekf_run_monte_carlo with host pointers)
    void *d_shared = nullptr;
    size_t d_shared_bytes = 0;
    uint8_t *d_mask = nullptr;       // detection front-end visibility mask [M]
    size_t d_mask_bytes = 0;
    // slot -> filter order of the Monte-Carlo replay (filters sorted by the start of their private dropout), and the
    // noise-spec fields it was derived from
    int32_t *d_perm = nullptr;
    void *perm_scratch = nullptr;    // staging buffer of the reordering passes (as large as the largest per-filter array)
    size_t perm_scratch_bytes = 0;
    bool in_slot_order = false;      // the per-filter arrays are currently reordered (only ever true inside qekf_run_monte_carlo)
    uint64_t perm_seed = 0;
    int64_t perm_gid0 = 0;
    int32_t perm_len = 0, perm_lo = 0, perm_hi = 0;
    bool perm_on = true;             // QEKF_NO_PERM=1 disables it (A/B runs)
    int64_t perm_min_steps = 256;    // shortest replay that is reordered (QEKF_PERM_MIN_STEPS overrides)
    // Delayed fusion: may a Monte-Carlo launch re-synthesise the IMU inputs of the history entries it finds instead of
    // reading the ring?  Yes if no filter has an entry after its checkpoint (hist_clean: fresh, reset or rebased handle),
    // or if they were all produced by Monte-Carlo launches of the same noise model and scenario ending where this one
    // starts (hist_key).  Any other entry point that touches the histories clears both.
    bool hist_clean = true, hist_key_valid = false, lazy_mr_on = true, lazy_now = false;     // QEKF_NO_LAZY_MR=1 disables the path (A/B runs)
    uint64_t hist_key[6] = { 0, 0, 0, 0, 0, 0 };
    int64_t hist_k_next = 0;
    // launch bookkeeping
    int64_t launches = 0;
    // mapping of the fused replay (qekf_set_mapping), where the kernels exist (FP64, single-rate): 2 = two role-specialised
    // warps per 32 filters (ekf_duo.cuh), 3 = three lanes per filter (ekf_coop.cuh), 1 = one thread per filter
    int lanes_per_filter = 1;
    int coop_groups = COOP_GROUPS_DEFAULT, duo_groups = DUO_GROUPS_DEFAULT;
    // CTA size of the per-tick step kernel (qekf_step, launch.hpp); QEKF_STEP_BLOCK overrides it (A/B runs)
    int step_block = 32;
};

namespace {

template <typename T> DeviceState<T> dstate(const qekf_handle *h)
{
    DeviceState<T> s;
    s.x = (T *)h->x; s.P = (T *)h->P; s.aux = (T *)h->aux; s.pend = h->pend;
    s.flags = h->flags; s.upds = h->upds; s.counts = h->counts; s.ld = h->ld; s.n = h->n;
    s.xc = (T *)h->xc; s.Pc = (T *)h->Pc; s.ring = (T *)h->ring;
    s.nh = h->nh; s.hpos = h->hpos; s.hlen = h->hlen;
    s.ring_len = h->ring_len; s.dmax_m1 = h->dmax - 1;
    s.pf = h->pf_on ? (const T *)h->pf : nullptr;
    s.pf_delay = h->pf_on ? h->pf_delay : nullptr;
    s.perm = nullptr;
    s.gid_perm = nullptr;
    s.hist_synth = 0;
    return s;
}

// the delayed-fusion histories are about to be touched by something other than a Monte-Carlo launch
void hist_touch(qekf_handle *h) { h->hist_clean = false; h->hist_key_valid = false; }
void hist_emptied(qekf_handle *h) { h->hist_clean = true; h->hist_key_valid = false; }

uint64_t fnv1a(const void *data, size_t bytes, uint64_t hsh = 1469598103934665603ULL)
{
    const unsigned char *p = static_cast<const unsigned char *>(data);
    for (size_t i = 0; i < bytes; ++i) { hsh ^= p[i]; hsh *= 1099511628211ULL; }
    return hsh;
}

int block_of(const qekf_handle *h) { return h->precision == QEKF_FP64 ? BlockOf<double>::value : BlockOf<float>::value; }
size_t smem_bytes(const qekf_handle *h)
{
#ifdef QEKF_EXP8
    size_t b = (size_t)block_of(h) * ((h->precision == QEKF_FP64 && h->np == 120) ? 105 : h->np) * h->tsize + VOTE_WORDS * sizeof(int);
#else
    size_t b = (size_t)block_of(h) * h->np * h->tsize + VOTE_WORDS * sizeof(int);
#endif
    b += (size_t)block_of(h) * (h->p.multirate_ekf ? MR_SCRATCH_INTS : SR_SCRATCH_INTS) * sizeof(int32_t);
#ifndef QEKF_EXP8
    b += consts_smem_bytes(h->precision == QEKF_FP64 ? sizeof(Consts<double>) : sizeof(Consts<float>));
#endif
    return b;
}
unsigned grid_of(const qekf_handle *h) { return (unsigned)((h->n + block_of(h) - 1) / block_of(h)); }

// dispatch over the code-shape flags (est_bias, direct_orien_method) and the precision
#define QEKF_DISPATCH(h, CALL)                                                             \
    do {                                                                                   \
        const bool b__ = (h)->p.est_bias != 0, d__ = (h)->p.direct_orien_method != 0;      \
        if ((h)->precision == QEKF_FP64) {                                                 \
            if (b__ && d__) { CALL(double, true, true); }                                  \
            else if (b__) { CALL(double, true, false); }                                   \
            else if (d__) { CALL(double, false, true); }                                   \
            else { CALL(double, false, false); }                                           \
        } else {                                                                           \
            if (b__ && d__) { CALL(float, true, true); }                                   \
            else if (b__) { CALL(float, true, false); }                                    \
            else if (d__) { CALL(float, false, true); }                                    \
            else { CALL(float, false, false); }                                            \
        }                                                                                  \
    } while (0)

int free_state(qekf_handle *h)
{
    cudaFree(h->x); cudaFree(h->P); cudaFree(h->aux); cudaFree(h->pend);
    cudaFree(h->flags); cudaFree(h->upds); cudaFree(h->d_tick); cudaFree(h->d_in);
    cudaFree(h->stats_acc); cudaFree(h->stats_red); cudaFree(h->d_shared); cudaFree(h->counts);
    cudaFree(h->xc); cudaFree(h->Pc); cudaFree(h->ring); cudaFree(h->nh); cudaFree(h->hpos); cudaFree(h->hlen);
    cudaFree(h->pf); cudaFree(h->pf_delay); cudaFree(h->d_mask); cudaFree(h->d_perm); cudaFree(h->perm_scratch);
    h->d_perm = nullptr; h->perm_len = 0; h->perm_scratch = nullptr; h->perm_scratch_bytes = 0; h->in_slot_order = false;
    h->d_mask = nullptr; h->d_mask_bytes = 0;
    h->xc = h->Pc = h->ring = nullptr; h->nh = h->hpos = h->hlen = nullptr; h->ring_len = 0;
    h->pf = nullptr; h->pf_delay = nullptr; h->pf_on = false;
    for (auto &v : h->pf_host) v.clear();
    h->counts = nullptr;
    h->stats_acc = h->stats_red = nullptr; h->stats_bins = 0; h->d_shared = nullptr; h->d_shared_bytes = 0;
    if (h->h_tick) cudaFreeHost(h->h_tick);
    if (h->tick_in) cudaFreeHost(h->tick_in);
    if (h->tick_out) cudaFreeHost(h->tick_out);
    h->tick_in = h->tick_in_dev = h->tick_out = h->tick_out_dev = nullptr; h->tick_out_cap = 0;
    h->x = h->P = h->aux = nullptr; h->pend = nullptr; h->flags = h->upds = nullptr;
    h->d_tick = nullptr; h->h_tick = nullptr; h->d_in = nullptr; h->d_in_bytes = 0;
    return QEKF_OK;
}

// largest step delay a correction of this handle can use (cpp:199-200)
int max_step_delay(const qekf_handle *h)
{
    if (h->p.dynamic_meas_delay) return step_of_delay(h->p.measurement_delay_max, h->p.update_freq);
    int d = step_of_delay(h->p.measurement_delay, h->p.update_freq);
    const std::vector<double> &v = h->pf_host[QEKF_PF_DELAY];
    for (int64_t i = 0; i < (int64_t)v.size() / 2; ++i) {
        const int di = step_of_delay(v[(size_t)i], h->p.update_freq);
        if (di > d) d = di;
    }
    return d;
}

// (re)allocate the delayed-fusion storage for the current parameters; histories restart from the heads
int alloc_history(qekf_handle *h)
{
    if (!h->p.multirate_ekf) return QEKF_OK;
    const size_t ld = (size_t)h->ld;
    const int dmax = max_step_delay(h);
    const int L = ring_length(dmax, h->p);
    if (!h->xc) {
        CUDA_TRY(cudaMalloc(&h->xc, 16 * ld * h->tsize));
        CUDA_TRY(cudaMalloc(&h->Pc, (size_t)h->np * ld * h->tsize));
        CUDA_TRY(cudaMalloc(&h->nh, ld * sizeof(int32_t)));
        CUDA_TRY(cudaMalloc(&h->hpos, ld * sizeof(int32_t)));
        CUDA_TRY(cudaMalloc(&h->hlen, ld * sizeof(int32_t)));
        CUDA_TRY(cudaMemsetAsync(h->xc, 0, 16 * ld * h->tsize, h->stream));
        CUDA_TRY(cudaMemsetAsync(h->Pc, 0, (size_t)h->np * ld * h->tsize, h->stream));
        CUDA_TRY(cudaMemsetAsync(h->nh, 0, ld * sizeof(int32_t), h->stream));
        CUDA_TRY(cudaMemsetAsync(h->hpos, 0, ld * sizeof(int32_t), h->stream));
        CUDA_TRY(cudaMemsetAsync(h->hlen, 0, ld * sizeof(int32_t), h->stream));
    }
    if (L != h->ring_len) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        cudaFree(h->ring);
        h->ring = nullptr; h->ring_len = 0;
        CUDA_TRY(cudaMalloc(&h->ring, (size_t)L * 6 * ld * h->tsize));
        CUDA_TRY(cudaMemsetAsync(h->ring, 0, (size_t)L * 6 * ld * h->tsize, h->stream));
        h->ring_len = L;
    }
    h->dmax = dmax;
    return QEKF_OK;
}

// history <- the current head, for every filter (a ring that changed size, or parameters that changed)
int rebase_all(qekf_handle *h)
{
    if (!h->p.multirate_ekf || !h->xc) return QEKF_OK;
    if (h->precision == QEKF_FP64) CUDA_TRY(launch_rebase<double>(dstate<double>(h), h->np, h->stream));
    else CUDA_TRY(launch_rebase<float>(dstate<float>(h), h->np, h->stream));
    hist_emptied(h);
    return QEKF_OK;
}

int alloc_state(qekf_handle *h)
{
    h->nstates = h->p.est_bias ? 15 : 9;
    h->np = h->nstates * (h->nstates + 1) / 2;
    h->tsize = (h->precision == QEKF_FP64) ? 8 : 4;
    const size_t ld = (size_t)h->ld;
    CUDA_TRY(cudaMalloc(&h->x, 16 * ld * h->tsize));
    CUDA_TRY(cudaMalloc(&h->P, (size_t)h->np * ld * h->tsize));
    CUDA_TRY(cudaMalloc(&h->aux, AUX_DIM * ld * h->tsize));
    CUDA_TRY(cudaMalloc(&h->pend, PEND_DIM * ld * sizeof(double)));
    CUDA_TRY(cudaMalloc(&h->flags, ld * sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(&h->upds, ld * sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(&h->counts, 8 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemsetAsync(h->counts, 0, 8 * sizeof(unsigned long long), h->stream));
    CUDA_TRY(cudaMalloc(&h->d_tick, 16 * sizeof(double)));
    CUDA_TRY(cudaMallocHost(&h->h_tick, 16 * sizeof(double)));
    CUDA_TRY(cudaMemsetAsync(h->x, 0, 16 * ld * h->tsize, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->P, 0, (size_t)h->np * ld * h->tsize, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->aux, 0, AUX_DIM * ld * h->tsize, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->pend, 0, PEND_DIM * ld * sizeof(double), h->stream));
    CUDA_TRY(cudaMemsetAsync(h->flags, 0, ld * sizeof(int32_t), h->stream));
    CUDA_TRY(cudaMemsetAsync(h->upds, 0, ld * sizeof(int32_t), h->stream));
    return alloc_history(h);
}

int reset_cov(qekf_handle *h, bool reset_nominal)
{
    if (h->precision == QEKF_FP64)
        CUDA_TRY(launch_reset<double>(dstate<double>(h), make_consts<double>(h->p), h->nstates, reset_nominal, h->stream));
    else
        CUDA_TRY(launch_reset<float>(dstate<float>(h), make_consts<float>(h->p), h->nstates, reset_nominal, h->stream));
    return QEKF_OK;
}

int check_params(const qekf_params *p)
{
    if (!p) return fail(QEKF_ERR_BAD_ARG, "params is NULL");
    if (!(p->update_freq > 0) || !(p->measurement_freq > 0)) return fail(QEKF_ERR_BAD_ARG, "rates must be positive");
    if (p->n_tags < 0 || p->n_tags > QEKF_MAX_TAGS) return fail(QEKF_ERR_BAD_ARG, "n_tags out of range");
    if (p->multirate_ekf) {
        if (!(p->measurement_delay_max >= 0) || !(p->measurement_delay >= 0))
            return fail(QEKF_ERR_BAD_ARG, "measurement delays must be non-negative");
        if (step_of_delay(p->dynamic_meas_delay ? p->measurement_delay_max : p->measurement_delay, p->update_freq) > 4096)
            return fail(QEKF_ERR_BAD_ARG, "measurement delay spans more than 4096 ticks");
    }
    return QEKF_OK;
}

template <typename T, bool BIAS, bool DIRECT>
int run_typed(qekf_handle *h, const StreamView &in, int64_t k0, int64_t n_steps, int32_t m0, const NoiseSpec *ns,
              const double *truth)
{
    RunArgs<T> a;
    std::memset(&a, 0, sizeof a);
    a.st = dstate<T>(h);
    a.in = in;
    a.c = make_consts<T>(h->p);
    a.k0 = k0; a.n_steps = n_steps; a.m0 = m0;
    if (ns) {
        a.ns = *ns;
        // a reordered launch (qekf_run_monte_carlo has gathered the per-filter arrays into slot order): row j of every
        // array belongs to filter d_perm[j], which is what keys its noise
        a.st.gid_perm = h->in_slot_order ? h->d_perm : nullptr;
        a.st.hist_synth = h->lazy_now ? 1 : 0;
    }
    // truth: the shared scenario truth [T+1][10] of a Monte-Carlo launch, or the per-filter truth of an explicit-stream
    // launch (qekf_run_with_truth: [bin][16][N], based so that absolute bin indices work)
    if (h->stats_acc && truth && h->stats_stride > 0) {
        a.stats.acc = h->stats_acc;
        if (ns) a.stats.truth = truth;
        else { a.stats.truth_pf = truth; a.stats.ld_t = h->n; }
        a.stats.n_bins = h->stats_bins; a.stats.stride = h->stats_stride;
        // two-sided 95% chi-square interval for n degrees of freedom
        a.stats.chi2_lo = BIAS ? 6.262137795043251 : 2.7003894999803584;
        a.stats.chi2_hi = BIAS ? 27.488392863442982 : 19.02276779864163;
    }
    const bool mr = h->p.multirate_ekf != 0, pf = h->pf_on;
    // explicit streams scored against per-filter truth run one thread per filter whatever the mapping says (the
    // cooperative kernels accumulate statistics for Monte-Carlo launches only)
    const bool coop_ok = ns != nullptr || a.stats.acc == nullptr;
    if constexpr (std::is_same<T, double>::value) {
        if (!mr && h->lanes_per_filter == 2 && coop_ok) {
            // two role-specialised warps per 32 filters (ekf_duo.cuh)
            cudaError_t e;
            if (ns) e = pf ? launch_run_duo<BIAS, DIRECT, true, true>(a, h->duo_groups, h->stream)
                           : launch_run_duo<BIAS, DIRECT, true, false>(a, h->duo_groups, h->stream);
            else e = pf ? launch_run_duo<BIAS, DIRECT, false, true>(a, h->duo_groups, h->stream)
                        : launch_run_duo<BIAS, DIRECT, false, false>(a, h->duo_groups, h->stream);
            if (e != cudaSuccess) return fail(QEKF_ERR_CUDA, std::string("two-role replay launch: ") + cudaGetErrorString(e));
            h->launches++;
            return QEKF_OK;
        }
        if (!mr && h->lanes_per_filter == 3 && coop_ok) {
            // three lanes per filter (ekf_coop.cuh)
            cudaError_t e;
            if (ns) e = pf ? launch_run_coop<BIAS, DIRECT, true, true>(a, h->coop_groups, h->stream)
                           : launch_run_coop<BIAS, DIRECT, true, false>(a, h->coop_groups, h->stream);
            else e = pf ? launch_run_coop<BIAS, DIRECT, false, true>(a, h->coop_groups, h->stream)
                        : launch_run_coop<BIAS, DIRECT, false, false>(a, h->coop_groups, h->stream);
            if (e != cudaSuccess) return fail(QEKF_ERR_CUDA, std::string("cooperative replay launch: ") + cudaGetErrorString(e));
            h->launches++;
            return QEKF_OK;
        }
    }
#define LAUNCH_(S, MR_, PF_, ST) CUDA_TRY((launch_run<T, BIAS, DIRECT, S, MR_, PF_, ST>(a, grid_of(h), smem_bytes(h), h->stream)))
#define LAUNCH_S(S, ST)                                                   \
    do {                                                                  \
        if (mr && pf) LAUNCH_(S, true, true, ST);                         \
        else if (mr) LAUNCH_(S, true, false, ST);                         \
        else if (pf) LAUNCH_(S, false, true, ST);                         \
        else LAUNCH_(S, false, false, ST);                                \
    } while (0)
    if (ns) LAUNCH_S(true, true);
    else if (a.stats.acc) LAUNCH_S(false, true);     // explicit streams scored against per-filter truth
    else LAUNCH_S(false, false);
#undef LAUNCH_S
#undef LAUNCH_
    h->launches++;
    return QEKF_OK;
}

int run_dispatch(qekf_handle *h, const StreamView &in, int64_t k0, int64_t n_steps, int32_t m0,
                 const NoiseSpec *ns = nullptr, const double *truth = nullptr)
{
#define CALL_RUN(T, B, D) return run_typed<T, B, D>(h, in, k0, n_steps, m0, ns, truth)
    QEKF_DISPATCH(h, CALL_RUN);
#undef CALL_RUN
    return QEKF_OK;
}

// copy a [rows][count] slab out of a [rows][ld] device array of element size tsize into doubles
int fetch_rows(qekf_handle *h, const void *dev, int rows, int64_t first, int64_t count, double *out)
{
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->precision == QEKF_FP64) {
        CUDA_TRY(cudaMemcpy2D(out, (size_t)count * 8, (const char *)dev + (size_t)first * 8, (size_t)h->ld * 8,
                              (size_t)count * 8, (size_t)rows, cudaMemcpyDeviceToHost));
    } else {
        std::vector<float> tmp((size_t)rows * (size_t)count);
        CUDA_TRY(cudaMemcpy2D(tmp.data(), (size_t)count * 4, (const char *)dev + (size_t)first * 4, (size_t)h->ld * 4,
                              (size_t)count * 4, (size_t)rows, cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < tmp.size(); ++k) out[k] = (double)tmp[k];
    }
    return QEKF_OK;
}

int store_rows(qekf_handle *h, void *dev, int rows, int64_t first, int64_t count, const double *in)
{
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->precision == QEKF_FP64) {
        CUDA_TRY(cudaMemcpy2D((char *)dev + (size_t)first * 8, (size_t)h->ld * 8, in, (size_t)count * 8,
                              (size_t)count * 8, (size_t)rows, cudaMemcpyHostToDevice));
    } else {
        std::vector<float> tmp((size_t)rows * (size_t)count);
        for (size_t k = 0; k < tmp.size(); ++k) tmp[k] = (float)in[k];
        CUDA_TRY(cudaMemcpy2D((char *)dev + (size_t)first * 4, (size_t)h->ld * 4, tmp.data(), (size_t)count * 4,
                              (size_t)count * 4, (size_t)rows, cudaMemcpyHostToDevice));
    }
    return QEKF_OK;
}

bool range_ok(const qekf_handle *h, int64_t first, int64_t count)
{
    return h && first >= 0 && count >= 0 && first + count <= h->n;
}

// Slot order of the Monte-Carlo replay: filters sorted (counting sort, stable) by the first tick of their private
// dropout window, a pure function of (seed, global id).  Rebuilt only when the fields it depends on change.
int ensure_perm(qekf_handle *h, const NoiseSpec &ns)
{
    const bool wanted = h->perm_on && ns.rdrop_len > 0 && ns.rdrop_hi > ns.rdrop_lo && h->n > 1;
    if (!wanted) {
        if (h->d_perm) { CUDA_TRY(cudaStreamSynchronize(h->stream)); cudaFree(h->d_perm); h->d_perm = nullptr; h->perm_len = 0; }
        return QEKF_OK;
    }
    if (h->d_perm && h->perm_seed == ns.seed && h->perm_gid0 == ns.gid0 && h->perm_len == ns.rdrop_len &&
        h->perm_lo == ns.rdrop_lo && h->perm_hi == ns.rdrop_hi)
        return QEKF_OK;
    const int64_t n = h->n;
    const int32_t span = ns.rdrop_hi - ns.rdrop_lo;
    std::vector<int32_t> start((size_t)n), perm((size_t)n);
    std::vector<int64_t> head((size_t)span + 1, 0);
    for (int64_t i = 0; i < n; ++i) {
        start[(size_t)i] = private_dropout_start(ns, ns.gid0 + i) - ns.rdrop_lo;
        head[(size_t)start[(size_t)i] + 1]++;
    }
    for (int32_t b = 0; b < span; ++b) head[(size_t)b + 1] += head[(size_t)b];
    for (int64_t i = 0; i < n; ++i) perm[(size_t)head[(size_t)start[(size_t)i]]++] = (int32_t)i;
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (!h->d_perm) CUDA_TRY(cudaMalloc(&h->d_perm, (size_t)n * sizeof(int32_t)));
    CUDA_TRY(cudaMemcpy(h->d_perm, perm.data(), (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice));
    h->perm_seed = ns.seed; h->perm_gid0 = ns.gid0; h->perm_len = ns.rdrop_len; h->perm_lo = ns.rdrop_lo; h->perm_hi = ns.rdrop_hi;
    return QEKF_OK;
}
// Reorder every per-filter array of the handle between filter order (row i = filter i: what every accessor and every
// other entry point assumes) and slot order (row j = filter d_perm[j]: what a reordered Monte-Carlo launch works on).
// Each array is gathered into the staging buffer and copied back: two streaming passes over the state per direction
// (~3 ms per million delayed-fusion filters), against seconds of replay.
int permute_state(qekf_handle *h, bool to_slots)
{
    if (h->in_slot_order == to_slots || !h->d_perm) return QEKF_OK;
    struct Arr { void *p; int64_t rows; size_t word; };
    const int64_t ld = h->ld;
    std::vector<Arr> arrs = { { h->x, 16, h->tsize }, { h->P, h->np, h->tsize }, { h->aux, AUX_DIM, h->tsize },
                              { h->pend, PEND_DIM, 8 }, { h->flags, 1, 4 }, { h->upds, 1, 4 } };
    if (h->xc) {
        arrs.push_back({ h->xc, 16, h->tsize });
        arrs.push_back({ h->Pc, h->np, h->tsize });
        arrs.push_back({ h->ring, (int64_t)h->ring_len * 6, h->tsize });
        arrs.push_back({ h->nh, 1, 4 });
        arrs.push_back({ h->hpos, 1, 4 });
        arrs.push_back({ h->hlen, 1, 4 });
    }
    if (h->pf_on) {
        arrs.push_back({ h->pf, PF_DIM, h->tsize });
        arrs.push_back({ h->pf_delay, 2, 8 });
    }
    size_t need = 0;
    for (const Arr &a : arrs) need = std::max(need, (size_t)a.rows * (size_t)ld * a.word);
    if (need > h->perm_scratch_bytes) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        cudaFree(h->perm_scratch);
        h->perm_scratch = nullptr; h->perm_scratch_bytes = 0;
        CUDA_TRY(cudaMalloc(&h->perm_scratch, need));
        h->perm_scratch_bytes = need;
    }
    for (const Arr &a : arrs) {
        if (a.word == 8)
            CUDA_TRY(launch_permute_rows<uint64_t>((uint64_t *)h->perm_scratch, (const uint64_t *)a.p, h->d_perm, a.rows, ld, h->n, to_slots, h->stream));
        else
            CUDA_TRY(launch_permute_rows<uint32_t>((uint32_t *)h->perm_scratch, (const uint32_t *)a.p, h->d_perm, a.rows, ld, h->n, to_slots, h->stream));
        CUDA_TRY(cudaMemcpyAsync(a.p, h->perm_scratch, (size_t)a.rows * (size_t)ld * a.word, cudaMemcpyDeviceToDevice, h->stream));
        h->launches++;
    }
    h->in_slot_order = to_slots;
    return QEKF_OK;
}

int ensure_in(qekf_handle *h, size_t bytes)
{
    if (bytes <= h->d_in_bytes) return QEKF_OK;
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->d_in);
    h->d_in = nullptr; h->d_in_bytes = 0;
    CUDA_TRY(cudaMalloc(&h->d_in, bytes));
    h->d_in_bytes = bytes;
    return QEKF_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// derive the device tables of the per-filter overrides: initialize_params (cpp:87-125) once per filter
template <typename T> int rebuild_pf_t(qekf_handle *h)
{
    const size_t N = (size_t)h->n, ld = (size_t)h->ld;
    std::vector<T> tab((size_t)PF_DIM * ld, T(0));
    std::vector<double> dl(2 * ld, 0.0);
    qekf_params p = h->p;
    for (size_t i = 0; i < N; ++i) {
        for (int k = 0; k < 3; ++k) {
            p.Q_a[k] = h->pf_host[QEKF_PF_Q][(0 + k) * N + i]; p.Q_w[k] = h->pf_host[QEKF_PF_Q][(3 + k) * N + i];
            p.Q_ab[k] = h->pf_host[QEKF_PF_Q][(6 + k) * N + i]; p.Q_wb[k] = h->pf_host[QEKF_PF_Q][(9 + k) * N + i];
            p.R_r[k] = h->pf_host[QEKF_PF_R][(0 + k) * N + i]; p.R_ang[k] = h->pf_host[QEKF_PF_R][(3 + k) * N + i];
            p.r_v_cv[k] = h->pf_host[QEKF_PF_R_V_CV][k * N + i];
        }
        for (int k = 0; k < 4; ++k) p.q_vc[k] = h->pf_host[QEKF_PF_Q_VC][k * N + i];
        fill_pf_column<T>(p, tab.data() + i, (int64_t)ld);
        dl[i] = h->pf_host[QEKF_PF_DELAY][0 * N + i];
        dl[ld + i] = h->pf_host[QEKF_PF_DELAY][1 * N + i];
    }
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    CUDA_TRY(cudaMemcpy(h->pf, tab.data(), tab.size() * sizeof(T), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->pf_delay, dl.data(), dl.size() * sizeof(double), cudaMemcpyHostToDevice));
    return QEKF_OK;
}
int rebuild_pf(qekf_handle *h)
{
    return h->precision == QEKF_FP64 ? rebuild_pf_t<double>(h) : rebuild_pf_t<float>(h);
}

// (re)seed the host copy of per-filter field `f` from the handle-wide parameters
void seed_pf_field(qekf_handle *h, int f)
{
    static const int dims[5] = { 12, 6, 3, 4, 2 };
    const size_t N = (size_t)h->n;
    const qekf_params &p = h->p;
    std::vector<double> &v = h->pf_host[f];
    v.assign((size_t)dims[f] * N, 0.0);
    for (size_t i = 0; i < N; ++i) {
        if (f == QEKF_PF_Q) {
            for (int k = 0; k < 3; ++k) {
                v[(0 + k) * N + i] = p.Q_a[k]; v[(3 + k) * N + i] = p.Q_w[k];
                v[(6 + k) * N + i] = p.Q_ab[k]; v[(9 + k) * N + i] = p.Q_wb[k];
            }
        } else if (f == QEKF_PF_R) {
            for (int k = 0; k < 3; ++k) { v[(0 + k) * N + i] = p.R_r[k]; v[(3 + k) * N + i] = p.R_ang[k]; }
        } else if (f == QEKF_PF_R_V_CV) {
            for (int k = 0; k < 3; ++k) v[k * N + i] = p.r_v_cv[k];
        } else if (f == QEKF_PF_Q_VC) {
            for (int k = 0; k < 4; ++k) v[k * N + i] = p.q_vc[k];
        } else {
            v[0 * N + i] = p.measurement_delay;
            v[1 * N + i] = p.dyn_measurement_delay_offset;
        }
    }
}

template <typename T, bool BIAS, bool DIRECT>
int tick_typed(qekf_handle *h, int tag_mode, double t_curr, int n_out)
{
    RunArgs<T> a;
    std::memset(&a, 0, sizeof a);
    a.st = dstate<T>(h);
    a.in.imu = h->tick_in_dev; a.in.cs = 1; a.in.is = 0; a.in.M = 0;
    a.in.tag_pose = h->tick_in_dev + 6;
    a.in.t_start = t_curr; a.in.update_freq = h->p.update_freq;
    a.c = make_consts<T>(h->p);
    a.k0 = 0; a.n_steps = 1; a.m0 = 0;
    if (h->p.multirate_ekf) CUDA_TRY((launch_tick<T, BIAS, DIRECT, true>(a, h->tick_in_dev + 6, tag_mode, h->tick_out_dev, n_out, h->stream)));
    else CUDA_TRY((launch_tick<T, BIAS, DIRECT, false>(a, h->tick_in_dev + 6, tag_mode, h->tick_out_dev, n_out, h->stream)));
    h->launches++;
    return QEKF_OK;
}

template <typename T, bool BIAS, bool DIRECT>
int step_typed(qekf_handle *h, double t_curr, const qekf_step_io *io)
{
    StepArgs<T> a;
    std::memset(&a, 0, sizeof a);
    a.st = dstate<T>(h);
    a.c = make_consts<T>(h->p);
    a.t_curr = t_curr;
    a.imu = io->imu; a.arrived = io->arrived; a.tag = io->tag;
    a.x_out = io->x_out; a.cov_out = io->cov_out; a.aux_out = io->aux_out; a.flags_out = io->flags_out;
    const bool mr = h->p.multirate_ekf != 0, pf = h->pf_on;
#define LAUNCH_STEP(MR_, PF_) CUDA_TRY((launch_step<T, BIAS, DIRECT, MR_, PF_>(a, h->step_block, h->stream)))
    if (mr && pf) LAUNCH_STEP(true, true);
    else if (mr) LAUNCH_STEP(true, false);
    else if (pf) LAUNCH_STEP(false, true);
    else LAUNCH_STEP(false, false);
#undef LAUNCH_STEP
    h->launches++;
    return QEKF_OK;
}

// the step kernels' launch attributes for the current parameters and precision, set here rather than at the launch, so
// that qekf_step issues nothing but the kernel (it may be captured into a CUDA graph); called wherever the handle is
// created or changes shape
int prep_step_kernels(qekf_handle *h)
{
#define PREP_ONE(T_, B_, D_, MR_, PF_) CUDA_TRY((prep_step<T_, B_, D_, MR_, PF_>(h->step_block)))
#define PREP_T(T_, B_, D_)                                                                                             \
    do {                                                                                                               \
        PREP_ONE(T_, B_, D_, false, false); PREP_ONE(T_, B_, D_, false, true);                                         \
        PREP_ONE(T_, B_, D_, true, false); PREP_ONE(T_, B_, D_, true, true);                                           \
    } while (0)
    QEKF_DISPATCH(h, PREP_T);
#undef PREP_T
#undef PREP_ONE
    return QEKF_OK;
}

// a pointer the step kernel may dereference: device memory of the handle's device, managed, or registered / pinned host
// memory (cudaPointerGetAttributes queries the driver's tables only: it enqueues nothing and is legal during capture)
int check_step_ptr(const qekf_handle *h, const void *p, const char *what)
{
    if (!p) return QEKF_OK;
    cudaPointerAttributes at;
    cudaError_t e = cudaPointerGetAttributes(&at, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(QEKF_ERR_BAD_ARG, std::string("qekf_step: cannot query ") + what);
    }
    if (at.type == cudaMemoryTypeUnregistered)
        return fail(QEKF_ERR_BAD_ARG, std::string("qekf_step: ") + what + " is unregistered host memory (it must be device memory)");
    if (at.type == cudaMemoryTypeDevice && at.device != h->device)
        return fail(QEKF_ERR_BAD_ARG, std::string("qekf_step: ") + what + " lives on another device");
    return QEKF_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char *qekf_last_error_string(void) { return g_err.c_str(); }

int qekf_default_params(qekf_params *p)
{
    if (!p) return fail(QEKF_ERR_BAD_ARG, "params is NULL");
    std::memset(p, 0, sizeof *p);
    p->update_freq = 100;                 // cpp:29
    p->measurement_freq = 10;             // cpp:30
    p->measurement_delay = 0.010;         // cpp:31
    p->measurement_delay_max = 0.200;     // cpp:32
    p->dyn_measurement_delay_offset = 0;  // node.cpp:35
    for (int i = 0; i < 3; ++i) {         // cpp:43-46
        p->Q_a[i] = 0.005; p->Q_w[i] = 0.0005; p->Q_ab[i] = 5e-5; p->Q_wb[i] = 5e-6;
    }
    p->R_r[0] = 0.005; p->R_r[1] = 0.005; p->R_r[2] = 0.015;        // cpp:50
    p->R_ang[0] = 0.0025; p->R_ang[1] = 0.0025; p->R_ang[2] = 0.025; // cpp:51
    p->r_cov_init = 0.1; p->v_cov_init = 0.1; p->ang_cov_init = 0.15; // node.cpp:89-93
    p->ab_cov_init = 0.5; p->wb_cov_init = 0.1;
    p->r_v_cv[2] = -0.073;                // cpp:55
    p->q_vc[0] = 0.70711; p->q_vc[1] = -0.70711;  // cpp:56 (w,x,y,z ctor) == node.cpp:109 (x,y,z,w array)
    p->camera_K[0] = 241.4268; p->camera_K[2] = 376.5;   // cpp:59-61
    p->camera_K[4] = 241.4268; p->camera_K[5] = 240.5; p->camera_K[8] = 1;
    p->camera_width = 752; p->camera_height = 480;       // cpp:62-63
    p->n_tags = 1; p->tag_in_view_margin = 0.02;         // cpp:66-67
    p->tag_widths[0] = 0.8;                              // cpp:69
    p->small_ang_tol = 1e-10; p->g[2] = -9.8;            // cpp:80-81
    p->est_bias = 1; p->limit_measurement_freq = 0; p->corner_margin_enbl = 1;   // cpp:34-36
    p->direct_orien_method = 0; p->multirate_ekf = 0; p->dynamic_meas_delay = 0; // cpp:37-38, node.cpp:64
    return QEKF_OK;
}

int qekf_params_from_yaml_text(const char *text, qekf_params *p)
{
    if (!text || !p) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    qekf::preset::Doc doc;
    std::string err = qekf::preset::parse(text, &doc);
    if (!err.empty()) return fail(QEKF_ERR_BAD_ARG, "parameter file: " + err);
    qekf_params q;
    qekf_default_params(&q);
    err = qekf::preset::apply(doc, &q);
    if (!err.empty()) return fail(QEKF_ERR_BAD_ARG, "parameter file: " + err);
    int rc = check_params(&q);
    if (rc) return rc;
    *p = q;
    return QEKF_OK;
}

int qekf_params_from_yaml(const char *path, qekf_params *p)
{
    if (!path || !p) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    FILE *f = std::fopen(path, "rb");
    if (!f) return fail(QEKF_ERR_BAD_ARG, std::string("cannot open parameter file ") + path);
    std::string text;
    char buf[4096];
    size_t n;
    while ((n = std::fread(buf, 1, sizeof buf, f)) > 0) text.append(buf, n);
    std::fclose(f);
    return qekf_params_from_yaml_text(text.c_str(), p);
}

int qekf_create(const qekf_params *p, int64_t n_filters, int device, int precision, qekf_handle **out)
{
    if (!out) return fail(QEKF_ERR_BAD_ARG, "out is NULL");
    *out = nullptr;
    int rc = check_params(p);
    if (rc) return rc;
    if (n_filters <= 0) return fail(QEKF_ERR_BAD_ARG, "n_filters must be positive");
    if (precision != QEKF_FP64 && precision != QEKF_FP32) return fail(QEKF_ERR_BAD_ARG, "precision must be 64 or 32");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        return fail(QEKF_ERR_NO_DEVICE, "no CUDA device available (libqekf has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return fail(QEKF_ERR_BAD_ARG, "device index out of range");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(QEKF_ERR_NO_DEVICE, "libqekf is built for sm_100a (B200) only");
    qekf_handle *h = new (std::nothrow) qekf_handle;
    if (!h) return fail(QEKF_ERR_ALLOC, "out of host memory");
    h->p = *p; h->precision = precision; h->device = device;
    h->step_block = step_block_default(precision == QEKF_FP64);
    {   // environment overrides of the default mapping (profiling / A-B runs): QEKF_LANES=1|3, QEKF_COOP_GROUPS=n
        const char *e = getenv("QEKF_LANES");
        if (e && atoi(e) >= 1 && atoi(e) <= 3) h->lanes_per_filter = atoi(e);
        e = getenv("QEKF_COOP_GROUPS");
        if (e && coop_groups_available(atoi(e), p->est_bias && p->direct_orien_method)) h->coop_groups = atoi(e);
        e = getenv("QEKF_NO_PERM");
        if (e && atoi(e) != 0) h->perm_on = false;
        e = getenv("QEKF_NO_LAZY_MR");
        if (e && atoi(e) != 0) h->lazy_mr_on = false;
        e = getenv("QEKF_PERM_MIN_STEPS");
        if (e && atoll(e) > 0) h->perm_min_steps = atoll(e);
        e = getenv("QEKF_DUO_GROUPS");
        if (e && duo_groups_available(atoi(e), p->est_bias && p->direct_orien_method)) h->duo_groups = atoi(e);
        e = getenv("QEKF_STEP_BLOCK");
        if (e) for (int b : STEP_BLOCKS) if (atoi(e) == b) h->step_block = b;
    }
    h->n = n_filters; h->ld = (n_filters + 31) / 32 * 32;
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return fail(QEKF_ERR_CUDA, "cudaStreamCreate failed");
    }
    h->own_stream = true;
    rc = alloc_state(h);
    if (!rc) rc = reset_cov(h, true);
    if (!rc) rc = prep_step_kernels(h);
    if (rc) { free_state(h); cudaStreamDestroy(h->stream); delete h; return rc; }
    *out = h;
    return QEKF_OK;
}

int qekf_destroy(qekf_handle *h)
{
    if (!h) return QEKF_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    free_state(h);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
    return QEKF_OK;
}

int qekf_set_params(qekf_handle *h, const qekf_params *p)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    int rc = check_params(p);
    if (rc) return rc;
    if (h->pf_on && h->pf_overridden[QEKF_PF_DELAY]) {
        // the per-filter delays stay in force: they must still fit the ring with the new update rate
        const std::vector<double> &v = h->pf_host[QEKF_PF_DELAY];
        for (size_t i = 0; i < (size_t)h->n; ++i)
            if (step_of_delay(v[i], p->update_freq) > 4096)
                return fail(QEKF_ERR_BAD_ARG, "a per-filter measurement_delay spans more than 4096 ticks at the new update_freq");
    }
    CUDA_TRY(cudaSetDevice(h->device));
    const bool shape_change = (p->est_bias != 0) != (h->p.est_bias != 0);
    h->p = *p;
    rc = prep_step_kernels(h);     // (est_bias, direct_orien_method and multirate_ekf pick the step kernel)
    if (rc) return rc;
    if (shape_change) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        free_state(h);
        rc = alloc_state(h);
        if (rc) return rc;
        return reset_cov(h, true);
    }
    rc = reset_cov(h, false);     // initialize_params: cov_pert = cov_init (cpp:114)
    if (rc) return rc;
    if (h->pf_on) {
        // fields never overridden follow the handle-wide value (include/qekf.h): re-seed them from the new parameters
        for (int f = 0; f < 5; ++f)
            if (!h->pf_overridden[f]) seed_pf_field(h, f);
        rc = rebuild_pf(h);
        if (rc) return rc;
    }
    if (!h->p.multirate_ekf) return QEKF_OK;
    // Delayed fusion: the history restarts from the current head.  (The reference keeps its old history
    // vectors here, so its next delayed correction would silently discard the covariance reset.)
    rc = alloc_history(h);
    if (rc) return rc;
    return rebase_all(h);
}

int qekf_get_params(const qekf_handle *h, qekf_params *p)
{
    if (!h || !p) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    *p = h->p;
    return QEKF_OK;
}

int qekf_set_filter_params(qekf_handle *h, int field, const double *values)
{
    static const int dims[5] = { 12, 6, 3, 4, 2 };
    if (!h || !values) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (field < 0 || field > QEKF_PF_DELAY) return fail(QEKF_ERR_BAD_ARG, "unknown per-filter field");
    const size_t N = (size_t)h->n;
    // validate before anything is allocated or enabled: a rejected call leaves the handle as it was
    if (field == QEKF_PF_DELAY)
        for (size_t i = 0; i < N; ++i)
            if (!(values[i] >= 0) || step_of_delay(values[i], h->p.update_freq) > 4096)
                return fail(QEKF_ERR_BAD_ARG, "per-filter measurement_delay out of range");
    CUDA_TRY(cudaSetDevice(h->device));
    const bool first = !h->pf_on;
    if (first) {
        // first override: every field starts from the handle-wide parameters
        for (int f = 0; f < 5; ++f) { seed_pf_field(h, f); h->pf_overridden[f] = false; }
        if (cudaMalloc(&h->pf, (size_t)PF_DIM * (size_t)h->ld * h->tsize) != cudaSuccess ||
            cudaMalloc(&h->pf_delay, 2 * (size_t)h->ld * sizeof(double)) != cudaSuccess) {
            cudaGetLastError();
            cudaFree(h->pf); cudaFree(h->pf_delay);
            h->pf = nullptr; h->pf_delay = nullptr;
            for (auto &v : h->pf_host) v.clear();
            return fail(QEKF_ERR_CUDA, "out of device memory for the per-filter parameter tables");
        }
    }
    std::vector<double> previous;
    if (!first) previous = h->pf_host[field];
    std::memcpy(h->pf_host[field].data(), values, (size_t)dims[field] * N * sizeof(double));
    int rc = rebuild_pf(h);
    if (rc) {
        // the device tables are not trustworthy: first call -> overrides stay off; later call -> previous values back
        if (first) {
            cudaFree(h->pf); cudaFree(h->pf_delay);
            h->pf = nullptr; h->pf_delay = nullptr;
            for (auto &v : h->pf_host) v.clear();
        } else {
            h->pf_host[field] = previous;
            rebuild_pf(h);
        }
        return rc;
    }
    h->pf_on = true;                 // only now do the replay kernels read the tables
    h->pf_overridden[field] = true;
    if (field == QEKF_PF_DELAY && h->p.multirate_ekf) {
        const int old_len = h->ring_len;
        rc = alloc_history(h);
        if (rc) return rc;
        if (h->ring_len != old_len) return rebase_all(h);
    }
    return QEKF_OK;
}

int qekf_num_states(const qekf_handle *h) { return h ? h->nstates : 0; }
int64_t qekf_num_filters(const qekf_handle *h) { return h ? h->n : 0; }

int qekf_set_mapping(qekf_handle *h, int lanes_per_filter, int groups)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    if (lanes_per_filter < 1 || lanes_per_filter > 3) return fail(QEKF_ERR_BAD_ARG, "lanes_per_filter must be 1, 2 or 3");
    const bool bench_variant = h->p.est_bias && h->p.direct_orien_method && !h->pf_on;
    if (lanes_per_filter == 3) {
        if (groups == 0) groups = COOP_GROUPS_DEFAULT;
        if (!coop_groups_available(groups, bench_variant))
            return fail(QEKF_ERR_BAD_ARG, "this build has no three-lane kernel with that many groups per CTA for this filter variant");
        h->coop_groups = groups;
    } else if (lanes_per_filter == 2) {
        if (groups == 0) groups = DUO_GROUPS_DEFAULT;
        if (!duo_groups_available(groups, bench_variant))
            return fail(QEKF_ERR_BAD_ARG, "this build has no two-role kernel with that many groups per CTA for this filter variant");
        h->duo_groups = groups;
    }
    h->lanes_per_filter = lanes_per_filter;
    return QEKF_OK;
}

int qekf_set_stream(qekf_handle *h, void *cuda_stream)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->own_stream) cudaStreamDestroy(h->stream);
    h->stream = (cudaStream_t)cuda_stream;
    h->own_stream = false;
    return QEKF_OK;
}

int qekf_sync(qekf_handle *h)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return QEKF_OK;
}

// ---- per-tick estimator interface ----------------------------------------------------------------

int qekf_set_imu(qekf_handle *h, const double accel[3], const double gyro[3])
{
    if (!h || !accel || !gyro) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    for (int i = 0; i < 3; ++i) { h->imu_latched[i] = accel[i]; h->imu_latched[3 + i] = gyro[i]; }
    return QEKF_OK;
}

static int deliver(qekf_handle *h, int force_init, int reinit_bias, int raise_ready = 1)
{
    if (h) hist_touch(h);
#define CALL_DELIVER(T, B, D)                                                                                          \
    do {                                                                                                               \
        if (h->pf_on)                                                                                                  \
            CUDA_TRY((launch_deliver<T, B, true>(dstate<T>(h), make_consts<T>(h->p), h->d_tick + 8, force_init,        \
                                                 reinit_bias, raise_ready, grid_of(h), smem_bytes(h), h->stream)));    \
        else                                                                                                           \
            CUDA_TRY((launch_deliver<T, B, false>(dstate<T>(h), make_consts<T>(h->p), h->d_tick + 8, force_init,       \
                                                  reinit_bias, raise_ready, grid_of(h), smem_bytes(h), h->stream)));   \
    } while (0)
    QEKF_DISPATCH(h, CALL_DELIVER);
#undef CALL_DELIVER
    h->launches++;
    return QEKF_OK;
}

static int stage_tag(qekf_handle *h, const double pos[3], const double quat_xyzw[4], double stamp)
{
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));   // the pinned staging buffer is reused
    for (int i = 0; i < 3; ++i) h->h_tick[8 + i] = pos[i];
    for (int i = 0; i < 4; ++i) h->h_tick[11 + i] = quat_xyzw[i];
    h->h_tick[15] = stamp;
    CUDA_TRY(cudaMemcpyAsync(h->d_tick + 8, h->h_tick + 8, 8 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    return QEKF_OK;
}

int qekf_set_tag(qekf_handle *h, const double pos[3], const double quat_xyzw[4], double stamp)
{
    if (!h || !pos || !quat_xyzw) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    int rc = stage_tag(h, pos, quat_xyzw, stamp);
    if (rc) return rc;
    return deliver(h, 0, 0, 1);
}

int qekf_latch_tag(qekf_handle *h, const double pos[3], const double quat_xyzw[4], double stamp)
{
    if (!h || !pos || !quat_xyzw) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    int rc = stage_tag(h, pos, quat_xyzw, stamp);
    if (rc) return rc;
    return deliver(h, 0, 0, 0);
}

int qekf_initialize_state(qekf_handle *h, int reinit_bias)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    return deliver(h, 1, reinit_bias);
}

int qekf_tick(qekf_handle *h, const double accel[3], const double gyro[3], int tag_mode, const double tag_pos[3],
              const double tag_quat_xyzw[4], double tag_stamp, double t_curr, int n_out, double *records)
{
    if (h) hist_touch(h);
    if (!h || !accel || !gyro) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (tag_mode < 0 || tag_mode > 2 || (tag_mode != 0 && (!tag_pos || !tag_quat_xyzw)))
        return fail(QEKF_ERR_BAD_ARG, "bad tag_mode, or a tag without a pose");
    if (n_out < 0 || n_out > h->n || n_out > 4096 || (n_out > 0 && !records)) return fail(QEKF_ERR_BAD_ARG, "bad record count");
    if (h->pf_on) return fail(QEKF_ERR_BAD_ARG, "qekf_tick does not serve handles with per-filter parameter overrides");
    CUDA_TRY(cudaSetDevice(h->device));
    if (!h->tick_in) {
        CUDA_TRY(cudaHostAlloc(&h->tick_in, 16 * sizeof(double), cudaHostAllocMapped));
        CUDA_TRY(cudaHostGetDevicePointer(&h->tick_in_dev, h->tick_in, 0));
    }
    if (n_out > h->tick_out_cap) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (h->tick_out) cudaFreeHost(h->tick_out);
        h->tick_out = nullptr; h->tick_out_cap = 0;
        CUDA_TRY(cudaHostAlloc(&h->tick_out, (size_t)n_out * TICK_REC * sizeof(double), cudaHostAllocMapped));
        CUDA_TRY(cudaHostGetDevicePointer(&h->tick_out_dev, h->tick_out, 0));
        h->tick_out_cap = n_out;
    }
    // (the previous tick ended with a stream synchronisation, so the mapped input words are free)
    for (int i = 0; i < 3; ++i) { h->tick_in[i] = accel[i]; h->tick_in[3 + i] = gyro[i]; h->imu_latched[i] = accel[i]; h->imu_latched[3 + i] = gyro[i]; }
    if (tag_mode != 0) {
        for (int i = 0; i < 3; ++i) h->tick_in[6 + i] = tag_pos[i];
        for (int i = 0; i < 4; ++i) h->tick_in[9 + i] = tag_quat_xyzw[i];
        h->tick_in[13] = tag_stamp;
    }
    int rc = QEKF_OK;
#define CALL_TICK(T, B, D) rc = tick_typed<T, B, D>(h, tag_mode, t_curr, n_out)
    QEKF_DISPATCH(h, CALL_TICK);
#undef CALL_TICK
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (n_out > 0) std::memcpy(records, h->tick_out, (size_t)n_out * TICK_REC * sizeof(double));
    return QEKF_OK;
}

int qekf_step(qekf_handle *h, double t_curr, const qekf_step_io *io)
{
    if (h) hist_touch(h);
    if (!h || !io || !io->imu) return fail(QEKF_ERR_BAD_ARG, "qekf_step: NULL handle, io or imu");
    if (io->arrived && !io->tag) return fail(QEKF_ERR_BAD_ARG, "qekf_step: arrived given without tag");
    CUDA_TRY(cudaSetDevice(h->device));
    const void *ptrs[7] = { io->imu, io->arrived, io->tag, io->x_out, io->cov_out, io->aux_out, io->flags_out };
    const char *names[7] = { "imu", "arrived", "tag", "x_out", "cov_out", "aux_out", "flags_out" };
    for (int k = 0; k < 7; ++k) {
        int rc = check_step_ptr(h, ptrs[k], names[k]);
        if (rc) return rc;
    }
    int rc = QEKF_OK;
#define CALL_STEP(T, B, D) rc = step_typed<T, B, D>(h, t_curr, io)
    QEKF_DISPATCH(h, CALL_STEP);
#undef CALL_STEP
    return rc;
}

int qekf_filter_update(qekf_handle *h, double t_curr)
{
    if (h) hist_touch(h);
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 6; ++i) h->h_tick[i] = h->imu_latched[i];
    CUDA_TRY(cudaMemcpyAsync(h->d_tick, h->h_tick, 6 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    StreamView in;
    std::memset(&in, 0, sizeof in);
    in.imu = h->d_tick; in.cs = 1; in.is = 0; in.M = 0;
    in.tag_pose = h->d_tick + 8;      // never read: M = 0 and the latched pose lives in st.pend
    in.t_start = t_curr; in.update_freq = h->p.update_freq;
    return run_dispatch(h, in, 0, 1, 0);
}

// ---- batch replay ----------------------------------------------------------------------------------

int qekf_run(qekf_handle *h, const qekf_streams *s, int64_t k0, int64_t n_steps)
{
    return qekf_run_with_truth(h, s, nullptr, k0, n_steps);
}

int qekf_run_with_truth(qekf_handle *h, const qekf_streams *s, const double *truth, int64_t k0, int64_t n_steps)
{
    if (h) hist_touch(h);
    if (!h || !s) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (truth && !h->stats_acc) return fail(QEKF_ERR_NOT_INITIALIZED, "truth given but statistics are not configured");
    if (n_steps == 0) return QEKF_OK;
    if (k0 < 0 || n_steps < 0 || k0 + n_steps > s->T) return fail(QEKF_ERR_BAD_ARG, "tick range outside the stream");
    if (k0 + n_steps > 2147483647LL) return fail(QEKF_ERR_BAD_ARG, "tick indices are limited to 31 bits (as tag_step is)");
    if (!s->imu) return fail(QEKF_ERR_BAD_ARG, "imu stream is NULL");
    if (s->M < 0 || (s->M > 0 && (!s->tag_step || !s->tag_pose || !s->tag_stamp)))
        return fail(QEKF_ERR_BAD_ARG, "tag streams are NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    const int64_t N = h->n, M = s->M, T = s->T;
    // the bins sampled by this call: bin b is sampled after tick (b+1)*stride - 1, so [k0, k0+n_steps) holds the bins
    // [k0/stride, (k0+n_steps)/stride), clipped to the configured ones.  None: a plain replay (nothing to score).
    int64_t b_lo = 0, b_hi = 0;
    if (truth) {
        b_lo = std::min<int64_t>(k0 / h->stats_stride, h->stats_bins);
        b_hi = std::min<int64_t>((k0 + n_steps) / h->stats_stride, h->stats_bins);
        if (b_hi <= b_lo) truth = nullptr;
    }

    // arrivals must be strictly increasing; the first one at or after k0 is where this launch starts
    std::vector<int32_t> steps_host;
    const int32_t *steps = s->tag_step;
    if (s->on_device && M > 0) {
        steps_host.resize((size_t)M);
        CUDA_TRY(cudaMemcpy(steps_host.data(), s->tag_step, (size_t)M * sizeof(int32_t), cudaMemcpyDeviceToHost));
        steps = steps_host.data();
    }
    int32_t m0 = 0;
    for (int64_t m = 0; m < M; ++m) {
        if (m > 0 && steps[m] <= steps[m - 1]) return fail(QEKF_ERR_BAD_ARG, "tag_step must be strictly increasing");
        if (steps[m] < k0) m0 = (int32_t)(m + 1);
    }

    StreamView in;
    std::memset(&in, 0, sizeof in);
    in.cs = N; in.is = 1; in.M = M; in.vs = N;
    in.t_start = s->t_start; in.update_freq = h->p.update_freq;
    if (s->on_device) {
        in.imu = s->imu; in.tag_step = s->tag_step; in.tag_pose = s->tag_pose;
        in.tag_stamp = s->tag_stamp; in.tag_valid = s->tag_valid;
    } else {
        // host streams: stage the ticks of this call (and every arrival), and the truth of the bins it samples, into one
        // device slab
        const size_t imu_b = (size_t)n_steps * 6 * (size_t)N * 8;
        const size_t pose_b = (size_t)M * 7 * (size_t)N * 8;
        const size_t stamp_b = (size_t)M * 8, step_b = (size_t)M * 4;
        const size_t valid_b = s->tag_valid ? (size_t)M * (size_t)N : 0;
        const size_t truth_b = truth ? (size_t)(b_hi - b_lo) * 16 * (size_t)N * 8 : 0;
        size_t o_imu = 0, o_pose = align_up(o_imu + imu_b, 256), o_stamp = align_up(o_pose + pose_b, 256);
        size_t o_step = align_up(o_stamp + stamp_b, 256), o_valid = align_up(o_step + step_b, 256);
        size_t o_truth = align_up(o_valid + valid_b, 256);
        size_t total = align_up(o_truth + truth_b, 256);
        int rc = ensure_in(h, total);
        if (rc) return rc;
        char *d = (char *)h->d_in;
        CUDA_TRY(cudaMemcpyAsync(d + o_imu, s->imu + (size_t)k0 * 6 * (size_t)N, imu_b, cudaMemcpyHostToDevice, h->stream));
        if (M > 0) {
            CUDA_TRY(cudaMemcpyAsync(d + o_pose, s->tag_pose, pose_b, cudaMemcpyHostToDevice, h->stream));
            CUDA_TRY(cudaMemcpyAsync(d + o_stamp, s->tag_stamp, stamp_b, cudaMemcpyHostToDevice, h->stream));
            CUDA_TRY(cudaMemcpyAsync(d + o_step, s->tag_step, step_b, cudaMemcpyHostToDevice, h->stream));
            if (valid_b) CUDA_TRY(cudaMemcpyAsync(d + o_valid, s->tag_valid, valid_b, cudaMemcpyHostToDevice, h->stream));
        }
        // the staged imu slab starts at tick k0: bias the base pointer so absolute tick indices work
        in.imu = (const double *)(d + o_imu) - (size_t)k0 * 6 * (size_t)N;
        in.tag_pose = (const double *)(d + o_pose);
        in.tag_stamp = (const double *)(d + o_stamp);
        in.tag_step = (const int32_t *)(d + o_step);
        in.tag_valid = valid_b ? (const uint8_t *)(d + o_valid) : nullptr;
        if (truth_b) {
            CUDA_TRY(cudaMemcpyAsync(d + o_truth, truth + (size_t)b_lo * 16 * (size_t)N, truth_b, cudaMemcpyHostToDevice,
                                     h->stream));
            // as the imu slab: the staged bins start at b_lo, bias the base pointer so absolute bin indices work
            truth = (const double *)(d + o_truth) - (size_t)b_lo * 16 * (size_t)N;
        }
    }
    (void)T;
    return run_dispatch(h, in, k0, n_steps, m0, nullptr, truth);
}

// ---- accessors ---------------------------------------------------------------------------------------

int qekf_get_state(qekf_handle *h, int64_t first, int64_t count, double *x16)
{
    if (!range_ok(h, first, count) || !x16) return fail(QEKF_ERR_BAD_ARG, "bad range or NULL output");
    CUDA_TRY(cudaSetDevice(h->device));
    return fetch_rows(h, h->x, 16, first, count, x16);
}

int qekf_get_cov(qekf_handle *h, int64_t first, int64_t count, double *P)
{
    if (!range_ok(h, first, count) || !P) return fail(QEKF_ERR_BAD_ARG, "bad range or NULL output");
    CUDA_TRY(cudaSetDevice(h->device));
    std::vector<double> packed((size_t)h->np * (size_t)count);
    int rc = fetch_rows(h, h->P, h->np, first, count, packed.data());
    if (rc) return rc;
    const int n = h->nstates;
    int e = 0;
    for (int a = 0; a < n; ++a)
        for (int b = a; b < n; ++b, ++e) {
            const double *src = packed.data() + (size_t)e * (size_t)count;
            std::memcpy(P + ((size_t)a * n + b) * (size_t)count, src, (size_t)count * 8);
            if (a != b) std::memcpy(P + ((size_t)b * n + a) * (size_t)count, src, (size_t)count * 8);
        }
    return QEKF_OK;
}

int qekf_get_aux(qekf_handle *h, int64_t first, int64_t count, double *aux11)
{
    if (!range_ok(h, first, count) || !aux11) return fail(QEKF_ERR_BAD_ARG, "bad range or NULL output");
    CUDA_TRY(cudaSetDevice(h->device));
    return fetch_rows(h, h->aux, AUX_DIM, first, count, aux11);
}

int qekf_get_flags(qekf_handle *h, int64_t first, int64_t count, int32_t *flags6)
{
    if (!range_ok(h, first, count) || !flags6) return fail(QEKF_ERR_BAD_ARG, "bad range or NULL output");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    std::vector<int32_t> fl((size_t)count), up((size_t)count), hl;
    CUDA_TRY(cudaMemcpy(fl.data(), h->flags + first, (size_t)count * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(up.data(), h->upds + first, (size_t)count * 4, cudaMemcpyDeviceToHost));
    if (h->hlen) {
        hl.resize((size_t)count);
        CUDA_TRY(cudaMemcpy(hl.data(), h->hlen + first, (size_t)count * 4, cudaMemcpyDeviceToHost));
    }
    for (int64_t i = 0; i < count; ++i) {
        const int32_t f = fl[(size_t)i];
        flags6[0 * count + i] = (f & FLAG_INIT) ? 1 : 0;
        flags6[1 * count + i] = (f & FLAG_READY) ? 1 : 0;
        flags6[2 * count + i] = (f & FLAG_CORRECTED) ? 1 : 0;
        flags6[3 * count + i] = (f & FLAG_ACTIVE) ? 1 : 0;
        flags6[4 * count + i] = up[(size_t)i];
        // x_hist.size(): single-rate filters keep the one entry initialize_state wrote (cpp:326-339)
        flags6[5 * count + i] = (f & FLAG_INIT) ? (hl.empty() ? 1 : hl[(size_t)i]) : 0;
    }
    return QEKF_OK;
}

int qekf_set_state(qekf_handle *h, int64_t first, int64_t count, const double *x16, const double *P)
{
    if (h) hist_touch(h);
    if (!range_ok(h, first, count) || !x16 || !P) return fail(QEKF_ERR_BAD_ARG, "bad range or NULL input");
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = store_rows(h, h->x, 16, first, count, x16);
    if (rc) return rc;
    const int n = h->nstates;
    std::vector<double> packed((size_t)h->np * (size_t)count);
    int e = 0;
    for (int a = 0; a < n; ++a)
        for (int b = a; b < n; ++b, ++e)
            std::memcpy(packed.data() + (size_t)e * (size_t)count, P + ((size_t)a * n + b) * (size_t)count, (size_t)count * 8);
    rc = store_rows(h, h->P, h->np, first, count, packed.data());
    if (rc) return rc;
    std::vector<int32_t> fl((size_t)count);
    CUDA_TRY(cudaMemcpy(fl.data(), h->flags + first, (size_t)count * 4, cudaMemcpyDeviceToHost));
    for (auto &f : fl) f |= FLAG_INIT;
    CUDA_TRY(cudaMemcpy(h->flags + first, fl.data(), (size_t)count * 4, cudaMemcpyHostToDevice));
    if (h->xc) {   // history <- this entry
        rc = store_rows(h, h->xc, 16, first, count, x16);
        if (!rc) rc = store_rows(h, h->Pc, h->np, first, count, packed.data());
        if (rc) return rc;
        std::vector<int32_t> ones((size_t)count, 1);
        CUDA_TRY(cudaMemset(h->nh + first, 0, (size_t)count * 4));
        CUDA_TRY(cudaMemcpy(h->hlen + first, ones.data(), (size_t)count * 4, cudaMemcpyHostToDevice));
    }
    return QEKF_OK;
}

// ---- exact checkpoint / resume ---------------------------------------------------------------------------
// Everything a later run depends on, as one flat host blob: the device arrays of the handle verbatim (in the
// handle's own precision and padded layout, so nothing is rounded or reordered) behind a header that pins what the
// receiving handle must look like.

namespace {

struct ExportHeader {
    char magic[8];                 // "QEKFCKP2"
    int32_t precision, nstates, multirate, ring_len, dmax, stats_bins, stats_stride, reserved;
    int64_t n, ld, total_bytes;
    double imu_latched[6];
    // provenance of the delayed-fusion history entries (qekf_handle::hist_clean / hist_key)
    int32_t hist_clean, hist_key_valid;
    uint64_t hist_key[6];
    int64_t hist_k_next;
    qekf_params p;
};

struct Segment { void *dev; size_t bytes; };

std::vector<Segment> export_segments(const qekf_handle *h)
{
    const size_t ld = (size_t)h->ld, ts = h->tsize;
    std::vector<Segment> v = {
        { h->x, 16 * ld * ts }, { h->P, (size_t)h->np * ld * ts }, { h->aux, AUX_DIM * ld * ts },
        { h->pend, PEND_DIM * ld * sizeof(double) }, { h->flags, ld * sizeof(int32_t) }, { h->upds, ld * sizeof(int32_t) },
        { h->counts, 8 * sizeof(unsigned long long) } };
    if (h->xc) {
        v.push_back({ h->xc, 16 * ld * ts });
        v.push_back({ h->Pc, (size_t)h->np * ld * ts });
        v.push_back({ h->ring, (size_t)h->ring_len * 6 * ld * ts });
        v.push_back({ h->nh, ld * sizeof(int32_t) });
        v.push_back({ h->hpos, ld * sizeof(int32_t) });
        v.push_back({ h->hlen, ld * sizeof(int32_t) });
    }
    if (h->stats_acc) v.push_back({ h->stats_acc, (size_t)STAT_REPL * h->stats_bins * STAT_DIM * 8 });
    return v;
}

}  // namespace

int64_t qekf_export_size(const qekf_handle *h)
{
    if (!h) return 0;
    size_t b = sizeof(ExportHeader);
    for (const Segment &s : export_segments(h)) b += s.bytes;
    return (int64_t)b;
}

int qekf_export_state(qekf_handle *h, void *buf, int64_t bytes)
{
    if (!h || !buf) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    const int64_t need = qekf_export_size(h);
    if (bytes < need) return fail(QEKF_ERR_BAD_ARG, "export buffer is smaller than qekf_export_size()");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    ExportHeader hd;
    std::memset(&hd, 0, sizeof hd);
    std::memcpy(hd.magic, "QEKFCKP2", 8);
    hd.precision = h->precision; hd.nstates = h->nstates; hd.multirate = h->xc ? 1 : 0;
    hd.ring_len = h->ring_len; hd.dmax = h->dmax;
    hd.stats_bins = h->stats_acc ? h->stats_bins : 0; hd.stats_stride = h->stats_acc ? h->stats_stride : 0;
    hd.n = h->n; hd.ld = h->ld; hd.total_bytes = need;
    std::memcpy(hd.imu_latched, h->imu_latched, sizeof hd.imu_latched);
    hd.hist_clean = h->hist_clean; hd.hist_key_valid = h->hist_key_valid; hd.hist_k_next = h->hist_k_next;
    std::memcpy(hd.hist_key, h->hist_key, sizeof hd.hist_key);
    hd.p = h->p;
    unsigned char *out = static_cast<unsigned char *>(buf);
    std::memcpy(out, &hd, sizeof hd);
    size_t off = sizeof hd;
    for (const Segment &s : export_segments(h)) {
        CUDA_TRY(cudaMemcpy(out + off, s.dev, s.bytes, cudaMemcpyDeviceToHost));
        off += s.bytes;
    }
    return QEKF_OK;
}

int qekf_import_state(qekf_handle *h, const void *buf, int64_t bytes)
{
    if (!h || !buf) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (bytes < (int64_t)sizeof(ExportHeader)) return fail(QEKF_ERR_BAD_ARG, "blob is shorter than its header");
    ExportHeader hd;
    std::memcpy(&hd, buf, sizeof hd);
    if (std::memcmp(hd.magic, "QEKFCKP2", 8) != 0) return fail(QEKF_ERR_BAD_ARG, "not a qekf_export_state blob");
    if (hd.total_bytes > bytes) return fail(QEKF_ERR_BAD_ARG, "blob is truncated");
    if (hd.n != h->n || hd.ld != h->ld || hd.precision != h->precision || hd.nstates != h->nstates)
        return fail(QEKF_ERR_BAD_ARG, "blob was exported from a handle of another size, precision or est_bias");
    if (std::memcmp(&hd.p, &h->p, sizeof(qekf_params)) != 0)
        return fail(QEKF_ERR_BAD_ARG, "blob was exported under other parameters (create the handle with the same qekf_params)");
    if (hd.multirate != (h->xc ? 1 : 0) || hd.ring_len != h->ring_len || hd.dmax != h->dmax)
        return fail(QEKF_ERR_BAD_ARG, "delayed-fusion history of the blob does not fit this handle (apply the same per-filter "
                                      "delay overrides before importing)");
    CUDA_TRY(cudaSetDevice(h->device));
    if (hd.stats_bins > 0 && (!h->stats_acc || h->stats_bins != hd.stats_bins || h->stats_stride != hd.stats_stride)) {
        int rc = qekf_stats_configure(h, hd.stats_bins, hd.stats_stride);
        if (rc) return rc;
    }
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    std::vector<Segment> segs = export_segments(h);
    if (hd.stats_bins == 0 && h->stats_acc) segs.pop_back();      // the blob carries no accumulators: keep ours
    size_t need = sizeof hd;
    for (const Segment &s : segs) need += s.bytes;
    if ((int64_t)need != hd.total_bytes) return fail(QEKF_ERR_BAD_ARG, "blob size does not match this handle's layout");
    const unsigned char *in = static_cast<const unsigned char *>(buf);
    size_t off = sizeof hd;
    for (const Segment &s : segs) {
        CUDA_TRY(cudaMemcpy(s.dev, in + off, s.bytes, cudaMemcpyHostToDevice));
        off += s.bytes;
    }
    std::memcpy(h->imu_latched, hd.imu_latched, sizeof hd.imu_latched);
    h->hist_clean = hd.hist_clean != 0; h->hist_key_valid = hd.hist_key_valid != 0; h->hist_k_next = hd.hist_k_next;
    std::memcpy(h->hist_key, hd.hist_key, sizeof hd.hist_key);
    return QEKF_OK;
}

// ---- stateless step functions ------------------------------------------------------------------------

static int stage_rows(qekf_handle *h, const double *host, int rows)
{
    // [rows][N] host -> [rows][ld] device slab in d_in
    int rc = ensure_in(h, (size_t)rows * (size_t)h->ld * 8);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpy2DAsync(h->d_in, (size_t)h->ld * 8, host, (size_t)h->n * 8, (size_t)h->n * 8, (size_t)rows,
                               cudaMemcpyHostToDevice, h->stream));
    return QEKF_OK;
}

int qekf_prediction_step(qekf_handle *h, const double *u)
{
    if (h) hist_touch(h);
    if (!h || !u) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = stage_rows(h, u, 6);
    if (rc) return rc;
#define CALL_PRED(T, B, D)                                                                                         \
    do {                                                                                                           \
        if (h->pf_on)                                                                                              \
            CUDA_TRY((launch_predict<T, B, true>(dstate<T>(h), make_consts<T>(h->p), (const double *)h->d_in,      \
                                                 grid_of(h), smem_bytes(h), h->stream)));                          \
        else                                                                                                       \
            CUDA_TRY((launch_predict<T, B, false>(dstate<T>(h), make_consts<T>(h->p), (const double *)h->d_in,     \
                                                  grid_of(h), smem_bytes(h), h->stream)));                         \
    } while (0)
    QEKF_DISPATCH(h, CALL_PRED);
#undef CALL_PRED
    h->launches++;
    return QEKF_OK;
}

int qekf_correction_step(qekf_handle *h, const double *tag_pose)
{
    if (h) hist_touch(h);
    if (!h || !tag_pose) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    int rc = stage_rows(h, tag_pose, 7);
    if (rc) return rc;
#define CALL_CORR(T, B, D)                                                                                         \
    do {                                                                                                           \
        if (h->pf_on)                                                                                              \
            CUDA_TRY((launch_correct<T, B, D, true>(dstate<T>(h), make_consts<T>(h->p), (const double *)h->d_in,   \
                                                    grid_of(h), smem_bytes(h), h->stream)));                       \
        else                                                                                                       \
            CUDA_TRY((launch_correct<T, B, D, false>(dstate<T>(h), make_consts<T>(h->p), (const double *)h->d_in,  \
                                                     grid_of(h), smem_bytes(h), h->stream)));                      \
    } while (0)
    QEKF_DISPATCH(h, CALL_CORR);
#undef CALL_CORR
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return QEKF_OK;
}

// ---- Monte-Carlo replay ---------------------------------------------------------------------------------

int qekf_noise_default(qekf_noise_spec *n)
{
    if (!n) return fail(QEKF_ERR_BAD_ARG, "noise spec is NULL");
    std::memset(n, 0, sizeof *n);
    n->seed = 0x5EEDull;
    n->sigma_accel = 0.02; n->sigma_gyro = 0.007;
    n->sigma_bias_accel = 0.05; n->sigma_bias_gyro = 0.002;
    n->sigma_tag_pos = 0.02; n->sigma_tag_ang = 0.01;
    return QEKF_OK;
}

static NoiseSpec to_device_noise(const qekf_noise_spec &n)
{
    NoiseSpec d;
    std::memset(&d, 0, sizeof d);
    d.seed = n.seed; d.gid0 = n.first_global_id;
    d.sig_a = (float)n.sigma_accel; d.sig_w = (float)n.sigma_gyro;
    d.sig_ba = (float)n.sigma_bias_accel; d.sig_bw = (float)n.sigma_bias_gyro;
    d.sig_p = (float)n.sigma_tag_pos; d.sig_th = (float)n.sigma_tag_ang;
    d.drop_k0 = n.dropout_k0; d.drop_k1 = n.dropout_k1;
    d.rdrop_len = n.rand_dropout_len; d.rdrop_lo = n.rand_dropout_lo; d.rdrop_hi = n.rand_dropout_hi;
    d.edge_loss = n.edge_loss;
    d.range_ref = n.range_ref; d.range_exp_p = n.range_exp_pos; d.range_exp_th = n.range_exp_ang;
    return d;
}

// Build the kernel's view of a shared clean scenario; host arrays are staged into the handle's slab.
static int shared_view(qekf_handle *h, const qekf_shared_streams *s, const qekf_noise_spec *n, StreamView *in,
                       const double **truth, std::vector<int32_t> *steps_host)
{
    if (!s->imu_clean || s->T <= 0) return fail(QEKF_ERR_BAD_ARG, "imu_clean is NULL or T <= 0");
    if (s->M < 0 || (s->M > 0 && (!s->tag_step || !s->tag_pose_clean || !s->tag_stamp)))
        return fail(QEKF_ERR_BAD_ARG, "tag streams are NULL");
    const int64_t T = s->T, M = s->M;
    steps_host->resize((size_t)M);
    if (M > 0) {
        if (s->on_device)
            CUDA_TRY(cudaMemcpy(steps_host->data(), s->tag_step, (size_t)M * 4, cudaMemcpyDeviceToHost));
        else
            std::memcpy(steps_host->data(), s->tag_step, (size_t)M * 4);
    }
    for (int64_t m = 1; m < M; ++m)
        if ((*steps_host)[m] <= (*steps_host)[m - 1]) return fail(QEKF_ERR_BAD_ARG, "tag_step must be strictly increasing");
    std::memset(in, 0, sizeof *in);
    in->cs = 1; in->is = 0; in->M = M; in->vs = 0;
    in->t_start = s->t_start; in->update_freq = h->p.update_freq;
    // detection front-end: which arrivals see the bundle inside the image, and their range-dependent sigmas (the
    // same for every filter: evaluated once here, on the clean poses)
    if ((n->edge_loss || n->range_ref > 0) && M > 0) {
        std::vector<double> pose((size_t)M * 7);
        if (s->on_device)
            CUDA_TRY(cudaMemcpy(pose.data(), s->tag_pose_clean, pose.size() * 8, cudaMemcpyDeviceToHost));
        else
            std::memcpy(pose.data(), s->tag_pose_clean, pose.size() * 8);
        std::vector<double> sig((size_t)M * 2);
        std::vector<uint8_t> mask((size_t)M, 1);
        range_sigmas(pose.data(), M, to_device_noise(*n), sig.data());
        if (n->edge_loss) visibility_mask(pose.data(), M, make_consts<double>(h->p), mask.data());
        const size_t need = (size_t)M * 16 + (size_t)M;
        if (need > h->d_mask_bytes) {
            CUDA_TRY(cudaStreamSynchronize(h->stream));
            cudaFree(h->d_mask);
            h->d_mask = nullptr; h->d_mask_bytes = 0;
            CUDA_TRY(cudaMalloc(&h->d_mask, need));
            h->d_mask_bytes = need;
        }
        CUDA_TRY(cudaStreamSynchronize(h->stream));      // the previous launch may still read these
        CUDA_TRY(cudaMemcpy(h->d_mask, sig.data(), (size_t)M * 16, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(h->d_mask + (size_t)M * 16, mask.data(), (size_t)M, cudaMemcpyHostToDevice));
        in->tag_sigma = (const double *)h->d_mask;
        if (n->edge_loss) in->tag_valid = h->d_mask + (size_t)M * 16;
    }
    if (s->on_device) {
        in->imu = s->imu_clean; in->tag_step = s->tag_step; in->tag_pose = s->tag_pose_clean;
        in->tag_stamp = s->tag_stamp; *truth = s->truth;
        return QEKF_OK;
    }
    const size_t imu_b = (size_t)T * 6 * 8, pose_b = (size_t)M * 7 * 8, stamp_b = (size_t)M * 8, step_b = (size_t)M * 4;
    const size_t truth_b = s->truth ? (size_t)(T + 1) * 10 * 8 : 0;
    const size_t o_imu = 0, o_pose = align_up(o_imu + imu_b, 256), o_stamp = align_up(o_pose + pose_b, 256);
    const size_t o_step = align_up(o_stamp + stamp_b, 256), o_truth = align_up(o_step + step_b, 256);
    const size_t total = align_up(o_truth + truth_b, 256);
    if (total > h->d_shared_bytes) {
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        cudaFree(h->d_shared);
        h->d_shared = nullptr; h->d_shared_bytes = 0;
        CUDA_TRY(cudaMalloc(&h->d_shared, total));
        h->d_shared_bytes = total;
    }
    char *d = (char *)h->d_shared;
    CUDA_TRY(cudaMemcpyAsync(d + o_imu, s->imu_clean, imu_b, cudaMemcpyHostToDevice, h->stream));
    if (M > 0) {
        CUDA_TRY(cudaMemcpyAsync(d + o_pose, s->tag_pose_clean, pose_b, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(cudaMemcpyAsync(d + o_stamp, s->tag_stamp, stamp_b, cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(cudaMemcpyAsync(d + o_step, s->tag_step, step_b, cudaMemcpyHostToDevice, h->stream));
    }
    if (truth_b) CUDA_TRY(cudaMemcpyAsync(d + o_truth, s->truth, truth_b, cudaMemcpyHostToDevice, h->stream));
    in->imu = (const double *)(d + o_imu); in->tag_pose = (const double *)(d + o_pose);
    in->tag_stamp = (const double *)(d + o_stamp); in->tag_step = (const int32_t *)(d + o_step);
    *truth = truth_b ? (const double *)(d + o_truth) : nullptr;
    return QEKF_OK;
}

int qekf_run_monte_carlo(qekf_handle *h, const qekf_shared_streams *s, const qekf_noise_spec *n, int64_t k0,
                         int64_t n_steps)
{
    if (!h || !s || !n) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (n_steps == 0) return QEKF_OK;
    if (k0 < 0 || n_steps < 0 || k0 + n_steps > s->T) return fail(QEKF_ERR_BAD_ARG, "tick range outside the stream");
    if (k0 + n_steps > 2147483647LL) return fail(QEKF_ERR_BAD_ARG, "tick indices are limited to 31 bits (as tag_step is)");
    CUDA_TRY(cudaSetDevice(h->device));
    StreamView in;
    const double *truth = nullptr;
    std::vector<int32_t> steps;
    int rc = shared_view(h, s, n, &in, &truth, &steps);
    if (rc) return rc;
    int32_t m0 = 0;
    for (size_t m = 0; m < steps.size(); ++m)
        if (steps[m] < k0) m0 = (int32_t)(m + 1);
    NoiseSpec ns = to_device_noise(*n);
    rc = ensure_perm(h, ns);
    if (rc) return rc;
    // Long replays of the thread-per-filter kernels run on reordered arrays (filters that share a CTA share the phase of
    // their private dropout); a short one (a trace chunk, a test) would not repay the two reordering passes
    const bool tpf = h->lanes_per_filter == 1 || h->precision != QEKF_FP64 || h->p.multirate_ekf;
    const bool reorder = h->d_perm && tpf && n_steps >= h->perm_min_steps;
    if (reorder) {
        rc = permute_state(h, true);
        if (rc) return rc;
    }
    // delayed fusion: may this launch re-synthesise the history entries it finds (see qekf_handle::hist_clean)?
    uint64_t key[6] = { 0, 0, 0, 0, 0, 0 };
    bool regenerable = false;
    if (h->p.multirate_ekf) {
        key[0] = ns.seed; key[1] = (uint64_t)ns.gid0;
        std::memcpy(&key[2], &ns.sig_a, 8);                 // sig_a, sig_w
        std::memcpy(&key[3], &ns.sig_ba, 8);                // sig_ba, sig_bw
        key[4] = s->on_device ? (uint64_t)(uintptr_t)s->imu_clean : fnv1a(s->imu_clean, (size_t)s->T * 6 * 8);
        key[5] = (uint64_t)s->T ^ ((uint64_t)s->on_device << 62);
        regenerable = h->hist_clean || (h->hist_key_valid && std::memcmp(key, h->hist_key, sizeof key) == 0 && k0 == h->hist_k_next);
    }
    h->lazy_now = regenerable && h->lazy_mr_on;
    rc = run_dispatch(h, in, k0, n_steps, m0, &ns, truth);
    h->lazy_now = false;
    if (h->p.multirate_ekf) {
        // (either kernel leaves entries that are this noise model's samples of this scenario -- if the ones it found were)
        h->hist_clean = false;
        h->hist_key_valid = regenerable && rc == QEKF_OK;
        std::memcpy(h->hist_key, key, sizeof key);
        h->hist_k_next = k0 + n_steps;
    }
    if (reorder) {
        const int rc2 = permute_state(h, false);
        if (!rc) rc = rc2;
    }
    return rc;
}

int qekf_synthesize_streams(qekf_handle *h, const qekf_shared_streams *s, const qekf_noise_spec *n, int64_t first,
                            int64_t count, double *imu, double *tag_pose, uint8_t *tag_valid, double *bias)
{
    if (!h || !s || !n || !imu || !bias) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (first < 0 || count <= 0) return fail(QEKF_ERR_BAD_ARG, "bad filter range");
    if (s->M > 0 && (!tag_pose || !tag_valid)) return fail(QEKF_ERR_BAD_ARG, "NULL tag outputs");
    CUDA_TRY(cudaSetDevice(h->device));
    StreamView in;
    const double *truth = nullptr;
    std::vector<int32_t> steps;
    int rc = shared_view(h, s, n, &in, &truth, &steps);
    if (rc) return rc;
    const size_t imu_b = (size_t)s->T * 6 * (size_t)count * 8, tag_b = (size_t)s->M * 7 * (size_t)count * 8;
    const size_t val_b = (size_t)s->M * (size_t)count, bias_b = 6 * (size_t)count * 8;
    const size_t o_tag = align_up(imu_b, 256), o_val = align_up(o_tag + tag_b, 256), o_bias = align_up(o_val + val_b, 256);
    rc = ensure_in(h, align_up(o_bias + bias_b, 256));
    if (rc) return rc;
    char *d = (char *)h->d_in;
    RunArgs<double> a;
    std::memset(&a, 0, sizeof a);
    a.in = in;
    a.c = make_consts<double>(h->p);
    a.ns = to_device_noise(*n);
    CUDA_TRY(launch_dump<double>(a, first, count, s->T, (double *)d, (double *)(d + o_tag), (uint8_t *)(d + o_val),
                                 (double *)(d + o_bias), h->stream));
    h->launches++;
    CUDA_TRY(cudaMemcpyAsync(imu, d, imu_b, cudaMemcpyDeviceToHost, h->stream));
    if (s->M > 0) {
        CUDA_TRY(cudaMemcpyAsync(tag_pose, d + o_tag, tag_b, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaMemcpyAsync(tag_valid, d + o_val, val_b, cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(cudaMemcpyAsync(bias, d + o_bias, bias_b, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return QEKF_OK;
}

int qekf_stats_configure(qekf_handle *h, int32_t n_bins, int32_t stride)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    if (n_bins <= 0 || stride <= 0) return fail(QEKF_ERR_BAD_ARG, "n_bins and stride must be positive");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(h->stats_acc); cudaFree(h->stats_red);
    h->stats_acc = h->stats_red = nullptr;
    CUDA_TRY(cudaMalloc(&h->stats_acc, (size_t)STAT_REPL * n_bins * STAT_DIM * 8));
    CUDA_TRY(cudaMalloc(&h->stats_red, (size_t)n_bins * STAT_DIM * 8));
    h->stats_bins = n_bins; h->stats_stride = stride;
    return qekf_stats_reset(h);
}

int qekf_stats_config(const qekf_handle *h, int32_t *n_bins, int32_t *stride)
{
    if (!h || !n_bins || !stride) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    *n_bins = h->stats_acc ? h->stats_bins : 0;
    *stride = h->stats_acc ? h->stats_stride : 0;
    return QEKF_OK;
}

int qekf_stats_reset(qekf_handle *h)
{
    if (!h || !h->stats_acc) return fail(QEKF_ERR_NOT_INITIALIZED, "statistics are not configured");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaMemsetAsync(h->stats_acc, 0, (size_t)STAT_REPL * h->stats_bins * STAT_DIM * 8, h->stream));
    return QEKF_OK;
}

int qekf_copy_stats_device(qekf_handle *h, void *dst_device)
{
    if (!h || !h->stats_acc) return fail(QEKF_ERR_NOT_INITIALIZED, "statistics are not configured");
    if (!dst_device) return fail(QEKF_ERR_BAD_ARG, "destination is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(launch_stats_reduce(h->stats_acc, h->stats_red, h->stats_bins, h->stream));
    h->launches++;
    CUDA_TRY(cudaMemcpyAsync(dst_device, h->stats_red, (size_t)h->stats_bins * STAT_DIM * 8, cudaMemcpyDeviceToDevice, h->stream));
    return QEKF_OK;
}

int qekf_get_stats(qekf_handle *h, double *out)
{
    if (!h || !h->stats_acc) return fail(QEKF_ERR_NOT_INITIALIZED, "statistics are not configured");
    if (!out) return fail(QEKF_ERR_BAD_ARG, "output is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(launch_stats_reduce(h->stats_acc, h->stats_red, h->stats_bins, h->stream));
    h->launches++;
    CUDA_TRY(cudaMemcpyAsync(out, h->stats_red, (size_t)h->stats_bins * STAT_DIM * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return QEKF_OK;
}

// ---- housekeeping ----------------------------------------------------------------------------------------

int qekf_reset_filters(qekf_handle *h)
{
    if (!h) return fail(QEKF_ERR_BAD_ARG, "handle is NULL");
    CUDA_TRY(cudaSetDevice(h->device));
    const size_t ld = (size_t)h->ld;
    CUDA_TRY(cudaMemsetAsync(h->x, 0, 16 * ld * h->tsize, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->aux, 0, AUX_DIM * ld * h->tsize, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->pend, 0, PEND_DIM * ld * sizeof(double), h->stream));
    CUDA_TRY(cudaMemsetAsync(h->flags, 0, ld * sizeof(int32_t), h->stream));
    CUDA_TRY(cudaMemsetAsync(h->upds, 0, ld * sizeof(int32_t), h->stream));
    if (h->xc) {
        CUDA_TRY(cudaMemsetAsync(h->xc, 0, 16 * ld * h->tsize, h->stream));
        CUDA_TRY(cudaMemsetAsync(h->nh, 0, ld * sizeof(int32_t), h->stream));
        CUDA_TRY(cudaMemsetAsync(h->hpos, 0, ld * sizeof(int32_t), h->stream));
        CUDA_TRY(cudaMemsetAsync(h->hlen, 0, ld * sizeof(int32_t), h->stream));
    }
    hist_emptied(h);
    return reset_cov(h, true);
}

int64_t qekf_launch_count(const qekf_handle *h) { return h ? h->launches : 0; }

int qekf_step_counts(qekf_handle *h, int64_t *n_predict, int64_t *n_correct, int reset)
{
    if (!h || !n_predict || !n_correct) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    unsigned long long c[8];
    CUDA_TRY(cudaMemcpy(c, h->counts, sizeof c, cudaMemcpyDeviceToHost));
    *n_predict = (int64_t)c[0]; *n_correct = (int64_t)c[1];
    if (getenv("QEKF_DIAG"))
        fprintf(stderr, "[qekf diag] predicts %llu corrects %llu | warp iterations %llu, with a correction %llu | stat samples %llu\n", c[0], c[1], c[2], c[3], c[4]);
    if (reset) CUDA_TRY(cudaMemset(h->counts, 0, sizeof c));
    return QEKF_OK;
}

int qekf_measure_fma_peak(int device, int precision, double *tflops)
{
    if (!tflops) return fail(QEKF_ERR_BAD_ARG, "output is NULL");
    if (precision != QEKF_FP64 && precision != QEKF_FP32) return fail(QEKF_ERR_BAD_ARG, "precision must be 64 or 32");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return fail(QEKF_ERR_NO_DEVICE, "no such CUDA device");
    }
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    void *sink = nullptr;
    CUDA_TRY(cudaMalloc(&sink, 64));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const unsigned block = 256, grid = (unsigned)prop.multiProcessorCount * 8;
    const int iters = (precision == QEKF_FP64) ? 8192 : 32768;
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        CUDA_TRY(cudaEventRecord(e0, 0));
        if (precision == QEKF_FP64) CUDA_TRY(launch_fma_peak<double>((double *)sink, iters, grid, block, 0));
        else CUDA_TRY(launch_fma_peak<float>((float *)sink, iters, grid, block, 0));
        CUDA_TRY(cudaEventRecord(e1, 0));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 16.0 * (double)iters * (double)block * (double)grid;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    *tflops = best;
    return QEKF_OK;
}

// ---- synthetic scenario (host) -----------------------------------------------------------------------

int qekf_scenario_default(qekf_scenario_spec *s)
{
    if (!s) return fail(QEKF_ERR_BAD_ARG, "spec is NULL");
    qekf::scenario::defaults(s);
    return QEKF_OK;
}

int qekf_scenario_sizes(const qekf_params *p, const qekf_scenario_spec *s, int64_t *T, int64_t *M)
{
    if (!p || !s || !T || !M) return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (!(p->update_freq > 0) || !(s->tag_rate_hz > 0) || s->tag_rate_hz > p->update_freq)
        return fail(QEKF_ERR_BAD_ARG, "need 0 < tag_rate_hz <= update_freq");
    qekf::scenario::sizes(*p, *s, T, M);
    return QEKF_OK;
}

int qekf_scenario_generate(const qekf_params *p, const qekf_scenario_spec *s, double *truth, double *imu_clean,
                           int32_t *tag_step, double *tag_pose_clean, double *tag_stamp)
{
    if (!p || !s || !truth || !imu_clean || !tag_step || !tag_pose_clean || !tag_stamp)
        return fail(QEKF_ERR_BAD_ARG, "NULL argument");
    if (!(p->update_freq > 0) || !(s->tag_rate_hz > 0) || s->tag_rate_hz > p->update_freq)
        return fail(QEKF_ERR_BAD_ARG, "need 0 < tag_rate_hz <= update_freq");
    qekf::scenario::generate(*p, *s, truth, imu_clean, tag_step, tag_pose_clean, tag_stamp);
    return QEKF_OK;
}

}  // extern "C"
