// ekf_synth.cuh -- Monte-Carlo machinery the reference does not have (it runs one filter on live
// sensors): counter-based per-filter noise realisations generated in-kernel, and on-chip accumulation
// of RMSE / NEES statistics against the scenario truth.
//
// Noise: Philox4x32-10, key = 64-bit seed, counter = (index, stream tag, global filter id lo, hi), so a
// realisation depends only on (seed, global filter id, tick/arrival index) -- never on the launch
// geometry, the time chunking or the number of GPUs.  One block gives six 21-bit uniforms; normals by Box-Muller in
// FP32 (the FP32/SFU pipes are idle while the FP64 pipe does the filter arithmetic), widened to the filter's real type.
//
// Measurement noise is applied in the camera frame, which is where the filter's R_k = N R N^T places it
// (relative_pose_EKF.cpp:462-472):  r_c += n_p,  q_ct <- exp(n_th) (x) q_ct.
#pragma once

#include <cmath>

#include "ekf_core.cuh"

namespace qekf {

struct NoiseSpec {
    uint64_t seed;
    int64_t gid0;                 // global id of the handle's filter 0 (multi-GPU shards share one id space)
    float sig_a, sig_w;           // IMU white noise (m/s^2, rad/s) per sample
    float sig_ba, sig_bw;         // constant true bias drawn per filter
    float sig_p, sig_th;          // tag position (m) and attitude (rad) noise
    int32_t drop_k0, drop_k1;     // common dropout: arrivals with k0 <= tag_step < k1 are lost
    int32_t rdrop_len, rdrop_lo, rdrop_hi;   // per-filter dropout of rdrop_len ticks starting in [lo, hi)
    int32_t edge_loss;            // detection front-end: lose arrivals whose bundle is not entirely in the image
    double range_ref, range_exp_p, range_exp_th;   // range_ref > 0: sigma * (|r_c| / range_ref)^exp
};

enum : uint32_t { STREAM_IMU = 0, STREAM_TAG = 2, STREAM_BIAS = 4, STREAM_DROPOUT = 6 };

QEKF_FN uint32_t mulhi32(uint32_t a, uint32_t b)
{
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

QEKF_FN void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// six 21-bit integers from the 128 bits of one Philox block (126 of them used)
QEKF_FN void uniforms21x6(const uint32_t w[4], uint32_t u[6])
{
    u[0] = w[0] & 0x1FFFFFu;
    u[1] = (w[0] >> 21) | ((w[1] & 0x3FFu) << 11);
    u[2] = (w[1] >> 10) & 0x1FFFFFu;
    u[3] = (w[1] >> 31) | ((w[2] & 0xFFFFFu) << 1);
    u[4] = (w[2] >> 20) | ((w[3] & 0x1FFu) << 12);
    u[5] = (w[3] >> 9) & 0x1FFFFFu;
}

// two standard normals from two 21-bit integers (Box-Muller, FP32): u = (a + 1/2) / 2^21 lies strictly inside (0, 1)
// and is exact in float; the largest |z| is sqrt(-2 ln 2^-22) = 5.5
QEKF_FN void box_muller(uint32_t a, uint32_t b, float &z0, float &z1)
{
    const float u1 = ((float)a + 0.5f) * (1.0f / 2097152.0f);
    const float u2 = ((float)b + 0.5f) * (1.0f / 2097152.0f);
    float s, c;
#ifdef __CUDA_ARCH__
    // r = sqrt(-2 ln u1) from the SFU (lg2.approx, sqrt.approx) instead of logf + sqrtf (41 -> ~15 instructions per pair,
    // the largest non-FP64 item of the tick).  lg2.approx is accurate to 2^-22 relative, or absolute on (0.5, 2); what
    // matters is dr = d(ln u1) / r, so for u1 > 15/16, where r gets small, -ln u1 comes from its series in t = 1 - u1
    // (exact in float; remainder t^6 / 6 <= 1.6e-7 relative).  r is then within ~1e-6 of the libm value everywhere.
    const float t = 1.0f - u1;
    const float ser = t * fmaf(t, fmaf(t, fmaf(t, fmaf(t, 0.2f, 0.25f), 0.33333334f), 0.5f), 1.0f);
    const float nl = (t < 0.0625f) ? ser : -0.69314718f * __log2f(u1);
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(2.0f * nl));
    // the SFU's sin / cos (absolute error < 7e-7 on [0, 2 pi): a relative 7e-7 of a noise sample) instead of sincospif's
    // range reduction and two polynomials: 6 instructions per pair instead of 35, on the per-tick path of every filter
    s = __sinf(6.2831853071795865f * u2);
    c = __cosf(6.2831853071795865f * u2);
#else
    const float r = sqrtf(-2.0f * logf(u1));
    s = (float)::sin(6.283185307179586 * (double)u2);
    c = (float)::cos(6.283185307179586 * (double)u2);
#endif
    z0 = r * c;
    z1 = r * s;
}

// six standard normals for (seed, global filter id, stream, index): ONE Philox block (two until late in round 2: the
// second block was 7 % of a tick's instructions for two of its four words)
QEKF_FN void normals6(uint64_t seed, int64_t gid, uint32_t stream, uint32_t index, float z[6])
{
    uint32_t w[4], u[6];
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t g0 = (uint32_t)(uint64_t)gid, g1 = (uint32_t)((uint64_t)gid >> 32);
    philox4x32_10(index, stream, g0, g1, k0, k1, w);
    uniforms21x6(w, u);
    box_muller(u[0], u[1], z[0], z[1]);
    box_muller(u[2], u[3], z[2], z[3]);
    box_muller(u[4], u[5], z[4], z[5]);
}
QEKF_FN void normals6(const NoiseSpec &ns, int64_t gid, uint32_t stream, uint32_t index, float z[6])
{
    normals6(ns.seed, gid, stream, index, z);
}

// the constant true IMU bias of a filter
QEKF_FN void true_bias(const NoiseSpec &ns, int64_t gid, double b[6])
{
    float z[6];
    normals6(ns, gid, STREAM_BIAS, 0u, z);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        b[i] = (double)ns.sig_ba * (double)z[i];
        b[3 + i] = (double)ns.sig_bw * (double)z[3 + i];
    }
}

// first tick of the filter's private dropout window (or INT32_MAX when disabled)
QEKF_FN int32_t private_dropout_start(const NoiseSpec &ns, int64_t gid)
{
    if (ns.rdrop_len <= 0 || ns.rdrop_hi <= ns.rdrop_lo) return INT32_MAX;
    uint32_t w[4];
    philox4x32_10(0u, STREAM_DROPOUT, (uint32_t)(uint64_t)gid, (uint32_t)((uint64_t)gid >> 32), (uint32_t)ns.seed,
                  (uint32_t)(ns.seed >> 32), w);
    const uint32_t span = (uint32_t)(ns.rdrop_hi - ns.rdrop_lo);
    return ns.rdrop_lo + (int32_t)mulhi32(w[0], span);
}

QEKF_FN bool arrival_valid(const NoiseSpec &ns, int32_t step, int32_t priv_start)
{
    if (step >= ns.drop_k0 && step < ns.drop_k1) return false;
    if (priv_start != INT32_MAX && step >= priv_start && step < priv_start + ns.rdrop_len) return false;
    return true;
}

// noisy IMU sample of tick k:  clean + bias + sigma * n          (doubles; the caller narrows)
// (the scalars of the noise model an IMU sample depends on; small enough to travel through a call in registers)
struct ImuSynth {
    uint64_t seed;
    float sig_a, sig_w, sig_ba, sig_bw;
};
QEKF_FN void synth_imu(const ImuSynth &nz, int64_t gid, int64_t k, const double clean[6], const double bias[6], double u[6])
{
    float z[6];
    normals6(nz.seed, gid, STREAM_IMU, (uint32_t)k, z);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        u[i] = clean[i] + bias[i] + (double)nz.sig_a * (double)z[i];
        u[3 + i] = clean[3 + i] + bias[3 + i] + (double)nz.sig_w * (double)z[3 + i];
    }
}
QEKF_FN void synth_imu(const NoiseSpec &ns, int64_t gid, int64_t k, const double clean[6], const double bias[6], double u[6])
{
    const ImuSynth nz{ ns.seed, ns.sig_a, ns.sig_w, ns.sig_ba, ns.sig_bw };
    synth_imu(nz, gid, k, clean, bias, u);
}

// Detection front-end, geometry: does at least one tag of the bundle project with all four corners strictly inside
// the image?  Same corner construction and pinhole projection as the reference's corner-margin gate
// (relative_pose_EKF.cpp:156-181) at margin 0, evaluated in double on the CLEAN pose, so that the set of
// detections does not depend on the filter's arithmetic type or noise realisation.
template <typename T> QEKF_FN bool bundle_in_image(const double tag[7], const Consts<T> &c)
{
    double R[9];
    quat_to_rot<double>(tag + 3, R);
    for (int i = 0; i < c.n_tags; ++i) {
        const double hw = (double)c.tag_hw[i], px0 = (double)c.tag_px[i], py0 = (double)c.tag_py[i];
        bool all_in = true;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double cx = ((k == 0 || k == 3) ? hw : -hw) + px0;
            const double cy = ((k < 2) ? hw : -hw) + py0;
            const double p0 = R[0] * cx + R[1] * cy + tag[0];
            const double p1 = R[3] * cx + R[4] * cy + tag[1];
            const double p2 = R[6] * cx + R[7] * cy + tag[2];
            const double iz = 1.0 / p2;
            const double xn = p0 * iz, yn = p1 * iz;
            const double uu = (double)c.Kcam[0] * xn + (double)c.Kcam[1] * yn + (double)c.Kcam[2];
            const double vv = (double)c.Kcam[3] * xn + (double)c.Kcam[4] * yn + (double)c.Kcam[5];
            all_in = all_in && (p2 > 0.0) && (uu > 0.0) && (uu < (double)c.cam_w) && (vv > 0.0) && (vv < (double)c.cam_h);
        }
        if (all_in) return true;
    }
    return false;
}

// The front-end's visibility mask of a whole clean scenario (host): it depends on the clean poses and the camera /
// bundle geometry only, so it is evaluated once per launch and shared by all filters.
inline void visibility_mask(const double *tag_pose_clean, int64_t M, const Consts<double> &c, uint8_t *out)
{
    for (int64_t m = 0; m < M; ++m) out[m] = bundle_in_image<double>(tag_pose_clean + m * 7, c) ? 1 : 0;
}

// The front-end's range-dependent tag noise (host): sigma_p, sigma_th of every arrival, [M][2].  Like the
// visibility mask it depends on the clean poses only and is shared by all filters.
inline void range_sigmas(const double *tag_pose_clean, int64_t M, const NoiseSpec &ns, double *out)
{
    for (int64_t m = 0; m < M; ++m) {
        const double *c = tag_pose_clean + m * 7;
        double sp = (double)ns.sig_p, sth = (double)ns.sig_th;
        if (ns.range_ref > 0.0) {
            const double rel = std::sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]) / ns.range_ref;
            if (ns.range_exp_p != 0.0) sp *= std::pow(rel, ns.range_exp_p);
            if (ns.range_exp_th != 0.0) sth *= std::pow(rel, ns.range_exp_th);
        }
        out[2 * m] = sp;
        out[2 * m + 1] = sth;
    }
}

// noisy tag pose of arrival m:  r_c + sigma_p n,  exp(sigma_th n) (x) q_ct   (sp, sth: this arrival's sigmas)
QEKF_FN void synth_tag(const NoiseSpec &ns, int64_t gid, int32_t m, const double clean[7], double tag[7], double sp,
                       double sth)
{
    float z[6];
    normals6(ns, gid, STREAM_TAG, (uint32_t)m, z);
#pragma unroll
    for (int i = 0; i < 3; ++i) tag[i] = clean[i] + sp * (double)z[i];
    double v[3] = { sth * (double)z[3], sth * (double)z[4], sth * (double)z[5] };
    double n2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    double n = sqrt(n2);
    double f = (n < 1e-10) ? 0.5 : sin(0.5 * n) / n;
    double dq[4] = { v[0] * f, v[1] * f, v[2] * f, cos(0.5 * n) };
    quat_mul<double>(dq, clean + 3, tag + 3);
}

// ------------------------------------------------------------------------------------------------
// statistics
// ------------------------------------------------------------------------------------------------
constexpr int STAT_DIM = 20;      // 0..14 sum e_i^2 | 15 sum NEES | 16 samples | 17 NEES inside the two-sided
                                  // 95% chi-square interval | 18 diverged (non-finite or P not SPD) | 19 sum |e_r|^2
constexpr int STAT_REPL = 32;     // replicas of the accumulator (spreads atomic contention), summed on read

struct StatsView {
    double *acc;                  // [STAT_REPL][n_bins][STAT_DIM]
    const double *truth;          // Monte-Carlo launches: [T+1][10] r v q_tv shared by all filters; state after tick k is truth[k+1]
    // explicit-stream launches: each filter's own truth, element (bin b, component c) of filter row i at
    // truth_pf[(b*16 + c)*ld_t + i], components r v q_tv ab wb (the state after the sampling tick of bin b)
    const double *truth_pf;
    int64_t ld_t;
    int32_t n_bins;
    int32_t stride;               // sample after tick k when (k+1) % stride == 0
    double chi2_lo, chi2_hi;
};

// Cholesky U^T U of a packed upper triangle held in registers (sym_idx<NN>), in place, with one right-hand side
// carried along: on return rhs = U^-T rhs and dinv[j] = 1 / U_jj.  All loops unrolled, all indices compile-time.
template <typename T, int NN> QEKF_FN bool chol_packed(T *A, T *rhs, T *dinv)
{
    bool ok = true;
#pragma unroll
    for (int j = 0; j < NN; ++j) {
        T d = A[sym_idx<NN>(j, j)];
        T yj = rhs[j];
#pragma unroll
        for (int k = 0; k < j; ++k) {
            d = M<T>::fma_(-A[sym_idx<NN>(k, j)], A[sym_idx<NN>(k, j)], d);
            yj = M<T>::fma_(-A[sym_idx<NN>(k, j)], rhs[k], yj);
        }
        ok = ok && (d > T(0));
        const T inv = M<T>::rsqrt_(ok ? d : T(1));
        dinv[j] = inv;
        A[sym_idx<NN>(j, j)] = d * inv;
        rhs[j] = yj * inv;
#pragma unroll
        for (int i = j + 1; i < NN; ++i) {
            T v = A[sym_idx<NN>(j, i)];
#pragma unroll
            for (int k = 0; k < j; ++k) v = M<T>::fma_(-A[sym_idx<NN>(k, j)], A[sym_idx<NN>(k, i)], v);
            A[sym_idx<NN>(j, i)] = v * inv;
        }
    }
    return ok;
}

// NEES = e^T P^-1 e WITHOUT touching P (round 2; the in-place factorisation it replaces had to park the covariance in HBM
// and read it back: 60 x 0.96 GB of dirty lines per benchmark launch, 14 GB of DRAM writes against 1.1 GB algorithmic).
// Block elimination in registers: the leading K x K block (K = 6, or 3 for the 9-state filter) is factored,
// W = U11^-T P12 and the Schur complement S = P22 - W^T W are formed from P read in place, S is factored;
// NEES = |U11^-T e1|^2 + |U22^-T (e2 - W^T y1)|^2.  Returns false when a pivot is not positive (P not SPD).
template <typename T, class PS> QEKF_FN bool nees_readonly(const PS &P, const T *e, T &nees)
{
    constexpr int N = PS::n;
    constexpr int K = (N == 15) ? 6 : 3;
    constexpr int R = N - K;
    T A[K * (K + 1) / 2], y1[K], dinv1[K];
#pragma unroll
    for (int i = 0; i < K; ++i) {
        y1[i] = e[i];
#pragma unroll
        for (int j = i; j < K; ++j) A[sym_idx<K>(i, j)] = P.ld(i, j);
    }
    bool ok = chol_packed<T, K>(A, y1, dinv1);
    T W[R * K], e2[R];
#pragma unroll
    for (int c = 0; c < R; ++c) {
        T ec = e[K + c];
#pragma unroll
        for (int j = 0; j < K; ++j) {                 // w = U11^-T P[0:K, K+c]
            T v = P.ld(j, K + c);
#pragma unroll
            for (int k = 0; k < j; ++k) v = M<T>::fma_(-A[sym_idx<K>(k, j)], W[c * K + k], v);
            v *= dinv1[j];
            W[c * K + j] = v;
            ec = M<T>::fma_(-v, y1[j], ec);
        }
        e2[c] = ec;
    }
    T S[R * (R + 1) / 2], dinv2[R];
#pragma unroll
    for (int c = 0; c < R; ++c)
#pragma unroll
        for (int d = c; d < R; ++d) {
            T v = P.ld(K + c, K + d);
#pragma unroll
            for (int k = 0; k < K; ++k) v = M<T>::fma_(-W[c * K + k], W[d * K + k], v);
            S[sym_idx<R>(c, d)] = v;
        }
    ok = chol_packed<T, R>(S, e2, dinv2) && ok;
    nees = T(0);
#pragma unroll
    for (int i = 0; i < K; ++i) nees = M<T>::fma_(y1[i], y1[i], nees);
#pragma unroll
    for (int i = 0; i < R; ++i) nees = M<T>::fma_(e2[i], e2[i], nees);
    return ok;
}

}  // namespace qekf
