// ekf_core.cuh -- per-filter arithmetic of the relative-pose error-state EKF, written for one CUDA
// thread per filter on sm_100a.  Templated on the real type (double = reference arithmetic,
// float = FP32 mode), on est_bias (15 vs 9 error states) and on the measurement model.
//
// What is computed follows the reference (quad_state_estimation/src/relative_pose_EKF.cpp and
// src/quaternion_helper.cpp; line numbers cited per function).  How it is computed does not: the
// reference forms dense 15x15 Jacobians and multiplies them out; here the block structure of F, W, G
// is used directly, the covariance is kept as a packed symmetric upper triangle, and the update never
// materialises K (15x6) or I-KG.  Results agree with the dense formulas to rounding (~1e-15).
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#define QEKF_FN __host__ __device__ __forceinline__

namespace qekf {

// ------------------------------------------------------------------------------------------------
// scalar math wrappers
// ------------------------------------------------------------------------------------------------
template <typename T> struct M;
template <> struct M<double> {
    static QEKF_FN double sqrt_(double x) { return sqrt(x); }
#ifdef __CUDA_ARCH__
    static QEKF_FN double rsqrt_(double x) { return rsqrt(x); }
    static QEKF_FN void sincos_(double x, double *s, double *c) { sincos(x, s, c); }
#else   // host instantiation exists only for the CPU-side unit tests of this header (tests/host_core)
    static QEKF_FN double rsqrt_(double x) { return 1.0 / ::sqrt(x); }
    static QEKF_FN void sincos_(double x, double *s, double *c) { *s = ::sin(x); *c = ::cos(x); }
#endif
    static QEKF_FN double atan2_(double y, double x) { return atan2(y, x); }
    static QEKF_FN double fma_(double a, double b, double c) { return fma(a, b, c); }
    static QEKF_FN double abs_(double x) { return fabs(x); }
    static QEKF_FN double min_(double a, double b) { return fmin(a, b); }
};
template <> struct M<float> {
    static QEKF_FN float sqrt_(float x) { return sqrtf(x); }
#ifdef __CUDA_ARCH__
    static QEKF_FN float rsqrt_(float x) { return rsqrtf(x); }
    static QEKF_FN void sincos_(float x, float *s, float *c) { sincosf(x, s, c); }
#else
    static QEKF_FN float rsqrt_(float x) { return 1.0f / ::sqrtf(x); }
    static QEKF_FN void sincos_(float x, float *s, float *c) { *s = ::sinf(x); *c = ::cosf(x); }
#endif
    static QEKF_FN float atan2_(float y, float x) { return atan2f(y, x); }
    static QEKF_FN float fma_(float a, float b, float c) { return fmaf(a, b, c); }
    static QEKF_FN float abs_(float x) { return fabsf(x); }
    static QEKF_FN float min_(float a, float b) { return fminf(a, b); }
};

// Which covariance update correction_step uses.  The reference computes P^ = (I - K G) P (relative_pose_EKF.cpp:480)
// and the FP64 path evaluates exactly that.  The FP32 mode uses the Joseph form
//     P^ = (I - K G) P (I - K G)^T + K R_k K^T = P - K B^T - D K^T,      B = P G^T,  D = B - K S  (the gain's residual).
// With K = B S^-1 the last term is D S^-1 B^T, so the form is evaluated block by block as P - K' B^T with the
// refined gain K' = K + D S^-1: if the computed S^-1 is off by a relative E, K is off by E but K' only by E^2 --
// the property the Joseph form is used for (first-order errors of the gain do not reach the covariance).
template <typename T> struct UpdateForm { static constexpr bool joseph = false; };
#ifndef QEKF_NO_JOSEPH      // (defined only by tests/test_core_host.py to measure what the form buys)
template <> struct UpdateForm<float> { static constexpr bool joseph = true; };
#endif

// Block indices of the error state: (dr, dv, dtheta, dab, dwb), relative_pose_EKF.cpp:484-485.
enum { BR = 0, BV = 1, BTH = 2, BAB = 3, BWB = 4 };

// ------------------------------------------------------------------------------------------------
// parameters shared by all filters of a launch (kernel-parameter / constant-bank resident)
// ------------------------------------------------------------------------------------------------
template <typename T> struct Consts {
    T dT;                 // dT_nom = 1/update_freq                       (cpp:90)
    T g[3];               //                                              (cpp:81)
    T ab_static[3], wb_static[3];
    T Q[12];              // diag: Q_a, Q_w, Q_ab, Q_wb (per step)        (cpp:96-112)
    T Rr[3], Ra[3];       // diag of R                                    (cpp:116-118)
    T RC[6];              // sym C_vc diag(R_r) C_vc^T   (derived, host)
    T RA[6];              // sym C_vc diag(R_ang) C_vc^T (derived, host)
    T D[9];               // diag(R_ang) C_vc^T          (derived, host)
    T C_vc[9];            // R(q_vc), row-major                           (cpp:121-122)
    T r_v_cv[3];
    T q_vc[4];            // normalised + clipped, xyzw                   (cpp:121)
    T cov_init[5];        // r, v, ang, ab, wb                            (cpp:102-113)
    // camera and bundle geometry in double whatever T: the corner-margin gate is evaluated in double (corner_gate)
    double Kcam[6];       // camera_K rows 0 and 1
    double u_lo, u_hi, v_lo, v_hi; // width*margin, width*(1-margin), height*margin, height*(1-margin)  (cpp:176-179)
    double cam_w, cam_h;      // camera_width, camera_height
    double tag_hw[16];    // tag_widths/2
    double tag_px[16], tag_py[16];
    T small_ang_tol;
    double meas_delay, meas_delay_max, dyn_offset;   // seconds; the delay -> step rounding is done in double (cpp:199-200)
    double dT_nom;        // 1/update_freq in double, for the same reason
    int n_tags;
    int upd_per_meas;     // ceil(update_freq/measurement_freq)           (cpp:91)
    int limit_measurement_freq, corner_margin_enbl, dynamic_meas_delay;
};

// Nominal state of one filter: x = [r v q(xyzw) ab wb]  (relative_pose_EKF.cpp:244-245)
template <typename T> struct Nominal {
    T r[3], v[3], q[4], ab[3], wb[3];
};

// ------------------------------------------------------------------------------------------------
// parameter views.  The step functions read the parameters a sweep may override per filter (Q, R and the
// camera extrinsic, BASELINE config 5) through a view: ParU serves them from the launch-wide constant
// block, ParF from this filter's column of a [PF_DIM][ld] table in global memory (derived quantities
// included, so the kernel does no per-filter parameter derivation).  Everything else comes from view.c.
// ------------------------------------------------------------------------------------------------
enum { PF_Q = 0, PF_RA = 12, PF_RC = 15, PF_RAS = 21, PF_D = 27, PF_CVC = 36, PF_RVCV = 45, PF_QVC = 48, PF_DIM = 52 };

// per-filter parameter tables are never written by a kernel that reads them: non-coherent loads, which the compiler may
// hoist out of the replay loops and merge (a plain load through a generic pointer has to be re-issued after every store
// to the covariance, which it cannot prove to be shared memory)
template <typename T> QEKF_FN T ld_ro(const T *p)
{
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

template <typename T> struct ParU {
    const Consts<T> &c;
    QEKF_FN T Q(int i) const { return c.Q[i]; }
    QEKF_FN T Ra(int i) const { return c.Ra[i]; }
    QEKF_FN T RC(int i) const { return c.RC[i]; }
    QEKF_FN T RA(int i) const { return c.RA[i]; }
    QEKF_FN T D(int i) const { return c.D[i]; }
    QEKF_FN T C_vc(int i) const { return c.C_vc[i]; }
    QEKF_FN T r_v_cv(int i) const { return c.r_v_cv[i]; }
    QEKF_FN T q_vc(int i) const { return c.q_vc[i]; }
    QEKF_FN double meas_delay() const { return c.meas_delay; }
    QEKF_FN double dyn_offset() const { return c.dyn_offset; }
    // launch-wide scalars the step functions need
    QEKF_FN T dT() const { return c.dT; }
    QEKF_FN T g(int i) const { return c.g[i]; }
    QEKF_FN T ab_static(int i) const { return c.ab_static[i]; }
    QEKF_FN T wb_static(int i) const { return c.wb_static[i]; }
    QEKF_FN T small_ang_tol() const { return c.small_ang_tol; }
    QEKF_FN T cov_init(int i) const { return c.cov_init[i]; }
};
template <typename T> struct ParF {
    const Consts<T> &c;
    const T *t;          // this filter's column of the [PF_DIM][ld] table
    const double *dl;    // this filter's column of the [2][ld] delay table (measurement_delay, dyn offset)
    int64_t ld;
    QEKF_FN T Q(int i) const { return ld_ro(t + (PF_Q + i) * ld); }
    QEKF_FN T Ra(int i) const { return ld_ro(t + (PF_RA + i) * ld); }
    QEKF_FN T RC(int i) const { return ld_ro(t + (PF_RC + i) * ld); }
    QEKF_FN T RA(int i) const { return ld_ro(t + (PF_RAS + i) * ld); }
    QEKF_FN T D(int i) const { return ld_ro(t + (PF_D + i) * ld); }
    QEKF_FN T C_vc(int i) const { return ld_ro(t + (PF_CVC + i) * ld); }
    QEKF_FN T r_v_cv(int i) const { return ld_ro(t + (PF_RVCV + i) * ld); }
    QEKF_FN T q_vc(int i) const { return ld_ro(t + (PF_QVC + i) * ld); }
    QEKF_FN double meas_delay() const { return ld_ro(dl); }
    QEKF_FN double dyn_offset() const { return ld_ro(dl + ld); }
    QEKF_FN T dT() const { return c.dT; }
    QEKF_FN T g(int i) const { return c.g[i]; }
    QEKF_FN T ab_static(int i) const { return c.ab_static[i]; }
    QEKF_FN T wb_static(int i) const { return c.wb_static[i]; }
    QEKF_FN T small_ang_tol() const { return c.small_ang_tol; }
    QEKF_FN T cov_init(int i) const { return c.cov_init[i]; }
};

#ifdef __CUDACC__
// The same two views over a copy of the constant block in SHARED memory, for code behind a real call (advance_call,
// correction_call): a reference to the kernel parameters that crosses a call turns into generic loads from their
// global-memory image (L2 latency), a generic pointer to a shared copy into generic loads the compiler must treat as
// long-latency; an explicit ld.shared is a 29-cycle access it can schedule.  The asm statements are deliberately not
// volatile: the block never changes during a launch, so they may be hoisted, merged and dropped like any pure load.
template <typename T> __device__ __forceinline__ T lds_at(uint32_t addr);
template <> __device__ __forceinline__ double lds_at<double>(uint32_t addr)
{
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
template <> __device__ __forceinline__ float lds_at<float>(uint32_t addr)
{
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
#define QEKF_CS_OFF(member) ((uint32_t)__builtin_offsetof(Consts<T>, member))
template <typename T> struct ParUS {
    uint32_t base;       // shared-state-space address of the Consts<T> copy
    __device__ __forceinline__ T at(uint32_t off, int i) const { return lds_at<T>(base + off + (uint32_t)i * (uint32_t)sizeof(T)); }
    __device__ __forceinline__ T Q(int i) const { return at(QEKF_CS_OFF(Q), i); }
    __device__ __forceinline__ T Ra(int i) const { return at(QEKF_CS_OFF(Ra), i); }
    __device__ __forceinline__ T RC(int i) const { return at(QEKF_CS_OFF(RC), i); }
    __device__ __forceinline__ T RA(int i) const { return at(QEKF_CS_OFF(RA), i); }
    __device__ __forceinline__ T D(int i) const { return at(QEKF_CS_OFF(D), i); }
    __device__ __forceinline__ T C_vc(int i) const { return at(QEKF_CS_OFF(C_vc), i); }
    __device__ __forceinline__ T r_v_cv(int i) const { return at(QEKF_CS_OFF(r_v_cv), i); }
    __device__ __forceinline__ T q_vc(int i) const { return at(QEKF_CS_OFF(q_vc), i); }
    __device__ __forceinline__ double meas_delay() const { return lds_at<double>(base + QEKF_CS_OFF(meas_delay)); }
    __device__ __forceinline__ double dyn_offset() const { return lds_at<double>(base + QEKF_CS_OFF(dyn_offset)); }
    __device__ __forceinline__ T dT() const { return at(QEKF_CS_OFF(dT), 0); }
    __device__ __forceinline__ T g(int i) const { return at(QEKF_CS_OFF(g), i); }
    __device__ __forceinline__ T ab_static(int i) const { return at(QEKF_CS_OFF(ab_static), i); }
    __device__ __forceinline__ T wb_static(int i) const { return at(QEKF_CS_OFF(wb_static), i); }
    __device__ __forceinline__ T small_ang_tol() const { return at(QEKF_CS_OFF(small_ang_tol), 0); }
    __device__ __forceinline__ T cov_init(int i) const { return at(QEKF_CS_OFF(cov_init), i); }
};
template <typename T> struct ParFS {
    uint32_t base;
    const T *t;
    const double *dl;
    int64_t ld;
    __device__ __forceinline__ T at(uint32_t off, int i) const { return lds_at<T>(base + off + (uint32_t)i * (uint32_t)sizeof(T)); }
    __device__ __forceinline__ T Q(int i) const { return ld_ro(t + (PF_Q + i) * ld); }
    __device__ __forceinline__ T Ra(int i) const { return ld_ro(t + (PF_RA + i) * ld); }
    __device__ __forceinline__ T RC(int i) const { return ld_ro(t + (PF_RC + i) * ld); }
    __device__ __forceinline__ T RA(int i) const { return ld_ro(t + (PF_RAS + i) * ld); }
    __device__ __forceinline__ T D(int i) const { return ld_ro(t + (PF_D + i) * ld); }
    __device__ __forceinline__ T C_vc(int i) const { return ld_ro(t + (PF_CVC + i) * ld); }
    __device__ __forceinline__ T r_v_cv(int i) const { return ld_ro(t + (PF_RVCV + i) * ld); }
    __device__ __forceinline__ T q_vc(int i) const { return ld_ro(t + (PF_QVC + i) * ld); }
    __device__ __forceinline__ double meas_delay() const { return ld_ro(dl); }
    __device__ __forceinline__ double dyn_offset() const { return ld_ro(dl + ld); }
    __device__ __forceinline__ T dT() const { return at(QEKF_CS_OFF(dT), 0); }
    __device__ __forceinline__ T g(int i) const { return at(QEKF_CS_OFF(g), i); }
    __device__ __forceinline__ T ab_static(int i) const { return at(QEKF_CS_OFF(ab_static), i); }
    __device__ __forceinline__ T wb_static(int i) const { return at(QEKF_CS_OFF(wb_static), i); }
    __device__ __forceinline__ T small_ang_tol() const { return at(QEKF_CS_OFF(small_ang_tol), 0); }
    __device__ __forceinline__ T cov_init(int i) const { return at(QEKF_CS_OFF(cov_init), i); }
};
#endif

// ------------------------------------------------------------------------------------------------
// packed symmetric covariance storage.  Element (i,j), i<=j, lives at index i*N - i(i-1)/2 + (j-i).
// All call sites pass compile-time indices (fully unrolled loops), so the index math folds away.
// ------------------------------------------------------------------------------------------------
template <int N> __host__ __device__ constexpr int sym_idx(int i, int j)
{
    return (i <= j) ? (i * N - (i * (i - 1)) / 2 + (j - i)) : (j * N - (j * (j - 1)) / 2 + (i - j));
}

// covariance in shared memory, element-major: element e of the filter of lane l at base[e*STRIDE]
// (base already points at the lane) -> conflict-free 8-byte accesses across a warp.
#ifdef QEKF_EXP8
#define QEKF_EXP8_MAP(e) ((sizeof(T) == 8 && N == 15 && (e) >= 105) ? (e) - 15 : (e))
#else
#define QEKF_EXP8_MAP(e) (e)
#endif
template <typename T, int N, int STRIDE> struct PShared {
    T *base;
    static constexpr int n = N;
    QEKF_FN T ld(int i, int j) const { return base[QEKF_EXP8_MAP(sym_idx<N>(i, j)) * STRIDE]; }
    QEKF_FN void st(int i, int j, T v) { base[QEKF_EXP8_MAP(sym_idx<N>(i, j)) * STRIDE] = v; }
    QEKF_FN T &el(int e) { return base[QEKF_EXP8_MAP(e) * STRIDE]; }
    QEKF_FN const T &el(int e) const { return base[QEKF_EXP8_MAP(e) * STRIDE]; }
};

// covariance in a thread-local array (registers when indices are static)
template <typename T, int N> struct PLocal {
    T p[N * (N + 1) / 2];
    static constexpr int n = N;
    QEKF_FN T ld(int i, int j) const { return p[sym_idx<N>(i, j)]; }
    QEKF_FN void st(int i, int j, T v) { p[sym_idx<N>(i, j)] = v; }
    QEKF_FN T &el(int e) { return p[e]; }
    QEKF_FN const T &el(int e) const { return p[e]; }
};

// load block (X,Y) as a full 3x3 (row-major) in (X,Y) orientation, whatever the storage orientation
template <class PS, typename T> QEKF_FN void ldb(const PS &P, int X, int Y, T b[9])
{
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) b[a * 3 + c] = P.ld(3 * X + a, 3 * Y + c);
}
// store block (X,Y) given in (X,Y) orientation; diagonal blocks store their upper triangle only
template <class PS, typename T> QEKF_FN void stb(PS &P, int X, int Y, const T b[9])
{
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (X == Y) {
                if (a <= c) P.st(3 * X + a, 3 * Y + c, b[a * 3 + c]);
            } else if (X < Y) {
                P.st(3 * X + a, 3 * Y + c, b[a * 3 + c]);
            } else {
                P.st(3 * Y + c, 3 * X + a, b[a * 3 + c]);
            }
        }
}

// ------------------------------------------------------------------------------------------------
// tiny 3x3 helpers (row-major, fully unrolled)
// ------------------------------------------------------------------------------------------------
// O += A * B
template <typename T> QEKF_FN void mm_acc(T O[9], const T A[9], const T B[9])
{
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            T s = O[a * 3 + c];
#pragma unroll
            for (int k = 0; k < 3; ++k) s = M<T>::fma_(A[a * 3 + k], B[k * 3 + c], s);
            O[a * 3 + c] = s;
        }
}
// O += A * B^T
template <typename T> QEKF_FN void mmt_acc(T O[9], const T A[9], const T B[9])
{
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            T s = O[a * 3 + c];
#pragma unroll
            for (int k = 0; k < 3; ++k) s = M<T>::fma_(A[a * 3 + k], B[c * 3 + k], s);
            O[a * 3 + c] = s;
        }
}
// O = A * B
template <typename T> QEKF_FN void mm_set(T O[9], const T A[9], const T B[9])
{
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            T s = A[a * 3 + 0] * B[0 * 3 + c];
            s = M<T>::fma_(A[a * 3 + 1], B[1 * 3 + c], s);
            s = M<T>::fma_(A[a * 3 + 2], B[2 * 3 + c], s);
            O[a * 3 + c] = s;
        }
}
template <typename T> QEKF_FN void mv(const T A[9], const T v[3], T o[3])
{
#pragma unroll
    for (int a = 0; a < 3; ++a) o[a] = M<T>::fma_(A[a * 3 + 2], v[2], M<T>::fma_(A[a * 3 + 1], v[1], A[a * 3] * v[0]));
}

// ------------------------------------------------------------------------------------------------
// quaternion helpers (xyzw)                                  quaternion_helper.cpp:9-100
// ------------------------------------------------------------------------------------------------
// normalise, then flip the sign iff w < -0.75                quaternion_helper.cpp:61-73
template <typename T> QEKF_FN void quat_normclip(T q[4])
{
    T n2 = M<T>::fma_(q[3], q[3], M<T>::fma_(q[2], q[2], M<T>::fma_(q[1], q[1], q[0] * q[0])));
    if (n2 > T(0)) {
        T inv = T(1) / M<T>::sqrt_(n2);
        q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
    }
    if (q[3] < T(-0.75)) { q[0] = -q[0]; q[1] = -q[1]; q[2] = -q[2]; q[3] = -q[3]; }
}
// Hamilton product
template <typename T> QEKF_FN void quat_mul(const T a[4], const T b[4], T o[4])
{
    T ax = a[0], ay = a[1], az = a[2], aw = a[3], bx = b[0], by = b[1], bz = b[2], bw = b[3];
    o[3] = aw * bw - ax * bx - ay * by - az * bz;
    o[0] = aw * bx + ax * bw + ay * bz - az * by;
    o[1] = aw * by + ay * bw + az * bx - ax * bz;
    o[2] = aw * bz + az * bw + ax * by - ay * bx;
}
// conj(a) (x) b
template <typename T> QEKF_FN void quat_conj_mul(const T a[4], const T b[4], T o[4])
{
    T c[4] = { -a[0], -a[1], -a[2], a[3] };
    quat_mul(c, b, o);
}
// rotation matrix of a unit quaternion (no normalisation), Eigen's toRotationMatrix convention
template <typename T> QEKF_FN void quat_to_rot(const T q[4], T R[9])
{
    T x = q[0], y = q[1], z = q[2], w = q[3];
    T tx = x + x, ty = y + y, tz = z + z;
    T twx = tx * w, twy = ty * w, twz = tz * w;
    T txx = tx * x, txy = ty * x, txz = tz * x;
    T tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = T(1) - (tyy + tzz); R[1] = txy - twz;          R[2] = txz + twy;
    R[3] = txy + twz;          R[4] = T(1) - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy;          R[7] = tyz + twx;          R[8] = T(1) - (txx + tyy);
}
// exp map, pure -> unit quaternion                             quaternion_helper.cpp:9-33
// also returns half-angle sin/cos and the norm so the caller can reuse them for Rodrigues.
template <typename T>
QEKF_FN void quat_exp(const T v[3], T q[4], T &norm, T &sh, T &ch)
{
    T n2 = M<T>::fma_(v[2], v[2], M<T>::fma_(v[1], v[1], v[0] * v[0]));
    norm = M<T>::sqrt_(n2);
    M<T>::sincos_(norm * T(0.5), &sh, &ch);
    T f;
    if (norm < T(1e-10)) f = T(0.5) * (T(1) - n2 / T(24));
    else f = sh / norm;
    q[0] = v[0] * f; q[1] = v[1] * f; q[2] = v[2] * f; q[3] = ch;
    quat_normclip(q);
}
// log map, unit -> pure quaternion (input is not normalised here)   quaternion_helper.cpp:36-58
template <typename T> QEKF_FN void quat_log(const T q[4], T v[3])
{
    T n2 = M<T>::fma_(q[2], q[2], M<T>::fma_(q[1], q[1], q[0] * q[0]));
    T vn = M<T>::sqrt_(n2);
    T f;
    if (vn < T(1e-10)) {
        T rw = vn / q[3];
        f = T(2) / q[3] * (T(1) - rw * rw / T(3));
    } else {
        f = T(2) * M<T>::atan2_(vn, q[3]) / vn;
    }
    v[0] = f * q[0]; v[1] = f * q[1]; v[2] = f * q[2];
}

// ------------------------------------------------------------------------------------------------
// attitude propagation of one tick                           relative_pose_EKF.cpp:383-401
//   q <- normclip(q (x) exp(dth)),   Phi = I - skew(dth)  (|dth| < small_ang_tol)  or  Rodrigues(-|dth|, dth/|dth|)
// returned as Phi = cs I + s1 K1 + s2 dth dth^T with K1 = -skew(dth).
//
// Fast path (|dth| < 0.2 rad per tick, i.e. < 40 rad/s at 200 Hz): sin(h)/|dth| and cos(h), h = |dth|/2, are
// even series in |dth|^2, so there is no square root, no division and no sincos on the per-tick dependency
// chain; sin(ang)/ang = 2 f ch and (1 - cos ang)/ang^2 = 2 f^2 follow from the half-angle values.  exp(dth) is
// a unit quaternion to rounding (the reference's normalisation of it changes the last bit only) and the
// product of two unit quaternions is renormalised with one Newton step of 1/sqrt about 1 (error 3/8 e^2,
// e = |q|^2 - 1 ~ 1e-16).  Anything else (large rates, a nominal quaternion that is not unit) takes the
// reference's literal sequence in attitude_step_exact.  Both agree to ~1e-16; the parity bar is 1e-9.
// ------------------------------------------------------------------------------------------------
template <typename T> struct PhiCoef { T cs, s1, s2; };

template <typename T> __host__ __device__ __noinline__ void attitude_step_exact(T q[4], const T dth[3], T small_ang_tol, PhiCoef<T> &pc)
{
    T qe[4], ang, sh, ch;
    quat_exp(dth, qe, ang, sh, ch);
    T qn[4];
    quat_mul(q, qe, qn);
    quat_normclip(qn);
#pragma unroll
    for (int i = 0; i < 4; ++i) q[i] = qn[i];
    if (ang < small_ang_tol) {
        pc.cs = T(1); pc.s1 = T(1); pc.s2 = T(0);
    } else {
        const T inv = T(1) / ang;
        pc.s1 = T(2) * sh * ch * inv;
        pc.s2 = T(2) * sh * sh * inv * inv;
        pc.cs = T(1) - T(2) * sh * sh;
    }
}

template <typename T> QEKF_FN void attitude_step(T q[4], const T dth[3], T small_ang_tol, PhiCoef<T> &pc)
{
    const T n2 = M<T>::fma_(dth[2], dth[2], M<T>::fma_(dth[1], dth[1], dth[0] * dth[0]));
    if (n2 < T(0.04)) {
        const T x = T(0.25) * n2;                      // h^2
        T sc = M<T>::fma_(x, T(-1.0 / 110.0), T(1));   // sin(h)/h = 1 - x/6 (1 - x/20 (1 - x/42 (1 - x/72 (1 - x/110))))
        sc = M<T>::fma_(-x * sc, T(1.0 / 72.0), T(1));
        sc = M<T>::fma_(-x * sc, T(1.0 / 42.0), T(1));
        sc = M<T>::fma_(-x * sc, T(1.0 / 20.0), T(1));
        sc = M<T>::fma_(-x * sc, T(1.0 / 6.0), T(1));
        T ch = M<T>::fma_(x, T(-1.0 / 132.0), T(1));   // cos(h) = 1 - x/2 (1 - x/12 (1 - x/30 (1 - x/56 (1 - x/90 (1 - x/132)))))
        ch = M<T>::fma_(-x * ch, T(1.0 / 90.0), T(1));
        ch = M<T>::fma_(-x * ch, T(1.0 / 56.0), T(1));
        ch = M<T>::fma_(-x * ch, T(1.0 / 30.0), T(1));
        ch = M<T>::fma_(-x * ch, T(1.0 / 12.0), T(1));
        ch = M<T>::fma_(-x * ch, T(0.5), T(1));
        const T f = T(0.5) * sc;                       // sin(h)/|dth|
        const T qe[4] = { dth[0] * f, dth[1] * f, dth[2] * f, ch };
        T qn[4];
        quat_mul(q, qe, qn);
        const T m2 = M<T>::fma_(qn[3], qn[3], M<T>::fma_(qn[2], qn[2], M<T>::fma_(qn[1], qn[1], qn[0] * qn[0])));
        const T e = m2 - T(1);
        if (M<T>::abs_(e) < T(1e-8)) {
            T sc2 = M<T>::fma_(T(-0.5), e, T(1));
            if (qn[3] < T(-0.75)) sc2 = -sc2;
#pragma unroll
            for (int i = 0; i < 4; ++i) q[i] = qn[i] * sc2;
            const bool small = n2 < small_ang_tol * small_ang_tol && small_ang_tol > T(0);
            const T f2 = T(2) * f;
            pc.s1 = small ? T(1) : f2 * ch;
            pc.s2 = small ? T(0) : f2 * f;
            pc.cs = small ? T(1) : M<T>::fma_(-f2 * f, n2, T(1));
            return;
        }
    }
    {   // (copies: the out-of-line call must not pin the caller's q / coefficients to local memory)
        T qq[4] = { q[0], q[1], q[2], q[3] };
        const T dd[3] = { dth[0], dth[1], dth[2] };
        PhiCoef<T> pp;
        attitude_step_exact(qq, dd, small_ang_tol, pp);
#pragma unroll
        for (int i = 0; i < 4; ++i) q[i] = qq[i];
        pc = pp;
    }
}

// Phi (row-major) from its coefficients
template <typename T> QEKF_FN void phi_matrix(const PhiCoef<T> &pc, const T dth[3], T Phi[9])
{
    const T a0 = pc.s2 * dth[0], a1 = pc.s2 * dth[1], a2 = pc.s2 * dth[2];
    const T b0 = pc.s1 * dth[0], b1 = pc.s1 * dth[1], b2 = pc.s1 * dth[2];
    Phi[0] = M<T>::fma_(a0, dth[0], pc.cs);
    Phi[4] = M<T>::fma_(a1, dth[1], pc.cs);
    Phi[8] = M<T>::fma_(a2, dth[2], pc.cs);
    Phi[1] = M<T>::fma_(a0, dth[1], b2);  Phi[3] = M<T>::fma_(a0, dth[1], -b2);
    Phi[2] = M<T>::fma_(a0, dth[2], -b1); Phi[6] = M<T>::fma_(a0, dth[2], b1);
    Phi[5] = M<T>::fma_(a1, dth[2], b0);  Phi[7] = M<T>::fma_(a1, dth[2], -b0);
}

// ------------------------------------------------------------------------------------------------
// initialize_state                                              relative_pose_EKF.cpp:305-344
// ------------------------------------------------------------------------------------------------
template <typename T, bool BIAS, class PS, class PAR>
QEKF_FN void initialize_state(Nominal<T> &s, PS &P, const T tag[7], const PAR &par, bool reinit_bias)
{
    T qq[4], Cvc[9];
    {
        T qvc[4] = { par.q_vc(0), par.q_vc(1), par.q_vc(2), par.q_vc(3) };
        quat_mul(qvc, tag + 3, qq);
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) Cvc[i] = par.C_vc(i);
    s.q[0] = -qq[0]; s.q[1] = -qq[1]; s.q[2] = -qq[2]; s.q[3] = qq[3];
    quat_normclip(s.q);
    T Rq[9], pc[3], ro[3];
    quat_to_rot(s.q, Rq);
    mv(Cvc, tag, pc);
#pragma unroll
    for (int i = 0; i < 3; ++i) pc[i] += par.r_v_cv(i);
    mv(Rq, pc, ro);
#pragma unroll
    for (int i = 0; i < 3; ++i) { s.r[i] = -ro[i]; s.v[i] = T(0); }
    if (reinit_bias) {
#pragma unroll
        for (int i = 0; i < 3; ++i) { s.ab[i] = T(0); s.wb[i] = T(0); }
    }
    constexpr int N = BIAS ? 15 : 9;
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = i; j < N; ++j) P.st(i, j, (i == j) ? par.cov_init(i / 3) : T(0));
}

// ------------------------------------------------------------------------------------------------
// prediction_step                                               relative_pose_EKF.cpp:346-415
//
// F = E3*E2*E1 with  E1: dr += dT dv ;  E2: dv += A dtheta + B dab ;  E3: dtheta <- Phi dtheta - dT dwb
// (A = -dT C skew(a), B = -dT C, Phi = F_theta_theta), so  F P F^T  is three in-place symmetric
// congruences, each touching one block row/column.  W Q W^T = blockdiag(0, C Qa C^T, Qw, Qab, Qwb).
// ------------------------------------------------------------------------------------------------
// Jacobian pieces of one tick: A = -dT C skew(a), B = -dT C, Phi = F_theta_theta, QV = C diag(Q_a) C^T (upper)
template <typename T> struct PredJac { T A[9], B[9], Phi[9], QV[6]; };

// the nominal half of prediction_step (cpp:346-401): kinematics, and the Jacobian pieces from the pre-update state
// (Measured: running the attitude step first, so that the rest of the tick is one basic block, costs 2 %.)
template <typename T, class PAR>
QEKF_FN void pred_nominal(Nominal<T> &s, const T u[6], const PAR &par, T accel[3], PredJac<T> &J)
{
    const T d = par.dT();
    T *A = J.A, *B = J.B, *Phi = J.Phi, *QV = J.QV;
    {
        T a[3], w[3], C[9];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            a[i] = u[i] - s.ab[i] - par.ab_static(i);
            w[i] = u[3 + i] - s.wb[i] - par.wb_static(i);
        }
        quat_to_rot(s.q, C);
        T acc[3];
        mv(C, a, acc);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            acc[i] += par.g(i);
            accel[i] = acc[i];
            s.r[i] = M<T>::fma_(d, s.v[i], s.r[i]);   // uses the old v (explicit Euler)
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) s.v[i] = M<T>::fma_(d, acc[i], s.v[i]);

        // Jacobian blocks from the pre-update C, a, w
#pragma unroll
        for (int i = 0; i < 9; ++i) B[i] = -d * C[i];
#pragma unroll
        for (int i = 0; i < 3; ++i) {      // A = B * skew(a)
            A[i * 3 + 0] = B[i * 3 + 1] * a[2] - B[i * 3 + 2] * a[1];
            A[i * 3 + 1] = B[i * 3 + 2] * a[0] - B[i * 3 + 0] * a[2];
            A[i * 3 + 2] = B[i * 3 + 0] * a[1] - B[i * 3 + 1] * a[0];
        }
        // QV = C diag(Q_a) C^T (upper triangle)
        {
            int e = 0;
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = i; j < 3; ++j) {
                    QV[e++] = C[i * 3 + 0] * par.Q(0) * C[j * 3 + 0] + C[i * 3 + 1] * par.Q(1) * C[j * 3 + 1] +
                              C[i * 3 + 2] * par.Q(2) * C[j * 3 + 2];
                }
        }
        // attitude: q <- normclip(q (x) exp(dT w)); Phi = I - skew(dT w) or Rodrigues(-|dT w|)
        T dth[3] = { d * w[0], d * w[1], d * w[2] };
        PhiCoef<T> pc;
        attitude_step(s.q, dth, par.small_ang_tol(), pc);
        phi_matrix(pc, dth, Phi);
    }
}

// the covariance half (cpp:402-414): P <- F P F^T + W Q W^T through the three congruences E1, E2, E3.
// Evaluated block ROW by block row rather than congruence by congruence: the dr row first (its E1 step needs the dv
// row as it was, and its E2 / E3 steps only the Jacobian pieces), then the dv row (E2, and E3 on its dtheta block),
// then the dtheta row (E3).  Every element sees the same operations in the same order as the congruence-by-congruence
// evaluation, so the results are identical to the last bit; what changes is that a block which two or three
// congruences touch stays in registers in between instead of going through shared memory each time
// (414 -> 324 block-element accesses per prediction in the source; the shared-memory pipe is the second-busiest unit of
// the kernel).
template <typename T, bool BIAS, class PS, class PAR>
QEKF_FN void pred_cov(PS &P, const PredJac<T> &J, const PAR &par)
{
    const T d = par.dT();
    const T *A = J.A, *B = J.B, *Phi = J.Phi, *QV = J.QV;
    // ---- dr row: E1 (dr += dT dv) on every block, E2 on (r,v), E3 on (r,th) ---------------------------------------
    {
        T rvn[9], rth[9];
        {
            T vv[9], rv[9];
            ldb(P, BV, BV, vv);
            ldb(P, BR, BV, rv);
#pragma unroll
            for (int i = 0; i < 9; ++i) rvn[i] = M<T>::fma_(d, vv[i], rv[i]);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = a; b < 3; ++b) {
                    T x = P.ld(a, b);
                    x = M<T>::fma_(d, rv[b * 3 + a] + rvn[a * 3 + b], x);
                    P.st(a, b, x);
                }
        }
        {
            T sblk[9];
            ldb(P, BR, BTH, rth);
            ldb(P, BV, BTH, sblk);
#pragma unroll
            for (int i = 0; i < 9; ++i) rth[i] = M<T>::fma_(d, sblk[i], rth[i]);          // (r,th) after E1
        }
        T n[9];
        if (BIAS) {
            {
                T rw[9], sblk[9];
                ldb(P, BR, BWB, rw);
                ldb(P, BV, BWB, sblk);
#pragma unroll
                for (int i = 0; i < 9; ++i) rw[i] = M<T>::fma_(d, sblk[i], rw[i]);
                stb(P, BR, BWB, rw);                                                       // final: E2, E3 leave (r,wb) alone
#pragma unroll
                for (int i = 0; i < 9; ++i) n[i] = -d * rw[i];
            }
            {
                T ra[9], sblk[9];
                ldb(P, BR, BAB, ra);
                ldb(P, BV, BAB, sblk);
#pragma unroll
                for (int i = 0; i < 9; ++i) ra[i] = M<T>::fma_(d, sblk[i], ra[i]);
                stb(P, BR, BAB, ra);                                                       // final
                mmt_acc(rvn, rth, A);                                                      // E2: (r,v) += (r,th) A^T + (r,ab) B^T
                mmt_acc(rvn, ra, B);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 9; ++i) n[i] = T(0);
            mmt_acc(rvn, rth, A);
        }
        stb(P, BR, BV, rvn);
        mmt_acc(n, rth, Phi);                                                              // E3: (r,th) Phi^T - dT (r,wb)
        stb(P, BR, BTH, n);
    }
    // ---- dv row: E2 (dv += A dtheta + B dab), E3 on (v,th) ---------------------------------------------------------
    {
        T vv[9];
        ldb(P, BV, BV, vv);   // full symmetric copy; only the upper triangle is finally stored
        T vthn[9];            // (v,th) after E3
        if (BIAS) {
            T nw[9], blk[9];
            ldb(P, BV, BWB, nw);
            ldb(P, BTH, BWB, blk);
            mm_acc(nw, A, blk);
            ldb(P, BAB, BWB, blk);
            mm_acc(nw, B, blk);
            stb(P, BV, BWB, nw);
#pragma unroll
            for (int i = 0; i < 9; ++i) vthn[i] = -d * nw[i];
        } else {
#pragma unroll
            for (int i = 0; i < 9; ++i) vthn[i] = T(0);
        }
        {
            T o[9], n[9], thth[9];
            ldb(P, BV, BTH, o);
            ldb(P, BTH, BTH, thth);
#pragma unroll
            for (int i = 0; i < 9; ++i) n[i] = o[i];
            mm_acc(n, A, thth);
            if (BIAS) {
                T ath[9];
                ldb(P, BAB, BTH, ath);
                mm_acc(n, B, ath);
            }
            mmt_acc(vv, A, o);     // + A (v,th)_old^T
            mmt_acc(vv, n, A);     // + (v,th)_new A^T
            mmt_acc(vthn, n, Phi); // E3: (v,th) Phi^T - dT (v,wb)
            stb(P, BV, BTH, vthn);
        }
        if (BIAS) {
            T o[9], n[9], blk[9];
            ldb(P, BV, BAB, o);
#pragma unroll
            for (int i = 0; i < 9; ++i) n[i] = o[i];
            ldb(P, BTH, BAB, blk);
            mm_acc(n, A, blk);
            ldb(P, BAB, BAB, blk);
            mm_acc(n, B, blk);
            mmt_acc(vv, B, o);
            mmt_acc(vv, n, B);
            stb(P, BV, BAB, n);
        }
        // + W Q W^T on the (v,v) block, then store its upper triangle
        vv[0] += QV[0]; vv[1] += QV[1]; vv[2] += QV[2]; vv[4] += QV[3]; vv[5] += QV[4]; vv[8] += QV[5];
        stb(P, BV, BV, vv);
    }
    // ---- dtheta row: E3 (dtheta <- Phi dtheta - dT dwb) --------------------------------------------------------------
    {
        T thw_o[9], thw_n[9];
        if (BIAS) {
            {
                T tha[9], wa[9], n[9];
                ldb(P, BTH, BAB, tha);
                ldb(P, BWB, BAB, wa);
#pragma unroll
                for (int i = 0; i < 9; ++i) n[i] = -d * wa[i];
                mm_acc(n, Phi, tha);
                stb(P, BTH, BAB, n);
            }
            T ww[9];
            ldb(P, BTH, BWB, thw_o);
            ldb(P, BWB, BWB, ww);
#pragma unroll
            for (int i = 0; i < 9; ++i) thw_n[i] = -d * ww[i];
            mm_acc(thw_n, Phi, thw_o);
        }
        {
            T thth[9], m[9], n[9];
            ldb(P, BTH, BTH, thth);
            if (BIAS) {
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) m[a * 3 + b] = -d * thw_o[b * 3 + a];
#pragma unroll
                for (int i = 0; i < 9; ++i) n[i] = -d * thw_n[i];
            } else {
#pragma unroll
                for (int i = 0; i < 9; ++i) { m[i] = T(0); n[i] = T(0); }
            }
            mm_acc(m, Phi, thth);       // m = Phi (th,th) - dT (wb,th)_old
            mmt_acc(n, m, Phi);         // n = m Phi^T - dT (th,wb)_new
            n[0] += par.Q(3); n[4] += par.Q(4); n[8] += par.Q(5);
            stb(P, BTH, BTH, n);
            if (BIAS) stb(P, BTH, BWB, thw_n);
        }
        if (BIAS) {
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                P.st(9 + i, 9 + i, P.ld(9 + i, 9 + i) + par.Q(6 + i));
                P.st(12 + i, 12 + i, P.ld(12 + i, 12 + i) + par.Q(9 + i));
            }
        }
    }
}

template <typename T, bool BIAS, class PS, class PAR>
QEKF_FN void prediction_step(Nominal<T> &s, PS &P, const T u[6], const PAR &par, T accel[3])
{
    PredJac<T> J;
    pred_nominal(s, u, par, accel, J);
    pred_cov<T, BIAS>(P, J, par);
}

// ------------------------------------------------------------------------------------------------
// symmetric 6x6 inverse through Cholesky.  S is SPD by construction (G P G^T + N R N^T).
// In: packed upper triangle s[21] (sym_idx<6>).  Out: packed upper triangle of S^-1.
// The reference uses a general LU inverse (relative_pose_EKF.cpp:475); same result to rounding.
// ------------------------------------------------------------------------------------------------
template <typename T> QEKF_FN void sym6_inverse(const T s[21], T inv[21])
{
    T L[21];      // lower factor stored at sym_idx<6>(j,i) for i>=j (i.e. L[i][j])
    T dinv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        T dsum = s[sym_idx<6>(j, j)];
#pragma unroll
        for (int k = 0; k < j; ++k) dsum = M<T>::fma_(-L[sym_idx<6>(k, j)], L[sym_idx<6>(k, j)], dsum);
        T r = M<T>::rsqrt_(dsum);
        dinv[j] = r;
        L[sym_idx<6>(j, j)] = dsum * r;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            T v = s[sym_idx<6>(j, i)];
#pragma unroll
            for (int k = 0; k < j; ++k) v = M<T>::fma_(-L[sym_idx<6>(k, i)], L[sym_idx<6>(k, j)], v);
            L[sym_idx<6>(j, i)] = v * r;    // L[i][j]
        }
    }
    // Li = L^-1 (lower), Li[i][j] stored at sym_idx<6>(j,i)
    T Li[21];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        Li[sym_idx<6>(j, j)] = dinv[j];
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            T v = T(0);
#pragma unroll
            for (int k = j; k < i; ++k) v = M<T>::fma_(-L[sym_idx<6>(k, i)], Li[sym_idx<6>(j, k)], v);
            Li[sym_idx<6>(j, i)] = v * dinv[i];
        }
    }
    // S^-1 = Li^T Li :  inv[i][j] = sum_{k>=max(i,j)} Li[k][i] Li[k][j]
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = i; j < 6; ++j) {
            T v = T(0);
#pragma unroll
            for (int k = j; k < 6; ++k) v = M<T>::fma_(Li[sym_idx<6>(i, k)], Li[sym_idx<6>(j, k)], v);
            inv[sym_idx<6>(i, j)] = v;
        }
}

// Joseph form, one gain row: k <- k + (b - k S) S^-1   (see UpdateForm)
template <typename T> QEKF_FN void refine_gain_row(const T b[6], const T S[21], const T Sinv[21], T k[6])
{
    T d[6];
#pragma unroll
    for (int m = 0; m < 6; ++m) {
        T v = b[m];
#pragma unroll
        for (int l = 0; l < 6; ++l) v = M<T>::fma_(-k[l], S[sym_idx<6>(l, m)], v);
        d[m] = v;
    }
#pragma unroll
    for (int m = 0; m < 6; ++m) {
        T v = k[m];
#pragma unroll
        for (int l = 0; l < 6; ++l) v = M<T>::fma_(d[l], Sinv[sym_idx<6>(l, m)], v);
        k[m] = v;
    }
}

// x + a[0] g[0] + a[sa] g[1] + a[2 sa] g[2] in double, returned as hi + lo in T: the conventional model's columns of
// B = P G^T (G = [I Gam; 0 I]) carried to about u^2 in the FP32 mode (see correction_step)
template <typename T> QEKF_FN T gam_dot(T x, const T *a, int sa, const T g[3], T &lo)
{
    double v = (double)x;
#pragma unroll
    for (int k = 0; k < 3; ++k) v = M<double>::fma_((double)a[k * sa], (double)g[k], v);
    const T hi = (T)v;
    lo = (T)(v - (double)hi);
    return hi;
}

// one gain row from the compensated B row in double: k = (b + blo) S^-1, blo covering columns 0..2
template <typename T> QEKF_FN void gain_row_f64(const T b[6], const T blo[3], const double Sinv[21], T k[6])
{
#pragma unroll
    for (int m = 0; m < 6; ++m) {
        double v = 0.0;
#pragma unroll
        for (int l = 0; l < 6; ++l)
            v = M<double>::fma_((double)b[l] + (l < 3 ? (double)blo[l] : 0.0), Sinv[sym_idx<6>(l, m)], v);
        k[m] = (T)v;
    }
}

// outputs of a correction that the reference keeps as members (cpp:431,438,443)
template <typename T> struct Observation {
    T r_t_vt_obs[3];
    T q_tv_obs[4];
};

// ------------------------------------------------------------------------------------------------
// correction_step                                               relative_pose_EKF.cpp:417-502
//
// G = [I 0 Gam 0 0; 0 0 I 0 0] (Gam = C skew(C^T r), zero for the direct-orientation model).
// With B_X = P_X. G^T (3x6 per state block X) the update is, block by block,
//     K_X = B_X S^-1,   P^_XY = P_XY - K_X B_Y^T,   dx_X = K_X dy,
// i.e. exactly  P^ = (I - K G) P  and  dx = K dy  without materialising K or I - K G.
// JOSEPH selects the symmetrised Joseph form used by the FP32 mode.
// The refined gain leaves an error of order (kappa(S) u)^2 in the covariance.  For the direct model S = P_obs + R_k and
// kappa(S) stays ~1e3 even for stiff updates; for the conventional model G mixes position and attitude through
// Gam = C skew(C^T r) and kappa(S) reaches ~1e5, where that error exceeds the smallest posterior eigenvalues of stiff
// updates (condition ~1e7) and the covariance came out indefinite.  So in the FP32 mode the conventional model (CB
// below) forms B's columns 0..2 = P_.r + P_.th Gam^T in double and keeps them as hi + lo, forms and inverts S in double,
// computes the gain rows in double (accurate to ~u, no refinement needed) and subtracts K (hi + lo)^T.  Once per
// correction; the FP64 path and the direct model are unchanged.
// ------------------------------------------------------------------------------------------------
// The measurement-model part of correction_step (cpp:417-472): observed pose, innovation dy, R_k = N R N^T
// (packed upper 6x6) and, for the conventional model, Gam = C skew(C^T r).  Needs the nominal attitude and
// position only; shared by the thread-per-filter update below and the cooperative one (ekf_coop.cuh).
template <typename T, bool DIRECT, class PAR>
QEKF_FN void correction_front(const T q[4], const T r[3], const T tag[7], const PAR &par, Observation<T> &obs, T dy[6],
                              T Rk[21], T Gam[9])
{
    T C[9];
    quat_to_rot(q, C);
    {
        T qq[4], qvc[4] = { par.q_vc(0), par.q_vc(1), par.q_vc(2), par.q_vc(3) };
        quat_mul(qvc, tag + 3, qq);
        obs.q_tv_obs[0] = -qq[0]; obs.q_tv_obs[1] = -qq[1]; obs.q_tv_obs[2] = -qq[2]; obs.q_tv_obs[3] = qq[3];
        quat_normclip(obs.q_tv_obs);
    }
    {
        T pc[3], ro[3], Cvc[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) Cvc[i] = par.C_vc(i);
        mv(Cvc, tag, pc);
#pragma unroll
        for (int i = 0; i < 3; ++i) pc[i] += par.r_v_cv(i);
        if (DIRECT) {
            T Ro[9];
            quat_to_rot(obs.q_tv_obs, Ro);
            mv(Ro, pc, ro);
        } else {
            mv(C, pc, ro);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) { obs.r_t_vt_obs[i] = -ro[i]; dy[i] = obs.r_t_vt_obs[i] - r[i]; }
    }
    {
        T dq[4];
        quat_conj_mul(q, obs.q_tv_obs, dq);
        quat_normclip(dq);
        quat_log(dq, dy + 3);
    }
    // R_k = N R N^T, packed upper 6x6
    {
        // (0,0) block: C RC C^T  (+ skew(r) diag(Ra) skew(r)^T for the direct model)
        const T rc1 = par.RC(1), rc2 = par.RC(2), rc4 = par.RC(4);
        T RCf[9] = { par.RC(0), rc1, rc2, rc1, par.RC(3), rc4, rc2, rc4, par.RC(5) };
        T t[9], r00[9];
        mm_set(t, C, RCf);
#pragma unroll
        for (int i = 0; i < 9; ++i) r00[i] = T(0);
        mmt_acc(r00, t, C);
        if (DIRECT) {
            const T rx = r[0], ry = r[1], rz = r[2];
            const T a0 = par.Ra(0), a1 = par.Ra(1), a2 = par.Ra(2);
            // skew(r) diag(a) skew(r)^T
            r00[0] += a1 * rz * rz + a2 * ry * ry;
            r00[1] += -a2 * rx * ry;
            r00[2] += -a1 * rx * rz;
            r00[4] += a0 * rz * rz + a2 * rx * rx;
            r00[5] += -a0 * ry * rz;
            r00[8] += a0 * ry * ry + a1 * rx * rx;
            // (0,1) block: skew(r) D
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const T d0 = par.D(0 + j), d1 = par.D(3 + j), d2 = par.D(6 + j);
                Rk[sym_idx<6>(0, 3 + j)] = -rz * d1 + ry * d2;
                Rk[sym_idx<6>(1, 3 + j)] = rz * d0 - rx * d2;
                Rk[sym_idx<6>(2, 3 + j)] = -ry * d0 + rx * d1;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) Rk[sym_idx<6>(i, 3 + j)] = T(0);
        }
        Rk[sym_idx<6>(0, 0)] = r00[0]; Rk[sym_idx<6>(0, 1)] = r00[1]; Rk[sym_idx<6>(0, 2)] = r00[2];
        Rk[sym_idx<6>(1, 1)] = r00[4]; Rk[sym_idx<6>(1, 2)] = r00[5]; Rk[sym_idx<6>(2, 2)] = r00[8];
        Rk[sym_idx<6>(3, 3)] = par.RA(0); Rk[sym_idx<6>(3, 4)] = par.RA(1); Rk[sym_idx<6>(3, 5)] = par.RA(2);
        Rk[sym_idx<6>(4, 4)] = par.RA(3); Rk[sym_idx<6>(4, 5)] = par.RA(4); Rk[sym_idx<6>(5, 5)] = par.RA(5);
    }
    if (!DIRECT) {
        // Gam = C skew(C^T r)
        T Ctr[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) Ctr[i] = C[0 * 3 + i] * r[0] + C[1 * 3 + i] * r[1] + C[2 * 3 + i] * r[2];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            Gam[i * 3 + 0] = C[i * 3 + 1] * Ctr[2] - C[i * 3 + 2] * Ctr[1];
            Gam[i * 3 + 1] = C[i * 3 + 2] * Ctr[0] - C[i * 3 + 0] * Ctr[2];
            Gam[i * 3 + 2] = C[i * 3 + 0] * Ctr[1] - C[i * 3 + 1] * Ctr[0];
        }
    }
}

template <typename T, bool BIAS, bool DIRECT, class PS, class PAR>
QEKF_FN void correction_step(Nominal<T> &s, PS &P, const T tag[7], const PAR &par, Observation<T> &obs)
{
    constexpr int NB = BIAS ? 5 : 3;
    constexpr bool CB = UpdateForm<T>::joseph && !DIRECT;     // compensated B (see above)
    T dy[6];
    T Sinv[21];
    T S[21];         // innovation covariance G P G^T + R_k, packed upper triangle
    T Brt[36];       // rows: dr(0..2), dtheta(3..5) of  P_[r,th],. G^T   (6x6)
    T BrtLo[18];     // CB: low parts of Brt's columns 0..2, [row][3]
    double SinvD[CB ? 21 : 1];   // CB: S^-1 in double
    T Gam[9];
    {
        T Rk[21];
        correction_front<T, DIRECT>(s.q, s.r, tag, par, obs, dy, Rk, Gam);
        // Brt = P_[r,th],. G^T  and  S = G Brt + R_k
        {
            T rr[9], rt[9], tt[9];
            ldb(P, BR, BR, rr);
            ldb(P, BR, BTH, rt);
            ldb(P, BTH, BTH, tt);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    Brt[a * 6 + b] = rr[a * 3 + b];
                    Brt[a * 6 + 3 + b] = rt[a * 3 + b];
                    Brt[(3 + a) * 6 + b] = rt[b * 3 + a];
                    Brt[(3 + a) * 6 + 3 + b] = tt[a * 3 + b];
                }
            if (CB) {
                // columns 0..2 += (.,th) Gam^T in double, kept as hi + lo; S = G B + R_k and S^-1 from them in double
                double Sd[21];
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) {
                        Brt[a * 6 + b] = gam_dot(Brt[a * 6 + b], rt + a * 3, 1, Gam + b * 3, BrtLo[a * 3 + b]);
                        Brt[(3 + a) * 6 + b] = gam_dot(Brt[(3 + a) * 6 + b], tt + a * 3, 1, Gam + b * 3, BrtLo[(3 + a) * 3 + b]);
                    }
#pragma unroll
                for (int i = 0; i < 6; ++i)
#pragma unroll
                    for (int j = i; j < 6; ++j) {
                        double x = (double)Brt[i * 6 + j] + (j < 3 ? (double)BrtLo[i * 3 + j] : 0.0);
                        if (i < 3) {
#pragma unroll
                            for (int k = 0; k < 3; ++k) {
                                const double bkj = (double)Brt[(3 + k) * 6 + j] + (j < 3 ? (double)BrtLo[(3 + k) * 3 + j] : 0.0);
                                x = M<double>::fma_((double)Gam[i * 3 + k], bkj, x);
                            }
                        }
                        Sd[sym_idx<6>(i, j)] = x + (double)Rk[sym_idx<6>(i, j)];
                    }
                sym6_inverse(Sd, SinvD);
            } else if (!DIRECT) {
                // columns 0..2 += (.,th) Gam^T
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) {
                        T x0 = Brt[a * 6 + b], x1 = Brt[(3 + a) * 6 + b];
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            x0 = M<T>::fma_(rt[a * 3 + k], Gam[b * 3 + k], x0);
                            x1 = M<T>::fma_(tt[a * 3 + k], Gam[b * 3 + k], x1);
                        }
                        Brt[a * 6 + b] = x0;
                        Brt[(3 + a) * 6 + b] = x1;
                    }
                // S rows 0..2 = Brt_r + Gam Brt_th ; rows 3..5 = Brt_th   (upper triangle)
#pragma unroll
                for (int i = 0; i < 6; ++i)
#pragma unroll
                    for (int j = i; j < 6; ++j) {
                        T x = Brt[i * 6 + j];
                        if (i < 3) {
#pragma unroll
                            for (int k = 0; k < 3; ++k) x = M<T>::fma_(Gam[i * 3 + k], Brt[(3 + k) * 6 + j], x);
                        }
                        S[sym_idx<6>(i, j)] = x + Rk[sym_idx<6>(i, j)];
                    }
            } else {
#pragma unroll
                for (int i = 0; i < 6; ++i)
#pragma unroll
                    for (int j = i; j < 6; ++j) S[sym_idx<6>(i, j)] = Brt[i * 6 + j] + Rk[sym_idx<6>(i, j)];
            }
            if (!CB) sym6_inverse(S, Sinv);
        }
    }

    // ---- state blocks not observed directly: X in {v, ab, wb} --------------------------------
    T dth[3] = { T(0), T(0), T(0) };
#pragma unroll
    for (int xi = 0; xi < NB - 2; ++xi) {
        const int X = (xi == 0) ? BV : (xi == 1 ? BAB : BWB);
        T Bx[18], Kx[18], BxLo[9];
        {
            T xr[9], xt[9];
            ldb(P, X, BR, xr);
            ldb(P, X, BTH, xt);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    T x0 = xr[a * 3 + b];
                    if (CB) {
                        x0 = gam_dot(x0, xt + a * 3, 1, Gam + b * 3, BxLo[a * 3 + b]);
                    } else if (!DIRECT) {
#pragma unroll
                        for (int k = 0; k < 3; ++k) x0 = M<T>::fma_(xt[a * 3 + k], Gam[b * 3 + k], x0);
                    }
                    Bx[a * 6 + b] = x0;
                    Bx[a * 6 + 3 + b] = xt[a * 3 + b];
                }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (CB) {
                gain_row_f64(Bx + a * 6, BxLo + a * 3, SinvD, Kx + a * 6);
                continue;
            }
#pragma unroll
            for (int m = 0; m < 6; ++m) {
                T v = T(0);
#pragma unroll
                for (int k = 0; k < 6; ++k) v = M<T>::fma_(Bx[a * 6 + k], Sinv[sym_idx<6>(k, m)], v);
                Kx[a * 6 + m] = v;
            }
            if (UpdateForm<T>::joseph) refine_gain_row(Bx + a * 6, S, Sinv, Kx + a * 6);
        }
        // inject dx_X = K_X dy
        {
            T dx[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                T v = T(0);
#pragma unroll
                for (int m = 0; m < 6; ++m) v = M<T>::fma_(Kx[a * 6 + m], dy[m], v);
                dx[a] = v;
            }
            if (X == BV) { s.v[0] += dx[0]; s.v[1] += dx[1]; s.v[2] += dx[2]; }
            if (X == BAB) { s.ab[0] += dx[0]; s.ab[1] += dx[1]; s.ab[2] += dx[2]; }
            if (X == BWB) { s.wb[0] += dx[0]; s.wb[1] += dx[1]; s.wb[2] += dx[2]; }
        }
        // P_XY -= K_X B_Y^T for Y in {v, ab, wb}, Y >= X
#pragma unroll
        for (int yi = xi; yi < NB - 2; ++yi) {
            const int Y = (yi == 0) ? BV : (yi == 1 ? BAB : BWB);
            T By[18], ByLo[9];
            if (yi == xi) {
#pragma unroll
                for (int i = 0; i < 18; ++i) By[i] = Bx[i];
                if (CB) {
#pragma unroll
                    for (int i = 0; i < 9; ++i) ByLo[i] = BxLo[i];
                }
            } else {
                T yr[9], yt[9];
                ldb(P, Y, BR, yr);
                ldb(P, Y, BTH, yt);
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int b = 0; b < 3; ++b) {
                        T x0 = yr[a * 3 + b];
                        if (CB) {
                            x0 = gam_dot(x0, yt + a * 3, 1, Gam + b * 3, ByLo[a * 3 + b]);
                        } else if (!DIRECT) {
#pragma unroll
                            for (int k = 0; k < 3; ++k) x0 = M<T>::fma_(yt[a * 3 + k], Gam[b * 3 + k], x0);
                        }
                        By[a * 6 + b] = x0;
                        By[a * 6 + 3 + b] = yt[a * 3 + b];
                    }
            }
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    if (X == Y && b < a) continue;
                    T v = P.ld(3 * X + a, 3 * Y + b);
#pragma unroll
                    for (int m = 0; m < 6; ++m) v = M<T>::fma_(-Kx[a * 6 + m], By[b * 6 + m], v);
                    if (CB) {
#pragma unroll
                        for (int m = 0; m < 3; ++m) v = M<T>::fma_(-Kx[a * 6 + m], ByLo[b * 3 + m], v);
                    }
                    P.st(3 * X + a, 3 * Y + b, v);
                }
        }
        // (X,r) and (X,th) columns:  P_X,[r th] -= K_X Brt^T   (stored transposed: r, th < X except (v,th))
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                T v0 = P.ld(3 * BR + b, 3 * X + a);     // (r, X) storage
                T v1 = (X == BV) ? P.ld(3 * X + a, 3 * BTH + b) : P.ld(3 * BTH + b, 3 * X + a);
#pragma unroll
                for (int m = 0; m < 6; ++m) {
                    v0 = M<T>::fma_(-Kx[a * 6 + m], Brt[b * 6 + m], v0);
                    v1 = M<T>::fma_(-Kx[a * 6 + m], Brt[(3 + b) * 6 + m], v1);
                }
                if (CB) {
#pragma unroll
                    for (int m = 0; m < 3; ++m) {
                        v0 = M<T>::fma_(-Kx[a * 6 + m], BrtLo[b * 3 + m], v0);
                        v1 = M<T>::fma_(-Kx[a * 6 + m], BrtLo[(3 + b) * 3 + m], v1);
                    }
                }
                P.st(3 * BR + b, 3 * X + a, v0);
                if (X == BV) P.st(3 * X + a, 3 * BTH + b, v1);
                else P.st(3 * BTH + b, 3 * X + a, v1);
            }
    }
    // ---- the observed blocks r, theta ---------------------------------------------------------
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        T k[6];
        if (CB) {
            gain_row_f64(Brt + i * 6, BrtLo + i * 3, SinvD, k);
        } else {
#pragma unroll
            for (int m = 0; m < 6; ++m) {
                T v = T(0);
#pragma unroll
                for (int l = 0; l < 6; ++l) v = M<T>::fma_(Brt[i * 6 + l], Sinv[sym_idx<6>(l, m)], v);
                k[m] = v;
            }
            if (UpdateForm<T>::joseph) refine_gain_row(Brt + i * 6, S, Sinv, k);
        }
        T dx = T(0);
#pragma unroll
        for (int m = 0; m < 6; ++m) dx = M<T>::fma_(k[m], dy[m], dx);
        if (i < 3) s.r[i] += dx;
        else dth[i - 3] = dx;
        const int gi = (i < 3) ? i : 3 + i;          // global state index: r -> 0..2, theta -> 6..8
#pragma unroll
        for (int j = i; j < 6; ++j) {
            const int gj = (j < 3) ? j : 3 + j;
            T v = P.ld(gi, gj);
#pragma unroll
            for (int m = 0; m < 6; ++m) v = M<T>::fma_(-k[m], Brt[j * 6 + m], v);
            if (CB) {
#pragma unroll
                for (int m = 0; m < 3; ++m) v = M<T>::fma_(-k[m], BrtLo[j * 3 + m], v);
            }
            P.st(gi, gj, v);
        }
    }
    // attitude injection: q <- normclip(q (x) exp(dtheta))          (cpp:488-489)
    {
        T qe[4], qn[4], nn, sh, ch;
        quat_exp(dth, qe, nn, sh, ch);
        quat_mul(s.q, qe, qn);
        quat_normclip(qn);
#pragma unroll
        for (int i = 0; i < 4; ++i) s.q[i] = qn[i];
    }
    if (!BIAS) {   // biases are forced to zero when not estimated (cpp:491-498)
#pragma unroll
        for (int i = 0; i < 3; ++i) { s.ab[i] = T(0); s.wb[i] = T(0); }
    }
}

// ------------------------------------------------------------------------------------------------
// corner-margin gate                                            relative_pose_EKF.cpp:156-186
// ------------------------------------------------------------------------------------------------
// Evaluated in double on the double tag pose whatever the filter's type T: the decision is discrete, and in float the
// rounding of the projection (~1e-4 px at 752 px) would flip the poses whose extreme corner lies that close to a
// margin line.  Once per arrival, so the FP32 mode pays nothing for it; in FP64 it is the same arithmetic as before.
template <typename T> QEKF_FN bool corner_gate(const double tag[7], const Consts<T> &c)
{
    double Rct[9];
    quat_to_rot(tag + 3, Rct);
    bool ok = false;
    for (int i = 0; i < c.n_tags; ++i) {
        const double hw = c.tag_hw[i], px0 = c.tag_px[i], py0 = c.tag_py[i];
        double min_u = 0.0, max_u = 0.0, min_v = 0.0, max_v = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double cx = ((k == 0 || k == 3) ? hw : -hw) + px0;
            const double cy = ((k < 2) ? hw : -hw) + py0;
            double pc0 = Rct[0] * cx + Rct[1] * cy + tag[0];
            double pc1 = Rct[3] * cx + Rct[4] * cy + tag[1];
            double pc2 = Rct[6] * cx + Rct[7] * cy + tag[2];
            double iz = 1.0 / pc2;
            double xn = pc0 * iz, yn = pc1 * iz, zn = pc2 * iz;
            double uu = c.Kcam[0] * xn + c.Kcam[1] * yn + c.Kcam[2] * zn;
            double vv = c.Kcam[3] * xn + c.Kcam[4] * yn + c.Kcam[5] * zn;
            if (k == 0) { min_u = max_u = uu; min_v = max_v = vv; }
            else {
                min_u = uu < min_u ? uu : min_u; max_u = uu > max_u ? uu : max_u;
                min_v = vv < min_v ? vv : min_v; max_v = vv > max_v ? vv : max_v;
            }
        }
        ok = (min_u > c.u_lo) && (min_v > c.v_lo) && (max_u < c.u_hi) && (max_v < c.v_hi);
        if (ok) break;
    }
    return ok;
}

}  // namespace qekf
