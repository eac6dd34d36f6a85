// ekf_params.hpp -- host-side derivation of the kernels' constant block from qekf_params:
// RelativePoseEKF::initialize_params (quad_state_estimation/src/relative_pose_EKF.cpp:87-125).
#pragma once

#include <cmath>
#include <cstring>

#include "../../include/qekf.h"
#include "ekf_core.cuh"

namespace qekf {

// ---- host-side quaternion helpers used only for parameter derivation (cpp:121-123) -------------
inline void h_normclip(double q[4])
{
    double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n > 0) for (int i = 0; i < 4; ++i) q[i] /= n;
    if (q[3] < -0.75) for (int i = 0; i < 4; ++i) q[i] = -q[i];
}
inline void h_rot(const double q[4], double R[9])
{
    double x = q[0], y = q[1], z = q[2], w = q[3];
    double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x;
    double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = 1 - (tyy + tzz); R[1] = txy - twz;       R[2] = txz + twy;
    R[3] = txy + twz;       R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy;       R[7] = tyz + twx;       R[8] = 1 - (txx + tyy);
}

// initialize_params (relative_pose_EKF.cpp:87-125) -> the constant block the kernels read
template <typename T> Consts<T> make_consts(const qekf_params &p)
{
    Consts<T> c;
    std::memset(&c, 0, sizeof c);
    c.dT = (T)(1 / p.update_freq);
    c.upd_per_meas = (int)std::ceil(p.update_freq / p.measurement_freq);
    for (int i = 0; i < 3; ++i) {
        c.g[i] = (T)p.g[i];
        c.ab_static[i] = (T)p.ab_static[i];
        c.wb_static[i] = (T)p.wb_static[i];
        c.Q[i] = (T)p.Q_a[i]; c.Q[3 + i] = (T)p.Q_w[i]; c.Q[6 + i] = (T)p.Q_ab[i]; c.Q[9 + i] = (T)p.Q_wb[i];
        c.Rr[i] = (T)p.R_r[i]; c.Ra[i] = (T)p.R_ang[i];
        c.r_v_cv[i] = (T)p.r_v_cv[i];
    }
    double q[4] = { p.q_vc[0], p.q_vc[1], p.q_vc[2], p.q_vc[3] };
    h_normclip(q);
    double C[9];
    h_rot(q, C);
    for (int i = 0; i < 4; ++i) c.q_vc[i] = (T)q[i];
    for (int i = 0; i < 9; ++i) c.C_vc[i] = (T)C[i];
    int e = 0;
    for (int i = 0; i < 3; ++i)
        for (int j = i; j < 3; ++j, ++e) {
            double rc = 0, ra = 0;
            for (int k = 0; k < 3; ++k) {
                rc += C[i * 3 + k] * p.R_r[k] * C[j * 3 + k];
                ra += C[i * 3 + k] * p.R_ang[k] * C[j * 3 + k];
            }
            c.RC[e] = (T)rc;
            c.RA[e] = (T)ra;
        }
    for (int k = 0; k < 3; ++k)
        for (int j = 0; j < 3; ++j) c.D[k * 3 + j] = (T)(p.R_ang[k] * C[j * 3 + k]);
    c.cov_init[0] = (T)p.r_cov_init; c.cov_init[1] = (T)p.v_cov_init; c.cov_init[2] = (T)p.ang_cov_init;
    c.cov_init[3] = (T)p.ab_cov_init; c.cov_init[4] = (T)p.wb_cov_init;
    for (int i = 0; i < 6; ++i) c.Kcam[i] = p.camera_K[i];
    c.u_lo = p.camera_width * p.tag_in_view_margin;
    c.u_hi = p.camera_width * (1 - p.tag_in_view_margin);
    c.v_lo = p.camera_height * p.tag_in_view_margin;
    c.v_hi = p.camera_height * (1 - p.tag_in_view_margin);
    c.cam_w = p.camera_width;
    c.cam_h = p.camera_height;
    c.n_tags = p.n_tags;
    for (int i = 0; i < QEKF_MAX_TAGS; ++i) {
        c.tag_hw[i] = p.tag_widths[i] / 2;
        c.tag_px[i] = p.tag_positions[3 * i + 0];
        c.tag_py[i] = p.tag_positions[3 * i + 1];
    }
    c.small_ang_tol = (T)p.small_ang_tol;
    c.meas_delay = p.measurement_delay;
    c.meas_delay_max = p.measurement_delay_max;
    c.dyn_offset = p.dyn_measurement_delay_offset;
    c.dT_nom = 1 / p.update_freq;
    c.limit_measurement_freq = p.limit_measurement_freq;
    c.corner_margin_enbl = p.corner_margin_enbl;
    c.dynamic_meas_delay = p.dynamic_meas_delay;
    return c;
}

// One filter's column of the per-filter parameter table ([PF_DIM][ld], ekf_core.cuh): the overridable
// parameters of p plus everything initialize_params derives from them.
template <typename T> void fill_pf_column(const qekf_params &p, T *col, int64_t ld)
{
    const Consts<T> c = make_consts<T>(p);
    for (int i = 0; i < 12; ++i) col[(PF_Q + i) * ld] = c.Q[i];
    for (int i = 0; i < 3; ++i) col[(PF_RA + i) * ld] = c.Ra[i];
    for (int i = 0; i < 6; ++i) { col[(PF_RC + i) * ld] = c.RC[i]; col[(PF_RAS + i) * ld] = c.RA[i]; }
    for (int i = 0; i < 9; ++i) { col[(PF_D + i) * ld] = c.D[i]; col[(PF_CVC + i) * ld] = c.C_vc[i]; }
    for (int i = 0; i < 3; ++i) col[(PF_RVCV + i) * ld] = c.r_v_cv[i];
    for (int i = 0; i < 4; ++i) col[(PF_QVC + i) * ld] = c.q_vc[i];
}

// largest step delay a correction can use (cpp:199-200) and the ring length that goes with it
inline int step_of_delay(double delay, double update_freq)
{
    const int s = (int)(delay / (1 / update_freq) + 0.5);
    return s < 1 ? 1 : s;
}
inline int ring_length(int dmax, const qekf_params &p)
{
    return dmax + 2 * (int)std::ceil(p.update_freq / p.measurement_freq) + 1;
}

}  // namespace qekf
