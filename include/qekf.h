/*
 * qekf.h -- C ABI of libqekf: a B200-native (sm_100a) batched relative-pose error-state EKF.
 *
 * This is the drop-in boundary for the estimator core of mbrymer/quadrotor_landing
 * (quad_state_estimation).  The reference has no FFI layer: its boundary is the public surface of
 * the C++ class RelativePoseEKF, used by RelativePoseEKFNode through direct member access.  Every
 * entry point below names the reference interface it replaces (paths relative to
 * quad_state_estimation/ in the reference repository).
 *
 * Conventions: plain pointers and sizes only; every function returns a qekf_status (0 = ok) and
 * never throws; quaternions are (x,y,z,w) as in the reference's 16-vector
 * (src/quaternion_helper.cpp:88-100); the nominal state is x = [r(3) v(3) q(4) ab(3) wb(3)]
 * (src/relative_pose_EKF.cpp:244-245) and the covariance is over (dr, dv, dtheta, dab, dwb)
 * (src/relative_pose_EKF.cpp:484-485), 15x15, or 9x9 when est_bias = 0.
 *
 * A handle owns N independent filters on one GPU.  N = 1 is the reference's single estimator; the
 * product use is N = 10^3..10^7 Monte-Carlo / parameter-sweep instances.  There is no CPU fallback:
 * qekf_create fails with QEKF_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef QEKF_H
#define QEKF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QEKF_MAX_TAGS 16

typedef enum qekf_status {
    QEKF_OK = 0,
    QEKF_ERR_BAD_ARG = 1,
    QEKF_ERR_CUDA = 2,
    QEKF_ERR_NOT_INITIALIZED = 3,
    QEKF_ERR_UNSUPPORTED = 4,
    QEKF_ERR_NO_DEVICE = 5,
    QEKF_ERR_ALLOC = 6
} qekf_status;

typedef enum qekf_precision { QEKF_FP64 = 64, QEKF_FP32 = 32 } qekf_precision;

/* Parameters the reference's caller writes into public members before initialize_params()
 * (src/relative_pose_EKF_node.cpp:53-136; declarations include/relative_pose_EKF.hpp:67-133). */
typedef struct qekf_params {
    double update_freq;                  /* hpp:67  */
    double measurement_freq;             /* hpp:69  */
    double measurement_delay;            /* hpp:70  */
    double measurement_delay_max;        /* hpp:71  */
    double dyn_measurement_delay_offset; /* hpp:72  */
    double Q_a[3], Q_w[3], Q_ab[3], Q_wb[3]; /* hpp:97-100, per-step process noise diagonals */
    double R_r[3], R_ang[3];             /* hpp:103-104 */
    double r_cov_init, v_cov_init, ang_cov_init, ab_cov_init, wb_cov_init; /* hpp:89-93 */
    double ab_static[3], wb_static[3];   /* hpp:55-56 */
    double r_v_cv[3];                    /* hpp:108, camera position in vehicle frame */
    double q_vc[4];                      /* hpp:109, x,y,z,w (node.cpp:108-110) */
    double camera_K[9];                  /* hpp:113, row-major (node.cpp:115-117) */
    double tag_in_view_margin;           /* hpp:119 */
    double tag_widths[QEKF_MAX_TAGS];    /* hpp:121 */
    double tag_positions[3 * QEKF_MAX_TAGS]; /* hpp:122, 3 per tag (node.cpp:128-136) */
    double small_ang_tol;                /* hpp:132 */
    double g[3];                         /* hpp:133 */
    int32_t camera_width, camera_height; /* hpp:114-115 */
    int32_t n_tags;                      /* hpp:118 */
    int32_t est_bias;                    /* hpp:75 */
    int32_t limit_measurement_freq;      /* hpp:76 */
    int32_t corner_margin_enbl;          /* hpp:77 */
    int32_t direct_orien_method;         /* hpp:78 */
    int32_t multirate_ekf;               /* hpp:79 */
    int32_t dynamic_meas_delay;          /* hpp:80 */
    int32_t reserved;
} qekf_params;

typedef struct qekf_handle qekf_handle;

/* ---- lifetime ------------------------------------------------------------------------------- */

/* RelativePoseEKF::RelativePoseEKF() defaults (src/relative_pose_EKF.cpp:29-81); members the
 * constructor leaves uninitialised take the node's defaults (node.cpp:35,64,89-93). */
int qekf_default_params(qekf_params *p);

/* Construct N filters on CUDA device `device` and run initialize_params()
 * (src/relative_pose_EKF.cpp:87-125).  precision: QEKF_FP64 (reference arithmetic) or QEKF_FP32. */
int qekf_create(const qekf_params *p, int64_t n_filters, int device, int precision, qekf_handle **out);
int qekf_destroy(qekf_handle *h);

/* Overwrite parameters and re-run initialize_params() (node.cpp:53-138 then :138).  Like the
 * reference this resets cov_pert to cov_init but keeps the nominal state.  With multirate_ekf the delayed-fusion
 * history restarts from the current estimate (the reference keeps its old history vectors, so its next delayed
 * correction would silently discard the covariance reset).  Changing est_bias re-allocates the filters and drops
 * per-filter overrides. */
int qekf_set_params(qekf_handle *h, const qekf_params *p);
int qekf_get_params(const qekf_handle *h, qekf_params *p);

/* Per-filter parameter overrides for sweeps (no reference equivalent: the reference has one
 * filter).  values is a HOST array [dim][N].  Each filter's derived quantities are recomputed exactly as
 * initialize_params() would (src/relative_pose_EKF.cpp:87-125); fields never overridden keep the handle-wide
 * value.  Meant to be called before the first run; with multirate_ekf a QEKF_PF_DELAY override that changes the
 * largest step delay restarts the delayed-fusion histories from the current estimates. */
enum {
    QEKF_PF_Q = 0,      /* dim 12: Q_a, Q_w, Q_ab, Q_wb */
    QEKF_PF_R = 1,      /* dim 6 : R_r, R_ang */
    QEKF_PF_R_V_CV = 2, /* dim 3 */
    QEKF_PF_Q_VC = 3,   /* dim 4 : x,y,z,w */
    QEKF_PF_DELAY = 4   /* dim 2 : measurement_delay, dyn_measurement_delay_offset */
};
int qekf_set_filter_params(qekf_handle *h, int field, const double *values);

/* The node's parameter file -> qekf_params, as RelativePoseEKFNode's constructor fills the class
 * (src/relative_pose_EKF_node.cpp:35-136): same keys, same `param<>` defaults for missing scalars, q_vc in
 * x,y,z,w array order, camera_K row-major, three numbers per tag position.  Reads the flat YAML subset of
 * config/relative_pose_EKF_{rotors,hardware}.yaml.  Host only (no GPU needed). */
int qekf_params_from_yaml(const char *path, qekf_params *p);
int qekf_params_from_yaml_text(const char *text, qekf_params *p);

const char *qekf_last_error_string(void);
int qekf_num_states(const qekf_handle *h);   /* RelativePoseEKF::num_states (hpp:83) */
int64_t qekf_num_filters(const qekf_handle *h);

/* All work of a handle is issued on one CUDA stream (default: a private non-blocking stream).
 * qekf_set_stream adopts a caller stream (a cudaStream_t passed as void*). */
/* How the fused replay (qekf_run, qekf_run_monte_carlo) maps filters onto the GPU (FP64 single-rate handles; other
 * handles use one thread per filter whatever is set here).
 *   lanes_per_filter = 1 (default): one thread per filter -- the fastest mapping by a factor of two to three
 *       (profiles/r2_04_mappings.md);
 *   lanes_per_filter = 2: two role-specialised warps per 32 filters -- one owns the (dr,dv,dth) core of the covariance
 *       and the measurement update, the other the nominal state, the noise and the bias columns;
 *   lanes_per_filter = 3: three lanes per filter, each owning one column of every 3x3 covariance block.
 * The cooperative mappings are kept as measured alternatives.  groups: 32-filter groups per CTA (0 = the build's
 * default).  Results of the mappings agree to rounding (~1e-15), all within the 1e-9 bar against
 * relative_pose_EKF.cpp:127-502.  A qekf_run_with_truth launch that scores its filters runs one thread per filter
 * whatever is set here (the cooperative mappings accumulate statistics for qekf_run_monte_carlo only). */
int qekf_set_mapping(qekf_handle *h, int lanes_per_filter, int groups);
int qekf_set_stream(qekf_handle *h, void *cuda_stream);
int qekf_sync(qekf_handle *h);

/* ---- the reference's per-tick estimator interface (same inputs to every filter of the handle) -- */

/* IMUSubCallback (node.cpp:144-151): latch the latest IMU sample (zero-order hold). */
int qekf_set_imu(qekf_handle *h, const double accel[3], const double gyro[3]);
/* AprilTagSubCallback (node.cpp:153-176): latch detections[0] pose + header stamp, raise
 * measurement_ready, and on the first call run initialize_state(false). */
int qekf_set_tag(qekf_handle *h, const double pos[3], const double quat_xyzw[4], double stamp);
/* RelativePoseEKF::initialize_state(bool) (src/relative_pose_EKF.cpp:305-344). */
int qekf_initialize_state(qekf_handle *h, int reinit_bias);
/* RelativePoseEKF::filter_update(double) (src/relative_pose_EKF.cpp:127-303): one tick, single-rate or with
 * delayed-measurement fusion (multirate_ekf, fixed or dynamic delay: cpp:196-264).  The x_hist / u_hist / P_hist
 * vectors of the reference are kept as a lagged checkpoint plus a ring of IMU inputs and re-evaluated on demand;
 * what the accessors return after the call is what the reference's members would hold. */
int qekf_filter_update(qekf_handle *h, double t_curr);
/* Latch a tag pose WITHOUT raising measurement_ready and without the first-detection initialisation: what
 * RelativePoseEKF::initialize_state needs when the caller re-initialises by hand (it reads the latched apriltag_pos /
 * apriltag_orien members and never touches measurement_ready, relative_pose_EKF.cpp:305-344). */
int qekf_latch_tag(qekf_handle *h, const double pos[3], const double quat_xyzw[4], double stamp);
/* One timer tick of the node in ONE launch (relative_pose_EKF_node.cpp:144-283): the tag callback if a detection
 * arrived since the last tick (tag_mode 1 = AprilTagSubCallback: latch + measurement_ready + first-detection
 * initialisation; 2 = latch only; 0 = none), the IMU sample, filter_update(t_curr), and the members the node reads
 * afterwards for the first n_out filters, QEKF_TICK_RECORD doubles each:
 *   x[16] | cov_pert[n*n] row-major (n = qekf_num_states) padded to 225 | aux[11] |
 *   state_initialized measurement_ready performed_correction filter_active upds_since_correction x_hist.size()
 * Inputs and records travel through mapped pinned memory: the host pays one launch and one stream synchronisation.
 * Same arithmetic and sequencing as qekf_set_tag + qekf_set_imu + qekf_filter_update + the getters.  Handles without
 * per-filter overrides. */
#define QEKF_TICK_RECORD 258
int qekf_tick(qekf_handle *h, const double accel[3], const double gyro[3], int tag_mode, const double tag_pos[3],
              const double tag_quat_xyzw[4], double tag_stamp, double t_curr, int n_out, double *records);

/* ---- batch replay: filter_update iterated n_steps times inside one kernel launch -------------- */

/* Explicit per-filter input streams.  Tick k (absolute index) runs at t_curr = t_start + k/update_freq.
 * Before tick k's update, arrival m with tag_step[m] == k is delivered exactly as AprilTagSubCallback
 * would (per filter, skipped where tag_valid[m][i] == 0), then imu[k] is latched as IMUSubCallback
 * would.  tag_step must be strictly increasing. */
typedef struct qekf_streams {
    int64_t T;               /* ticks held in imu */
    const double *imu;       /* [T][6][N]  accel xyz, gyro xyz */
    int64_t M;               /* tag arrivals */
    const int32_t *tag_step; /* [M] */
    const double *tag_pose;  /* [M][7][N]  r_c_tc xyz, q_ct xyzw */
    const double *tag_stamp; /* [M]  capture time (s), used by dynamic_meas_delay */
    const uint8_t *tag_valid;/* [M][N] or NULL (= all valid) */
    double t_start;
    int32_t on_device;       /* 0: host pointers (copied in by the call); 1: device pointers */
    int32_t reserved;
} qekf_streams;

int qekf_run(qekf_handle *h, const qekf_streams *s, int64_t k0, int64_t n_steps);

/* qekf_run plus the on-chip statistics of qekf_stats_configure, scored against per-filter truth (recorded flights
 * with motion-capture truth, streams of another simulator, one trajectory per filter).  truth: [n_bins][16][N]
 * doubles, in the memory space s->on_device names.  Row block b is the true state after tick (b+1)*stride - 1, the
 * tick after which bin b is sampled, in the layout of qekf_get_state: r v q_tv(xyzw) ab wb.  ab and wb are the true
 * biases as the filter's ab_nom / wb_nom would hold them, without ab_static / wb_static; rows 10..15 are ignored
 * when est_bias = 0.  Sampling rule, bins and statistics are those of qekf_run_monte_carlo: only initialised filters
 * count, samples outside [0, n_bins) are dropped, and qekf_get_stats / qekf_stats_reset / export and import work
 * unchanged.  Host truth: only the bins this call samples are copied in.  truth == NULL is exactly qekf_run.
 * QEKF_ERR_NOT_INITIALIZED when truth is given and statistics are not configured. */
int qekf_run_with_truth(qekf_handle *h, const qekf_streams *s, const double *truth, int64_t k0, int64_t n_steps);

/* ---- accessors (what the node reads after each tick, node.cpp:184-281) ------------------------ */
/* All outputs are HOST arrays in [component][count] layout (component-major). */
int qekf_get_state(qekf_handle *h, int64_t first, int64_t count, double *x16);   /* r_nom v_nom q_nom ab_nom wb_nom */
int qekf_get_cov(qekf_handle *h, int64_t first, int64_t count, double *P);       /* cov_pert, [n*n][count], symmetric */
/* aux: accel_rel(3) r_t_vt_obs(3) q_tv_obs(4,xyzw) measurement_delay_curr(1) -> [11][count] */
int qekf_get_aux(qekf_handle *h, int64_t first, int64_t count, double *aux11);
/* flags: state_initialized, measurement_ready, performed_correction, filter_active,
 *        upds_since_correction, history length -> [6][count] */
int qekf_get_flags(qekf_handle *h, int64_t first, int64_t count, int32_t *flags6);
/* Overwrite nominal state and covariance (marks the filters initialised; history <- this entry).
 * x16 [16][count], P [n*n][count] (upper triangle is used).  Checkpoint/resume and step tests. */
int qekf_set_state(qekf_handle *h, int64_t first, int64_t count, const double *x16, const double *P);

/* ---- exact checkpoint / resume (no reference equivalent: the reference restarts from its constructor) ----
 * qekf_export_state writes everything a later tick depends on into one HOST blob of qekf_export_size(h) bytes:
 * nominal state, covariance, aux, the latched tag pose + stamp, flags, upds_since_correction, the latched IMU sample,
 * step counters, and -- with multirate_ekf -- the delayed-fusion history in the form the handle keeps it (lagged
 * checkpoint, ring of IMU inputs, ring head, entries after the checkpoint, x_hist.size(); together they determine
 * every entry of the reference's x_hist / u_hist / P_hist vectors, relative_pose_EKF.cpp:196-264), plus the
 * Monte-Carlo statistics accumulators when configured.  Arrays travel verbatim in the handle's precision, so
 * export -> destroy -> create (same params, N, precision, per-filter overrides) -> import -> run continues
 * bit-identically to the uninterrupted run, single-rate and delayed fusion alike (unlike qekf_set_state, which
 * restarts the history from the given entry).  qekf_import_state rejects a blob whose size, precision, parameters or
 * history geometry differ from the receiving handle's. */
int64_t qekf_export_size(const qekf_handle *h);
int qekf_export_state(qekf_handle *h, void *buf, int64_t bytes);
int qekf_import_state(qekf_handle *h, const void *buf, int64_t bytes);

/* ---- stateless step functions over a batch (private methods of the reference class) ----------- */
/* prediction_step (src/relative_pose_EKF.cpp:346-415) applied to the handle's current state with
 * per-filter inputs u [6][N] (host).  Writes accel_rel. */
int qekf_prediction_step(qekf_handle *h, const double *u);
/* correction_step (src/relative_pose_EKF.cpp:417-502) with per-filter tag pose [7][N] (host). */
int qekf_correction_step(qekf_handle *h, const double *tag_pose);

/* ---- Monte-Carlo replay: one clean scenario shared by all filters, per-filter noise generated in-kernel ----
 * (no reference equivalent: the reference runs one filter on live sensors).  The noise realisation of a
 * filter depends only on (seed, global filter id, tick / arrival index): Philox4x32-10 keyed by the seed
 * with counter (index, stream, id), one block = six 21-bit uniforms = three Box-Muller pairs.  IMU: u = clean + bias_i + sigma n.  Tag, in the
 * camera frame like the filter's R_k = N R N^T (src/relative_pose_EKF.cpp:462-472): r_c += sigma_p n,
 * q_ct <- exp(sigma_th n) (x) q_ct.  Dropouts: arrivals with dropout_k0 <= tag_step < dropout_k1 are lost
 * for every filter, plus rand_dropout_len ticks starting at a per-filter uniform tick in [lo, hi).
 * Optional detection front-end (edge_loss, range_*): detections are lost when the bundle leaves the image and the
 * pose noise grows with the camera-to-tag range, instead of a fixed sigma. */
typedef struct qekf_noise_spec {
    uint64_t seed;
    int64_t first_global_id;     /* global id of this handle's filter 0 (shards of one job share the id space) */
    double sigma_accel, sigma_gyro;
    double sigma_bias_accel, sigma_bias_gyro;
    double sigma_tag_pos, sigma_tag_ang;
    int32_t dropout_k0, dropout_k1;
    int32_t rand_dropout_len, rand_dropout_lo, rand_dropout_hi;
    int32_t edge_loss;           /* detection front-end: 1 = an arrival is lost for a filter's realisation when no tag of
                                    the bundle (tag_widths / tag_positions) projects with all four corners inside the
                                    camera_width x camera_height image (clean pose, camera_K; the geometry of the
                                    reference's corner-margin gate, src/relative_pose_EKF.cpp:156-181, at margin 0) */
    double range_ref;            /* detection front-end: > 0 makes the tag noise range dependent,                  */
    double range_exp_pos;        /*   sigma_tag_pos * (|r_c_tc| / range_ref)^range_exp_pos                         */
    double range_exp_ang;        /*   sigma_tag_ang * (|r_c_tc| / range_ref)^range_exp_ang   (0 = as configured)   */
} qekf_noise_spec;

typedef struct qekf_shared_streams {
    int64_t T;
    const double *imu_clean;      /* [T][6] */
    int64_t M;
    const int32_t *tag_step;      /* [M] strictly increasing */
    const double *tag_pose_clean; /* [M][7] */
    const double *tag_stamp;      /* [M] */
    const double *truth;          /* [T+1][10] r, v, q_tv; NULL = no statistics */
    double t_start;
    int32_t on_device;
    int32_t reserved;
} qekf_shared_streams;

int qekf_noise_default(qekf_noise_spec *n);
/* filter_update iterated n_steps times for every filter, inputs synthesised on the fly. */
int qekf_run_monte_carlo(qekf_handle *h, const qekf_shared_streams *s, const qekf_noise_spec *n, int64_t k0,
                         int64_t n_steps);
/* The realisation of filters [first, first+count) as explicit streams in the qekf_streams layout, HOST
 * outputs: imu [T][6][count], tag_pose [M][7][count], tag_valid [M][count], bias [6][count]. */
int qekf_synthesize_streams(qekf_handle *h, const qekf_shared_streams *s, const qekf_noise_spec *n, int64_t first,
                            int64_t count, double *imu, double *tag_pose, uint8_t *tag_valid, double *bias);

/* On-chip RMSE / NEES accumulation during qekf_run_monte_carlo (against the scenario truth and each filter's true
 * bias) and qekf_run_with_truth (against per-filter truth): a sample is taken after tick k whenever
 * (k+1) % stride == 0, into bin (k+1)/stride - 1.  Per bin, QEKF_STAT_DIM doubles:
 *   [0..14] sum of squared error per error-state component (dr, dv, dtheta, dab, dwb)
 *   [15] sum NEES  [16] samples  [17] samples with NEES inside the two-sided 95% chi-square interval
 *   [18] diverged samples (non-finite state or covariance not SPD)  [19] sum |dr|^2 */
#define QEKF_STAT_DIM 20
int qekf_stats_configure(qekf_handle *h, int32_t n_bins, int32_t stride);
/* The current configuration (0, 0 when statistics are not configured; qekf_import_state may have configured them). */
int qekf_stats_config(const qekf_handle *h, int32_t *n_bins, int32_t *stride);
int qekf_stats_reset(qekf_handle *h);
int qekf_get_stats(qekf_handle *h, double *out /* host [n_bins][QEKF_STAT_DIM] */);
/* Reduced statistics copied into a caller-owned DEVICE buffer [n_bins][QEKF_STAT_DIM] on the handle's
 * stream, so that the caller can all-reduce them across GPUs (NCCL) without a host round trip. */
int qekf_copy_stats_device(qekf_handle *h, void *dst_device);

/* ---- housekeeping for benchmarking ------------------------------------------------------------------- */
/* Back to the freshly constructed state: every filter uninitialised, cov_pert = cov_init, counters 0. */
int qekf_reset_filters(qekf_handle *h);
/* Number of kernels this handle has launched since creation. */
int64_t qekf_launch_count(const qekf_handle *h);
/* prediction_step / correction_step calls executed by the fused kernels since creation (or the last
 * reset): the exact work count behind a filter-steps/s or FLOP/s figure. */
int qekf_step_counts(qekf_handle *h, int64_t *n_predict, int64_t *n_correct, int reset);
/* Self-measured FMA peak of the device (independent FMA chains, no memory traffic), in TFLOP/s counting an
 * FMA as 2 flops.  precision: QEKF_FP64 or QEKF_FP32.  The roofline denominator for this compute-bound path
 * (MEASURED_PEAKS.json carries no CUDA-core FP64/FP32 figure). */
int qekf_measure_fma_peak(int device, int precision, double *tflops);

/* ---- synthetic landing scenario (host; no reference equivalent: the reference was fed by Gazebo) ---- */
/* Hover `hover_s` at z_start, then smooth-step descent to z_end; lateral sway x = ax sin(wx t),
 * y = ay sin(wy t + phase); yaw = amp sin(w t).  The truth is advanced with the filter's own discrete
 * kinematics (src/relative_pose_EKF.cpp:365-371) and measurements are the inverse of its measurement
 * model (src/relative_pose_EKF.cpp:310-313,431-443), so a noise-free replay converges onto the truth. */
typedef struct qekf_scenario_spec {
    double duration_s, hover_s;
    double z_start, z_end;
    double sway_ax, sway_wx, sway_ay, sway_wy, sway_phase_y;
    double yaw_amp, yaw_w;
    double tag_rate_hz;      /* tag arrivals per second */
    double tag_latency_s;    /* capture -> arrival latency (0 for the single-rate filter) */
    double t_start;          /* time of tick 0 */
} qekf_scenario_spec;

int qekf_scenario_default(qekf_scenario_spec *s);
/* T = ticks, M = tag arrivals for this (params, spec). */
int qekf_scenario_sizes(const qekf_params *p, const qekf_scenario_spec *s, int64_t *T, int64_t *M);
/* HOST outputs: truth [T+1][10] (r, v, q_tv after j ticks; the state after tick k is truth[k+1]),
 * imu_clean [T][6], tag_step [M], tag_pose_clean [M][7], tag_stamp [M]. */
int qekf_scenario_generate(const qekf_params *p, const qekf_scenario_spec *s, double *truth, double *imu_clean,
                           int32_t *tag_step, double *tag_pose_clean, double *tag_stamp);

#ifdef __cplusplus
}
#endif
#endif /* QEKF_H */
