/* dekf_b200.h -- C ABI of the B200-native batched legged-robot estimator (libdekf_b200.so).
 *
 * Drop-in boundary for the estimator hot path of well-robotics/Decentralized_EKF_MHE.  The
 * reference has no FFI layer: its boundary is the C++ class API.  Each entry point below names the
 * reference interface it replaces (paths relative to /root/reference/src):
 *
 *   dekf_config / dekf_create   struct robot_params                decentral_legged_est/include/decentral_legged_est/DecentralEst.hpp:18-63
 *                               + orien_ekf ctor parameters        orien_est/src/orien_ekf.cpp:13-33
 *                               + DecentralizedEstimation::initialize(sub, params)   DecentralEst.hpp:101, DecentralEst.cpp:9-150
 *   dekf_inputs                 struct robot_store                 DecentralEst.hpp:65-94 (the per-tick sensor snapshot;
 *                               filled by go1Sub::imu_callback / lo_callback, go1_example/src/go1Sub.cpp:30-126,
 *                               robotSub::vo_callback / orien_filter_callback, EstSub.cpp:34-55, orien_ekf callbacks :47-75)
 *   dekf_ekf_step               orien_ekf::timerCallback           orien_est/src/orien_ekf.cpp:77-89
 *                               (= get_measurement :156, gyro_nonlinear_predict :108, gyro_nonlinear_correct :125,
 *                                vo_nonlinear_correct :144)        orien_est/include/orien_ekf.hpp:79-83
 *   dekf_mhe_step               DecentralizedEstimation::initialize (T==0) / ::update(int T) (T>=1)
 *                               DecentralEst.hpp:101-102, DecentralEst.cpp:9,152; inside it MHEproblem::updateQP /
 *                               marginalizeQP / initQP / solveQP / getsolution, MheSrb.hpp:99-103.
 *                               cfg.est_type == 1 selects the KF alternative instead (InitializeKF / UpdateKF,
 *                               DecentralEst.cpp:592-861): outputs x / v_body are then x_KF_ / v_KF_b_ (valid from
 *                               T == 0) and dekf_get_arrival_cov returns (C_KF_, x_KF_)
 *   dekf_step                   both timers in lock-step (EKF tick, then MHE update on its quaternion)
 *   dekf_run                    S such ticks over a [step][field][instance] stream (robotSub::timerCallback driven S
 *                               times, EstSub.cpp:58-91)
 *   dekf_outputs                public result members R_sb_, x_MHE_, v_MHE_b_ (DecentralEst.hpp:279-285) and the
 *                               imu/filter quaternion (orien_ekf.cpp:92-95)
 *   dekf_get_arrival_cost       MHEproblem::M_p, n_p               MheSrb.hpp:86-87
 *   dekf_get_window             MHEproblem::solution (state blocks)   MheSrb.hpp:58-112 (getsolution narrows it to x_T,
 *                               MheSrb.cpp:715-723)
 *   dekf_get_window_cov         posterior covariance of each state of MHEproblem::solution (not exported by the reference)
 *   dekf_get_foot_window        MHEproblem::solution and its covariances for leg_odom_type 1 (9 + 3 num_legs rows per state)
 *   dekf_get_constrained_window MHEproblem::solution, its covariances and active bounds with addConstraints rows (MheSrb.cpp:58-68)
 *   dekf_get_window_cross_cov   lag-one cross-covariances of the states of MHEproblem::solution (not exported by the reference)
 *   dekf_get_p_vo               DecentralizedEstimation::p_vo_accmulate_   DecentralEst.hpp:280
 *   dekf_reset                  DecentralizedEstimation::reset()   DecentralEst.hpp:103
 *
 * Conventions
 *   - One handle steps `n_instances` independent estimator instances; instance i never reads
 *     instance j.  One caller thread per handle (like the reference's single-threaded executor).
 *   - Every array is SoA `[field][instance]`, instance fastest, `instance stride == n_instances`.
 *   - `dekf_*_step` take DEVICE pointers and are stream-ordered on the handle's stream (no host
 *     synchronisation); `dekf_step_host` takes HOST pointers (pinned for full speed), copies in,
 *     steps, copies the results out and synchronises -- the end-to-end path.
 *   - Quaternions are [w,x,y,z].  Times are seconds in double; they are compared in double even in
 *     the fp32 arithmetic path so that index logic stays bit-exact.
 *   - Return value: 0 on success, a negative DEKF_E* code otherwise; never throws, never aborts.
 *     Per-instance conditions (dropped VO, non-finite state) are reported through `status` bits.
 *   - There is NO CPU fallback: without a CUDA device dekf_create fails with DEKF_ENODEV.
 */
#ifndef DEKF_B200_H
#define DEKF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DEKF_ABI_VERSION 3

enum {
  DEKF_OK = 0,
  DEKF_EINVAL = -1,   /* bad argument / unsupported configuration */
  DEKF_ENODEV = -2,   /* no CUDA device / wrong architecture */
  DEKF_ENOMEM = -3,   /* device allocation failed */
  DEKF_ECUDA = -4,    /* CUDA runtime error (see dekf_last_error) */
  DEKF_ESTATE = -5    /* call order violated (e.g. T does not follow the previous T) */
};

enum { DEKF_ROBOT_GO1 = 0, DEKF_ROBOT_CASSIE = 1, DEKF_ROBOT_POGOX = 2 };
enum { DEKF_FP64 = 0, DEKF_FP32 = 1 };
enum { DEKF_SOLVE_FULL = 0, DEKF_SOLVE_INCREMENTAL = 1 };

/* per-instance status bits (OR-ed over the calls of one step) */
enum {
  DEKF_ST_EKF_VO_DROPPED = 1,    /* VO stamp older than all stored IMU samples (orien_ekf.cpp:178-183) */
  DEKF_ST_EKF_VO_NO_REPLAY = 2,  /* rel <= 1: state rolled back, VO not applied (orien_ekf.cpp:191) */
  DEKF_ST_EKF_HIST_OVERFLOW = 4, /* VO older than the device-side history ring (reference keeps everything) */
  DEKF_ST_MHE_VO_DROPPED = 8,    /* DecentralEst.cpp:898-904 */
  DEKF_ST_MHE_VO_BOUNDED = 16,   /* VO bounds were inserted this step (vo_to_be_processed_flag_) */
  DEKF_ST_NONFINITE = 32,
  DEKF_ST_QP_MAXITER = 64        /* state-constrained solve (v_box_enable): active set still changing at the iteration cap */
};

typedef struct dekf_config {
  int32_t abi_version;   /* DEKF_ABI_VERSION */
  int32_t n_instances;
  int32_t device;        /* CUDA device ordinal */
  int32_t precision;     /* DEKF_FP64 | DEKF_FP32 (arithmetic + state type; inputs/outputs stay double) */
  int32_t robot;         /* DEKF_ROBOT_* (kinematics compiled as __device__ functions) */
  int32_t ekf_hist_depth;/* EKF replay ring depth in ticks.  The reference keeps UNBOUNDED stacks (orien_ekf.cpp:158-163) and can rewind to
                          * any past tick; here a VO pose older than ekf_hist_depth ticks is dropped with DEKF_ST_EKF_HIST_OVERFLOW set.
                          * Needs >= (largest VO latency in seconds) * ekf_rate + 2; the default 64 covers 128 ms at the reference's
                          * 500 Hz and 320 ms at the benchmark's 200 Hz (VO latency 40 ms); 216 bytes per instance and tick. */
  int32_t debug_taps;    /* allocate b_meas / Q_meas / index-logic taps (parity tests) */
  int32_t reserved0;

  /* ---- robot_params (DecentralEst.hpp:18-63; YAML names in EstSub.cpp:125-207) */
  double p_process_std[3], accel_input_std[3], accel_bias_std[3], gyro_input_std[3];
  double quaternion_ib[4], p_ib[3];
  int32_t num_legs, leg_odom_type;
  double joint_position_std[8], joint_velocity_std[8]; /* per joint of a leg (reference: 3) */
  double foot_slide_std[3], foot_swing_std[3];
  double contact_effort_threshold;
  double p_init_std[3], v_init_std[3], foot_init_std[3], accel_bias_init_std[3];
  double vo_p_std[3];
  int32_t rate, N, est_type;
  /* DEKF_SOLVE_FULL (default): every update(T) re-sweeps the whole window, like the reference re-solves the whole QP
   * (tier A of SURVEY.md 8d).  DEKF_SOLVE_INCREMENTAL: restart the sweep from the checkpoint of the first stage that
   * changed (tier B; bit-identical results, about twice the throughput; ignored with v_box_enable, est_type 1 or
   * leg_odom_type 1). */
  int32_t window_solve;
  /* OSQP settings are accepted for source compatibility and ignored: the window is solved
   * directly (exactly), see DESIGN.md section 4. */
  double rho, alpha, delta, sigma;
  int32_t verbose, adaptRho, polish, maxQPIter;
  double realtiveTol, absTol, primTol, dualTol, timeLimit;

  /* ---- orien_ekf parameters (orien_ekf.cpp:13-18) */
  double ekf_init_std[4], ekf_process_std[3], ekf_gravity_meas_std[3], ekf_vo_meas_std[4];
  double ekf_quaternion_init[4];
  int32_t ekf_rate, reserved2;

  /* ---- state constraints (builder extension; the reference's MHEproblem::addConstraints(name, lb, ub) with
   * lb < ub, MheSrb.cpp:58-68, is never exercised by DecentralEst.cpp).  v_box_enable != 0 adds the rows
   * v_box_lo <= v_s of x_k <= v_box_hi for every state of the window at solve time (est_type 0 only). */
  int32_t v_box_enable, v_box_max_iter; /* max_iter 0 = default (50 factorisations) */
  double v_box_lo[3], v_box_hi[3];

  /* ---- lever arm from the IMU to the point whose body velocity is reported: v_MHE_b_ = R_sb (v_s + omega x p_imu_2_opti)
   * (DecentralEst.cpp:181-185 hard-codes the Go1 mocap marker offset (0.016041, 0.089061, 0.0579875); the Go1 defaults
   * carry that value, the builder-defined Cassie / PogoX defaults carry zero). */
  double p_imu_2_opti[3];
  /* est_type 1 only: keep the per-leg measurement information of the newest sample so that DEKF_GET_KF_GAIN can return
   * K_KF_ (DecentralEst.hpp:290); costs 6 * num_legs doubles per instance of state and their write per tick. */
  int32_t kf_export_gain, reserved3;

  /* ---- general per-component state bounds: what MHEproblem::addConstraints(name, lb, ub) with lb < ub plus a dependency on
   * x_k through a selector row would add (MheSrb.cpp:58-68, :217-270; never exercised by the reference).  Bit a of x_box_mask
   * (a = 0..8: p_s xyz, v_s xyz, accel bias xyz) adds the rows  x_box_lo[a] <= x_k[a] <= x_box_hi[a]  for every state of the
   * window at solve time; combines with v_box_* (components 3..5; x_box_* wins where both bound a component).  est_type 0,
   * leg_odom_type 0.  Bounds on p_s or bias components are solved by the one-thread-per-instance active-set kernel
   * (k_solve_box), velocity-only bounds by the team kernel. */
  int32_t x_box_mask, reserved4;
  double x_box_lo[9], x_box_hi[9];
} dekf_config;

/* Per-tick sensor snapshot of all instances.  NULL vo_flag == no VO message for anybody. */
typedef struct dekf_inputs {
  const double *gyro;        /* [3][n]  robot_store.angular_b_  (rad/s, body) */
  const double *accel;       /* [3][n]  robot_store.accel_b_    (m/s^2, body, incl. gravity) */
  const double *imu_time;    /* [n]     robot_store.imu_time_ */
  const double *joint_pos;   /* [num_legs*nj][n] joint_states_position_[0..] */
  const double *joint_vel;   /* [num_legs*nj][n] joint_states_velocity_ */
  const double *foot_force;  /* [num_legs][n]    joint_states_position_[12+i] (go1Sub.cpp:74) */
  const uint8_t *vo_flag;    /* [n]     robot_store.vo_new_ / orien_ekf vo_new_ */
  const double *vo_quat;     /* [4][n]  orb/pos orientation (orien_ekf.cpp:47-58) */
  const double *vo_time_pre; /* [n]     robot_store.vo_time_pre_ */
  const double *vo_time_now; /* [n]     robot_store.vo_time_now_ (also the orb/pos stamp) */
  const double *vo_rel_p;    /* [3][n]  robot_store.vo_p_body_pre_2_body_ */
  const double *quat;        /* [4][n]  robot_store.quaternion_ for dekf_mhe_step; NULL = use the EKF state */
} dekf_inputs;

typedef struct dekf_outputs {
  double *quat;     /* [4][n] EKF quaternion after the tick (may be NULL) */
  double *x;        /* [ds][n] x_MHE_ = [p_s, v_s, accel bias (, foot positions if leg_odom_type 1)], ds = dekf_state_dim()
                     * (valid for T>=1; may be NULL) */
  double *v_body;   /* [3][n] v_MHE_b_ (may be NULL) */
  uint8_t *contact; /* [num_legs][n] contact flags (may be NULL) */
  int32_t *status;  /* [n] status bits of this call (may be NULL) */
} dekf_outputs;

typedef struct dekf_handle dekf_handle;

/* parameters_go1.yaml (go1_example/config) with the EKF block of the same file */
int dekf_config_default_go1(dekf_config *cfg);
/* builder-defined model parameter sets (the reference ships Go1 only) */
int dekf_config_default_cassie(dekf_config *cfg);
int dekf_config_default_pogox(dekf_config *cfg);

int dekf_create(const dekf_config *cfg, dekf_handle **out);
int dekf_destroy(dekf_handle *h);
int dekf_reset(dekf_handle *h);
/* cudaStream_t to order the step calls on (default: a private non-blocking stream) */
int dekf_set_stream(dekf_handle *h, void *cuda_stream);
void *dekf_get_stream(dekf_handle *h);
const char *dekf_last_error(const dekf_handle *h);
int dekf_num_joints(const dekf_handle *h); /* num_legs * joints per leg */
int dekf_state_dim(const dekf_handle *h);  /* dim_state_ = 9 + 3 * leg_odom_type * num_legs (DecentralEst.cpp:20) = rows of dekf_outputs.x */

/* Device-pointer, stream-ordered entry points. */
int dekf_ekf_step(dekf_handle *h, const dekf_inputs *in, const dekf_outputs *out);
int dekf_mhe_step(dekf_handle *h, int32_t T, const dekf_inputs *in, const dekf_outputs *out);
int dekf_step(dekf_handle *h, int32_t T, const dekf_inputs *in, const dekf_outputs *out);

/* S consecutive lock-step ticks T0 .. T0+S-1 in one call (trajectory sweeps, Monte-Carlo runs): every non-NULL array of
 * `in` is a stream [S][rows][n] (tick stride = rows*n elements; vo_flag is [S][n]).  `vo_steps` (HOST array [S], may be
 * NULL) marks the ticks at which any instance carries a VO message; the other ticks skip the VO arrays.  With
 * out_per_step != 0 the arrays of `out` are streams [S][rows][n] too, otherwise they receive the last tick only.
 * Device pointers, stream-ordered, no host synchronisation. */
int dekf_run(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const uint8_t *vo_steps, const dekf_outputs *out,
             int32_t out_per_step);

/* Host-pointer entry points (pinned memory for full speed): H2D copies of `in`, the device call, D2H copies of `out`,
 * stream sync.  dekf_mhe_step_host / dekf_ekf_step_host are what a single-robot ROS node binds (INTEGRATION.md 2). */
int dekf_step_host(dekf_handle *h, int32_t T, const dekf_inputs *in, const dekf_outputs *out);
int dekf_mhe_step_host(dekf_handle *h, int32_t T, const dekf_inputs *in, const dekf_outputs *out);
int dekf_ekf_step_host(dekf_handle *h, const dekf_inputs *in, const dekf_outputs *out);
/* dekf_run with HOST streams: a three-stream software pipeline (H2D of tick s+1 | kernels of tick s | D2H of tick s-1)
 * over two device staging sets; returns after the last result has landed in host memory. */
int dekf_run_host(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs *in, const uint8_t *vo_steps,
                  const dekf_outputs *out, int32_t out_per_step);
/* dekf_run_host for sensor streams delivered in single precision -- what the robot's SDK produces (Unitree LowState: float
 * IMU, joint and foot-force fields; the reference's callbacks widen them into the double members of robot_store,
 * go1Sub.cpp:30-75).  The five sensor arrays travel over PCIe as float32 (136 instead of 272 bytes per instance-tick) and are
 * widened to double on the device; time stamps and VO messages stay double; ALL arithmetic is unchanged, so for values
 * representable in float32 the results equal dekf_run_host bit for bit. */
typedef struct dekf_inputs_f32 {
  const float *gyro;        /* [S][3][n] */
  const float *accel;       /* [S][3][n] */
  const double *imu_time;   /* [S][n] */
  const float *joint_pos;   /* [S][num_legs*nj][n] */
  const float *joint_vel;   /* [S][num_legs*nj][n] */
  const float *foot_force;  /* [S][num_legs][n] */
  const uint8_t *vo_flag;    /* [S][n] or NULL */
  const double *vo_quat;     /* [S][4][n] */
  const double *vo_time_pre; /* [S][n] */
  const double *vo_time_now; /* [S][n] */
  const double *vo_rel_p;    /* [S][3][n] */
} dekf_inputs_f32;
int dekf_run_host_f32(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs_f32 *in, const uint8_t *vo_steps,
                      const dekf_outputs *out, int32_t out_per_step);
/* The same with the RESULTS delivered in single precision as well (the ROS messages the reference publishes them in carry
 * float64, but a fleet logger / controller consuming 65,536 robots' states rarely needs more than float32): quaternion,
 * x_MHE_ and v_MHE_b_ are computed in double on the device exactly as in dekf_run_host, rounded to float32 once (round to
 * nearest) by a device kernel and copied out as 64 instead of 128 bytes per instance-tick.  Contact flags and status words are
 * unchanged.  Every value equals (float) of what dekf_run_host_f32 returns for the same call. */
typedef struct dekf_outputs_f32 {
  float *quat;      /* [4][n]  (per step: [S][4][n]) */
  float *x;         /* [ds][n] */
  float *v_body;    /* [3][n] */
  uint8_t *contact; /* [num_legs][n] */
  int32_t *status;  /* [n] */
} dekf_outputs_f32;
int dekf_run_host_f32io(dekf_handle *h, int32_t T0, int32_t S, const dekf_inputs_f32 *in, const uint8_t *vo_steps,
                        const dekf_outputs_f32 *out, int32_t out_per_step);
int dekf_synchronize(dekf_handle *h);

/* Getters (device pointers, stream-ordered). */
int dekf_get_arrival_cost(dekf_handle *h, double *M_p /*[ds*ds][n]*/, double *n_p /*[ds][n]*/);
int dekf_get_arrival_cov(dekf_handle *h, double *P /*[81][n]*/, double *x /*[9][n]*/); /* leg_odom_type 0 only */
int dekf_get_p_vo(dekf_handle *h, double *p /*[3][n]*/);
int dekf_get_R_sb(dekf_handle *h, double *R /*[9][n]*/);
int dekf_get_ekf_cov(dekf_handle *h, double *P /*[16][n]*/);
/* number of window stages whose VO row is currently an equality (LinearConstraint.equality, MheSrb.hpp:38) */
int dekf_get_window_vo_count(dekf_handle *h, int32_t *count /*[n]*/);
/* Smoothed window of the last update(T) (T >= 1): the state blocks of MHEproblem::solution (MheSrb.hpp:58-112) -- the exact
 * optimum of the window QP for every state, not only x_T.  x receives [K][9][n] (device pointer, stream-ordered),
 * K = min(T+1, N), row j = stage T-K+1+j, row K-1 equal to dekf_outputs.x of that update bit for bit.  *len (host, may be
 * NULL) receives K.  est_type 0, leg_odom_type 0, no state bounds / rows; both window_solve modes (DEKF_SOLVE_FULL runs a
 * forward sweep from the arrival cost into a scratch ring allocated on first use, counted in dekf_device_bytes).
 * DEKF_EINVAL for a null x or an unsupported handle, DEKF_ESTATE before the first update(T >= 1) and after dekf_reset. */
int dekf_get_window(dekf_handle *h, double *x, int32_t *len);
/* Smoothed covariances of the same window: for every state its 9x9 block of the window QP's posterior covariance (the x_k
 * block of the inverse of the QP's KKT matrix over its equality rows; the scaling of dekf_get_arrival_cov, M_p = P^-1).
 * P receives [K][81][n] (device pointer, stream-ordered), block j = stage T-K+1+j, each block row-major over (p_s, v_s,
 * accel bias) and exactly symmetric; block K-1 is the filtered covariance of x_T.  *len (host, may be NULL) receives K.  Same
 * handles, modes, scratch ring and errors as dekf_get_window (DEKF_EINVAL for a null P). */
int dekf_get_window_cov(dekf_handle *h, double *P, int32_t *len);
/* Smoothed window of a foot-state handle (leg_odom_type 1, est_type 0): for every state of the last update's window its QP
 * optimum over all ds = dekf_state_dim(h) = 9 + 3 num_legs components (p_s, v_s, accel bias, p_foot_1 .. p_foot_L) and,
 * optionally, its ds x ds posterior covariance (the x_k block of the inverse of the window's normal matrix, in the scaling
 * where M_p is the information; row-major, exactly symmetric).  x receives [K][ds][n], P receives [K][ds * ds][n] (device
 * pointers, stream-ordered; either may be NULL, not both), row / block j = stage T-K+1+j, K = min(T+1, N); row K-1 equals
 * dekf_outputs.x of that update.  *len (host, may be NULL) receives K.  A device ring of the stage factors is allocated on
 * first use and counted in dekf_device_bytes.  DEKF_EINVAL for null x and P, est_type 1 and leg_odom_type 0 handles (those
 * use dekf_get_window / dekf_get_window_cov); DEKF_ESTATE before the first update(T >= 1) and after dekf_reset. */
int dekf_get_foot_window(dekf_handle *h, double *x, double *P, int32_t *len);
/* Window of a state-constrained handle (v_box_enable, x_box_mask or dekf_add_state_rows; est_type 0, leg_odom_type 0) after
 * the last update(T): for every state of the window QP (with its inequality rows) the optimum x (p_s, v_s, accel bias; on
 * rows handles V y), its 9x9 posterior covariance P -- the x_k block of the inverse KKT matrix with the equality rows and the
 * bounds active at the optimum as equalities, scaling M_p = P^-1, row-major, exactly symmetric, zero rows and columns for a
 * component fixed at a bound (rows handles: a_i P = 0 for every active row i) -- and the active set: bit a = lower bound of
 * row a active, bit 9 + a = upper bound (rows a = the components 0..8, or on dekf_add_state_rows handles the rows of that
 * call in order followed by the config's component bounds in ascending component order).  x receives [K][9][n], P [K][81][n],
 * active [K][n] (device pointers, stream-ordered; any may be NULL, not all three), row / block j = stage T-K+1+j,
 * K = min(T+1, N); row K-1 of x equals dekf_outputs.x of that update.  An instance whose last solve hit the iteration cap
 * (DEKF_ST_QP_MAXITER) returns the iterate the step reported in x, all-NaN P blocks and the active set as it stands.
 * *len (host, may be NULL) receives K.  DEKF_EINVAL for all-null outputs and for handles without state constraints (those
 * use dekf_get_window / dekf_get_window_cov); DEKF_ESTATE before the first update(T >= 1) and after dekf_reset. */
int dekf_get_constrained_window(dekf_handle *h, double *x, double *P, uint32_t *active, int32_t *len);
/* Lag-one cross-covariances of the window of the last update(T) (T >= 1), for every est_type 0 handle (9-state, foot states,
 * state-constrained).  C receives [K-1][ds*ds][n]: block j is Cov(x_{T-K+1+j}, x_{T-K+2+j}), row-major, with rows over the
 * components of the EARLIER state and columns over the later one.  Blocks are not symmetric.  ds = 9, or dekf_state_dim(h)
 * on leg_odom_type 1 handles.  P (may be NULL) receives in the same pass the [K][ds*ds][n] diagonal blocks, bit for bit what
 * the handle kind's covariance getter returns.  K = min(T+1, N); *len (host, may be NULL) receives K.  The scaling is that of
 * the covariance getters.  Device pointers, stream-ordered.  State-constrained handles: the bounds active at the optimum are
 * equalities, so the rows of components fixed at the earlier stage and the columns of those fixed at the later one are 0
 * (rows handles: a_i C = 0 for a row active at the earlier stage, C a_i' = 0 for one active at the later); an instance whose
 * last solve hit the iteration cap gets all-NaN blocks.  With the diagonal blocks these determine the whole joint posterior
 * of the window (it is Gauss-Markov): Cov(x_i, x_j) = C_i P_{i+1}^-1 C_{i+1} ... P_{j-1}^-1 C_{j-1}.  Scratch as in the
 * kind's getter; a 9-state handle called without P also allocates a [2][81][n] ring on first use, counted in
 * dekf_device_bytes.  DEKF_EINVAL for a null C and for est_type 1 handles; DEKF_ESTATE before the first update(T >= 1) and
 * after dekf_reset. */
int dekf_get_window_cross_cov(dekf_handle *h, double *P, double *C, int32_t *len);
/* Host-pointer getter for callers without a CUDA runtime of their own (the C++ facade, a ROS node): `what` selects one
 * of the arrays above, `host_out` receives it (same [rows][n] layout, double; int32 for DEKF_GET_VO_COUNT).
 * Synchronises the handle's stream. */
enum {
  DEKF_GET_R_SB = 0,       /* [9][n]  */
  DEKF_GET_P_VO = 1,       /* [3][n]  */
  DEKF_GET_ARRIVAL_M = 2,  /* [81][n] M_p */
  DEKF_GET_ARRIVAL_N = 3,  /* [9][n]  n_p */
  DEKF_GET_EKF_COV = 4,    /* [16][n] */
  DEKF_GET_VO_COUNT = 5,   /* [n] int32 */
  DEKF_GET_ARRIVAL_COV = 6,  /* [81][n] arrival covariance; est_type 1: C_KF_ (DecentralEst.hpp:288) */
  DEKF_GET_ARRIVAL_MEAN = 7, /* [9][n]  arrival mean;       est_type 1: x_KF_ */
  DEKF_GET_KF_GAIN = 8,      /* [9 * 3 * num_legs][n] K_KF_ (DecentralEst.hpp:290, DecentralEst.cpp:858), row-major 9 x 3L per
                              * instance; est_type 1, leg_odom_type 0 and cfg.kf_export_gain only */
  DEKF_GET_WINDOW_X = 9,     /* [K * 9][n] smoothed window (dekf_get_window); K <= N, so room for N * 9 rows suffices */
  DEKF_GET_WINDOW_P = 10,    /* [K * 81][n] smoothed covariances (dekf_get_window_cov); room for N * 81 rows suffices */
  DEKF_GET_FOOT_WINDOW_X = 11, /* [K * ds][n] smoothed window of a foot-state handle (dekf_get_foot_window); room for N * ds rows */
  DEKF_GET_FOOT_WINDOW_P = 12, /* [K * ds * ds][n] its covariances (dekf_get_foot_window); room for N * ds * ds rows */
  DEKF_GET_BOX_WINDOW_X = 13,  /* [K * 9][n] window of a state-constrained handle (dekf_get_constrained_window); room for N * 9 rows */
  DEKF_GET_BOX_WINDOW_P = 14,  /* [K * 81][n] its covariances (dekf_get_constrained_window); room for N * 81 rows */
  DEKF_GET_BOX_WINDOW_ACTIVE = 15, /* [K][n] uint32 its active sets (dekf_get_constrained_window); room for N rows */
  DEKF_GET_WINDOW_C = 16  /* [(K-1) * ds * ds][n] lag-one cross-covariances, any est_type 0 handle (dekf_get_window_cross_cov);
                           * room for (N-1) * ds * ds rows */
};
int dekf_get_host(dekf_handle *h, int32_t what, void *host_out);
/* debug taps of the last step (only when cfg.debug_taps != 0): copied into caller DEVICE buffers, any may be NULL.
 * b_meas/Q_meas: DecentralEst.cpp:515-546 per leg (Q as symmetric 3x3: 00,01,02,11,12,22);
 * vo_idx: processed,i_pre,i_now,w0,i0,ins,num,disc0 of DecentralEst.cpp:883-945 (-2 = not set);
 * ekf_idx: cur,idx,nreplay of orien_ekf.cpp:186-205. */
int dekf_debug_taps(dekf_handle *h, double *b_meas /*[3*legs][n]*/, double *Q_meas /*[legs][6][n]*/,
                    int32_t *vo_idx /*[8][n]*/, int32_t *ekf_idx /*[3][n]*/);

/* Per-kernel device time of the step kernels (CUDA events on the handle's stream around every launch while
 * enabled).  ms[4] / count[4]: 0 = EKF tick, 1 = stage assembly, 2 = window solve (full sweep, one-stage incremental
 * step, KF step, constrained solve or the fused kernel), 3 = incremental re-sweep on a VO tick (k_solve_incr_tma).
 * Reading synchronises the stream and clears the accumulators. */
int dekf_profile_enable(dekf_handle *h, int32_t enable);
int dekf_profile_read(dekf_handle *h, double *ms /*[4]*/, int64_t *count /*[4]*/);
/* Incremental solve bookkeeping of the last tick (device pointers, either may be NULL): stages re-swept per instance
 * (1 on a tick without VO bounds) and how many of them carry a VO row -- the operands of the algorithmic flop tally. */
int dekf_get_resweep_info(dekf_handle *h, int32_t *depth /*[n]*/, int32_t *n_vo /*[n]*/);

/* Roofline denominators measured on the device (the driver's MEASURED_PEAKS.json has no FP64/FP32 FMA figure):
 * dense non-tensor FMA throughput in TFLOP/s (FMA = 2 flop) and a device-to-device copy in GB/s (read+write). */
int dekf_measure_fma_peak(int32_t device, int32_t precision, double *tflops);
int dekf_measure_copy_bw(int32_t device, double *gbs);

/* General inequality rows on the window states: lb[i] <= a[i] . x_k <= ub[i] for EVERY state x_k of the window, i < count.
 * Replaces MHEproblem::addConstraints(name, lb, ub) + a dependency row on x_k
 * (/root/reference/src/decentral_legged_est/src/MheSrb.cpp:58-68, :217-270 -- the mechanism the reference offers for state
 * constraints and never exercises).  `a` is [count][9] row-major over (p_s, v_s, accel bias), count <= 9 together with the component
 * bounds of dekf_config (v_box / x_box, which count as unit rows); all rows must be linearly independent, lb < ub.  Call after
 * dekf_create and before the first step (DEKF_ESTATE afterwards); est_type 0, leg_odom_type 0.  The window QP is then solved
 * exactly by the active-set iteration of the state-constrained solve in the basis y = W x whose first coordinates are the rows
 * (host arrays).  Repeated calls replace the rows. */
int dekf_add_state_rows(dekf_handle *h, int32_t count, const double *a /*[count][9]*/, const double *lb /*[count]*/,
                        const double *ub /*[count]*/);

/* State-constrained solve bookkeeping of the last step (device pointers, any may be NULL): factorisations used and
 * number of active bounds in the window, per instance.  DEKF_EINVAL unless the handle has v_box_enable. */
int dekf_get_qp_info(dekf_handle *h, int32_t *iters /*[n]*/, int32_t *n_active /*[n]*/);

/* Number of kernel launches issued by this handle so far (bench.py "gpu_launches"). */
int64_t dekf_launch_count(const dekf_handle *h);
/* Bytes of device memory held by the handle. */
int64_t dekf_device_bytes(const dekf_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* DEKF_B200_H */
