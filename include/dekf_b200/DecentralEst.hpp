// C++ facade over libdekf_b200.so with the reference's class names (header-only, C++17, no Eigen, no CUDA headers).
//
//   reference (under /root/reference/src/decentral_legged_est/)            here (namespace dekf)
//   struct robot_params   include/decentral_legged_est/DecentralEst.hpp:18-63   dekf::robot_params  (same field names)
//   struct robot_store    DecentralEst.hpp:65-94                                 dekf::robot_store   (same field names; every
//                                                                                 field gains a trailing instance axis)
//   class DecentralizedEstimation  DecentralEst.hpp:96-104, 278-291              dekf::DecentralizedEstimation
//        initialize(std::shared_ptr<robot_store>, std::shared_ptr<robot_params>) / update(int T) / reset()
//        public results R_sb_, p_vo_accmulate_, x_MHE_, v_MHE_b_
//   class MHEproblem::M_p, n_p    include/decentral_legged_est/MheSrb.hpp:86-87   dekf::DecentralizedEstimation::mhe_qp_.M_p()/n_p()
//   MHEproblem::solution (state blocks) MheSrb.hpp:58-112                          dekf::DecentralizedEstimation::mhe_qp_.x_window()
//   (posterior covariance of each state block, not in the reference)               dekf::DecentralizedEstimation::mhe_qp_.P_window()
//   (both for leg_odom_type 1: 9 + 3 num_legs rows per state block)                 the same, through dekf_get_foot_window
//   (both with state constraints, and the active bounds)                            the same and mhe_qp_.active_window(),
//                                                                                   through dekf_get_constrained_window
//   (lag-one cross-covariances of the state blocks, not in the reference)          mhe_qp_.P_window_cross(),
//                                                                                   through dekf_get_window_cross_cov
//
// The reference estimates ONE robot and stores Eigen vectors; this facade steps `n_instances` robots per call and stores
// flat SoA arrays `[rows][n_instances]` (instance fastest).  With n_instances == 1 every array has exactly the layout of the
// reference's Eigen member (Vector3d -> 3 doubles, quaternion -> w,x,y,z).
//
// Differences that are part of the boundary (INTEGRATION.md):
//   * robot_store carries the RAW joint message (positions, velocities, foot forces at rows nq.., go1Sub.cpp:68-75) --
//     contact flags, foot positions and Jacobians (go1Sub.cpp:74-121) are computed on the device, so `contact_`,
//     `p_imu_2_foot_`, `J_imu_2_foot_` are outputs here, not inputs.
//   * update() never throws for per-instance conditions; `status_` holds DEKF_ST_* bits (the reference prints and goes on).
//   * Errors of the library itself (no device, bad config) throw std::runtime_error from initialize(), like the reference's
//     FROST wrappers throw on size mismatch (go1_example/include/Expressions/math2mat.hpp:21-40).
#pragma once
#include <cstdint>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../dekf_b200.h"

namespace dekf {

struct robot_params {
  // ros params (DecentralEst.hpp:20-41, YAML names in EstSub.cpp:125-207)
  std::vector<double> p_process_std_, accel_input_std_, accel_bias_std_, gyro_input_std_;
  std::vector<double> quaternion_ib_, p_ib_;
  int num_legs_ = 4;
  int leg_odom_type_ = 0;
  std::vector<double> joint_position_std_, joint_velocity_std_, foot_slide_std_, foot_swing_std_;
  double contact_effort_theshold_ = 150.0;  // (sic) reference spelling
  std::vector<double> p_init_std_, v_init_std_, foot_init_std_, accel_bias_init_std_;
  std::vector<double> vo_p_std_;
  // estimator params (:44-46)
  int rate_ = 200, N_ = 20, est_type_ = 0;
  // osqp params (:49-61) -- accepted for source compatibility; the window is solved exactly (DESIGN.md 2)
  double rho_ = 0.1, alpha_ = 1.6, delta_ = 1e-5, sigma_ = 1e-5;
  bool verbose_ = false, adaptRho_ = true, polish_ = false;
  int maxQPIter_ = 4000;
  double realtiveTol_ = 1e-6, absTol_ = 1e-6, primTol_ = 1e-6, dualTol_ = 1e-6, timeLimit_ = 0.0028;
  // orien_ekf node parameters (orien_est/src/orien_ekf.cpp:13-18)
  std::vector<double> ekf_init_std_, ekf_process_std_, ekf_gravity_meas_std_, ekf_vo_meas_std_, ekf_quaternion_init_;
  int ekf_rate_ = 500;
  // batch / device (not in the reference)
  int robot_ = DEKF_ROBOT_GO1;
  int n_instances_ = 1, device_ = 0, precision_ = DEKF_FP64, ekf_hist_depth_ = 64;
  // state constraints lo <= v_s <= hi on every window state (what MHEproblem::addConstraints(name, lb, ub),
  // MheSrb.cpp:58-68, would add; never exercised by the reference)
  bool v_box_enable_ = false;
  std::vector<double> v_box_lo_{-1e30, -1e30, -1e30}, v_box_hi_{1e30, 1e30, 1e30};
  // lever arm of v_MHE_b_ (DecentralEst.cpp:181-185 hard-codes this Go1 mocap marker offset)
  std::vector<double> p_imu_2_opti_{0.016041, 0.089061, 0.0579875};
  bool kf_export_gain_ = false;  // est_type_ 1: make K_KF_() available (DecentralEst.hpp:290)
  // general rows lb <= x_k[a] <= ub on any state component a = 0..8 (MHEproblem::addConstraints with a selector row, MheSrb.cpp:58-68)
  int x_box_mask_ = 0;
  std::vector<double> x_box_lo_ = std::vector<double>(9, -1e30), x_box_hi_ = std::vector<double>(9, 1e30);

  // go1_example/config/parameters_go1.yaml
  static robot_params go1() {
    dekf_config c;
    dekf_config_default_go1(&c);
    return from_config(c);
  }
  static robot_params from_config(const dekf_config &c) {
    robot_params p;
    auto v = [](const double *a, int n) { return std::vector<double>(a, a + n); };
    p.p_process_std_ = v(c.p_process_std, 3);
    p.accel_input_std_ = v(c.accel_input_std, 3);
    p.accel_bias_std_ = v(c.accel_bias_std, 3);
    p.gyro_input_std_ = v(c.gyro_input_std, 3);
    p.quaternion_ib_ = v(c.quaternion_ib, 4);
    p.p_ib_ = v(c.p_ib, 3);
    p.num_legs_ = c.num_legs;
    p.leg_odom_type_ = c.leg_odom_type;
    p.joint_position_std_ = v(c.joint_position_std, 8);
    p.joint_velocity_std_ = v(c.joint_velocity_std, 8);
    p.foot_slide_std_ = v(c.foot_slide_std, 3);
    p.foot_swing_std_ = v(c.foot_swing_std, 3);
    p.contact_effort_theshold_ = c.contact_effort_threshold;
    p.p_init_std_ = v(c.p_init_std, 3);
    p.v_init_std_ = v(c.v_init_std, 3);
    p.foot_init_std_ = v(c.foot_init_std, 3);
    p.accel_bias_init_std_ = v(c.accel_bias_init_std, 3);
    p.vo_p_std_ = v(c.vo_p_std, 3);
    p.rate_ = c.rate;
    p.N_ = c.N;
    p.est_type_ = c.est_type;
    p.rho_ = c.rho;
    p.alpha_ = c.alpha;
    p.delta_ = c.delta;
    p.sigma_ = c.sigma;
    p.verbose_ = c.verbose != 0;
    p.adaptRho_ = c.adaptRho != 0;
    p.polish_ = c.polish != 0;
    p.maxQPIter_ = c.maxQPIter;
    p.realtiveTol_ = c.realtiveTol;
    p.absTol_ = c.absTol;
    p.primTol_ = c.primTol;
    p.dualTol_ = c.dualTol;
    p.timeLimit_ = c.timeLimit;
    p.ekf_init_std_ = v(c.ekf_init_std, 4);
    p.ekf_process_std_ = v(c.ekf_process_std, 3);
    p.ekf_gravity_meas_std_ = v(c.ekf_gravity_meas_std, 3);
    p.ekf_vo_meas_std_ = v(c.ekf_vo_meas_std, 4);
    p.ekf_quaternion_init_ = v(c.ekf_quaternion_init, 4);
    p.ekf_rate_ = c.ekf_rate;
    p.robot_ = c.robot;
    p.ekf_hist_depth_ = c.ekf_hist_depth;
    p.p_imu_2_opti_ = v(c.p_imu_2_opti, 3);
    p.kf_export_gain_ = c.kf_export_gain != 0;
    p.x_box_mask_ = c.x_box_mask;
    if (c.x_box_mask) {
      p.x_box_lo_ = v(c.x_box_lo, 9);
      p.x_box_hi_ = v(c.x_box_hi, 9);
    }
    p.v_box_enable_ = c.v_box_enable != 0;
    if (p.v_box_enable_) {
      p.v_box_lo_ = v(c.v_box_lo, 3);
      p.v_box_hi_ = v(c.v_box_hi, 3);
    }
    return p;
  }
  dekf_config to_config() const {
    dekf_config c;
    std::memset(&c, 0, sizeof(c));
    auto put = [](double *dst, const std::vector<double> &src, size_t n, const char *name) {
      if (src.size() < n && !(n == 8 && src.size() >= 3)) throw std::runtime_error(std::string("robot_params.") + name + " is too short");
      for (size_t i = 0; i < n; ++i) dst[i] = i < src.size() ? src[i] : src.back();
    };
    c.abi_version = DEKF_ABI_VERSION;
    c.n_instances = n_instances_;
    c.device = device_;
    c.precision = precision_;
    c.robot = robot_;
    c.ekf_hist_depth = ekf_hist_depth_;
    put(c.p_process_std, p_process_std_, 3, "p_process_std_");
    put(c.accel_input_std, accel_input_std_, 3, "accel_input_std_");
    put(c.accel_bias_std, accel_bias_std_, 3, "accel_bias_std_");
    put(c.gyro_input_std, gyro_input_std_, 3, "gyro_input_std_");
    put(c.quaternion_ib, quaternion_ib_, 4, "quaternion_ib_");
    put(c.p_ib, p_ib_, 3, "p_ib_");
    c.num_legs = num_legs_;
    c.leg_odom_type = leg_odom_type_;
    put(c.joint_position_std, joint_position_std_, 8, "joint_position_std_");  // reference: 3 per leg; padded
    put(c.joint_velocity_std, joint_velocity_std_, 8, "joint_velocity_std_");
    put(c.foot_slide_std, foot_slide_std_, 3, "foot_slide_std_");
    put(c.foot_swing_std, foot_swing_std_, 3, "foot_swing_std_");
    c.contact_effort_threshold = contact_effort_theshold_;
    put(c.p_init_std, p_init_std_, 3, "p_init_std_");
    put(c.v_init_std, v_init_std_, 3, "v_init_std_");
    put(c.foot_init_std, foot_init_std_, 3, "foot_init_std_");
    put(c.accel_bias_init_std, accel_bias_init_std_, 3, "accel_bias_init_std_");
    put(c.vo_p_std, vo_p_std_, 3, "vo_p_std_");
    c.rate = rate_;
    c.N = N_;
    c.est_type = est_type_;
    c.v_box_enable = v_box_enable_;
    put(c.v_box_lo, v_box_lo_, 3, "v_box_lo_");
    put(c.v_box_hi, v_box_hi_, 3, "v_box_hi_");
    put(c.p_imu_2_opti, p_imu_2_opti_, 3, "p_imu_2_opti_");
    c.kf_export_gain = kf_export_gain_;
    c.x_box_mask = x_box_mask_;
    if (x_box_lo_.size() < 9 || x_box_hi_.size() < 9) throw std::runtime_error("robot_params.x_box_lo_/x_box_hi_ need 9 entries");
    for (int a = 0; a < 9; ++a) {
      c.x_box_lo[a] = x_box_lo_[(size_t)a];
      c.x_box_hi[a] = x_box_hi_[(size_t)a];
    }
    c.rho = rho_;
    c.alpha = alpha_;
    c.delta = delta_;
    c.sigma = sigma_;
    c.verbose = verbose_;
    c.adaptRho = adaptRho_;
    c.polish = polish_;
    c.maxQPIter = maxQPIter_;
    c.realtiveTol = realtiveTol_;
    c.absTol = absTol_;
    c.primTol = primTol_;
    c.dualTol = dualTol_;
    c.timeLimit = timeLimit_;
    put(c.ekf_init_std, ekf_init_std_, 4, "ekf_init_std_");
    put(c.ekf_process_std, ekf_process_std_, 3, "ekf_process_std_");
    put(c.ekf_gravity_meas_std, ekf_gravity_meas_std_, 3, "ekf_gravity_meas_std_");
    put(c.ekf_vo_meas_std, ekf_vo_meas_std_, 4, "ekf_vo_meas_std_");
    put(c.ekf_quaternion_init, ekf_quaternion_init_, 4, "ekf_quaternion_init_");
    c.ekf_rate = ekf_rate_;
    return c;
  }
};

// Per-tick sensor snapshot of all instances (host arrays, `[rows][n]`).
struct robot_store {
  // IMU (DecentralEst.hpp:68-72)
  std::vector<double> imu_time_;   // [n]
  std::vector<double> accel_b_;    // [3][n]
  std::vector<double> angular_b_;  // [3][n]
  // Encoder & contact (:75-78): raw joint message, foot forces in the rows after the joints (go1Sub.cpp:68-75)
  std::vector<double> joint_states_position_;  // [nq + num_legs][n]
  std::vector<double> joint_states_velocity_;  // [nq][n]
  std::vector<uint8_t> contact_;               // [num_legs][n]  OUTPUT of update() (go1Sub.cpp:74)
  // VO (:84-88)
  std::vector<double> vo_time_pre_, vo_time_now_;  // [n]
  std::vector<uint8_t> vo_new_;                    // [n]; cleared by update() like DecentralEst.cpp:891
  std::vector<double> vo_p_body_pre_2_body_;       // [3][n]
  std::vector<double> vo_quaternion_;              // [4][n] w,x,y,z (consumed by orien_ekf)
  // Decentralized filter (:91): orientation from imu/filter, w,x,y,z
  std::vector<double> quaternion_;  // [4][n]

  void resize(int n, int nq, int num_legs) {
    imu_time_.assign(n, 0.0);
    accel_b_.assign(3 * (size_t)n, 0.0);
    angular_b_.assign(3 * (size_t)n, 0.0);
    joint_states_position_.assign((size_t)(nq + num_legs) * n, 0.0);
    joint_states_velocity_.assign((size_t)nq * n, 0.0);
    contact_.assign((size_t)num_legs * n, 0);
    vo_time_pre_.assign(n, 0.0);
    vo_time_now_.assign(n, 0.0);
    vo_new_.assign(n, 0);
    vo_p_body_pre_2_body_.assign(3 * (size_t)n, 0.0);
    vo_quaternion_.assign(4 * (size_t)n, 0.0);
    quaternion_.assign(4 * (size_t)n, 0.0);
    for (int i = 0; i < n; ++i) quaternion_[i] = vo_quaternion_[i] = 1.0;
  }
  bool any_vo() const {
    for (uint8_t f : vo_new_)
      if (f) return true;
    return false;
  }
};

namespace detail {
inline void check(int rc, dekf_handle *h, const char *what) {
  if (rc != DEKF_OK) throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + (h ? dekf_last_error(h) : ""));
}
inline int joints_per_leg(int robot) { return robot == DEKF_ROBOT_CASSIE ? 5 : 3; }
}  // namespace detail

class DecentralizedEstimation {
 public:
  DecentralizedEstimation() = default;
  DecentralizedEstimation(const DecentralizedEstimation &) = delete;
  DecentralizedEstimation &operator=(const DecentralizedEstimation &) = delete;
  ~DecentralizedEstimation() {
    if (h_) dekf_destroy(h_);
  }

  // Optional: create the device handle (allocations, first CUDA context use) ahead of time, e.g. in a node constructor, so that
  // the first timer tick is not the one that pays for it; initialize() with the same parameter object then only steps T = 0.
  void prepare(std::shared_ptr<robot_params> params_ptr) {
    create_handle(*params_ptr);
    prepared_for_ = params_ptr.get();
  }
  // DecentralEst.hpp:101, DecentralEst.cpp:9-150 (T == 0: prior, first measurement; no solve)
  void initialize(std::shared_ptr<robot_store> sub_ptr, std::shared_ptr<robot_params> params_ptr) {
    robot_sub_ptr_ = std::move(sub_ptr);
    params_ptr_ = std::move(params_ptr);
    if (h_ && prepared_for_ == params_ptr_.get()) {
      prepared_for_ = nullptr;  // a later initialize() starts from a fresh handle like the reference's re-initialisation
    } else {
      create_handle(*params_ptr_);
    }
    step(0);
  }
  // DecentralEst.hpp:102, DecentralEst.cpp:152-198
  void update(int T) {
    if (!h_) throw std::runtime_error("DecentralizedEstimation::update before initialize");
    step(T);
  }

 private:
  void create_handle(const robot_params &prm) {
    if (h_) {
      dekf_destroy(h_);
      h_ = nullptr;
    }
    const dekf_config cfg = prm.to_config();
    detail::check(dekf_create(&cfg, &h_), nullptr, "dekf_create");
    if (!rows_lb_.empty())
      detail::check(dekf_add_state_rows(h_, (int32_t)rows_lb_.size(), rows_a_.data(), rows_lb_.data(), rows_ub_.data()), h_,
                    "dekf_add_state_rows");
    n_ = cfg.n_instances;
    N_ = cfg.N;
    last_T_ = -1;
    nl_ = cfg.num_legs;
    nq_ = dekf_num_joints(h_);
    kf_ = cfg.est_type == 1;
    constrained_ = cfg.v_box_enable || cfg.x_box_mask || !rows_lb_.empty();
    ds_ = dekf_state_dim(h_);
    x_MHE_.assign(kf_ ? 0 : ds_ * (size_t)n_, 0.0);
    v_MHE_b_.assign(kf_ ? 0 : 3 * (size_t)n_, 0.0);
    x_KF_.assign(kf_ ? ds_ * (size_t)n_ : 0, 0.0);
    v_KF_b_.assign(kf_ ? 3 * (size_t)n_ : 0, 0.0);
    R_sb_.assign(9 * (size_t)n_, 0.0);
    p_vo_accmulate_.assign(3 * (size_t)n_, 0.0);
    status_.assign(n_, 0);
  }

 public:
  // General inequality rows  lb[i] <= a[i] . x_k <= ub[i]  on every window state -- what MHEproblem::addConstraints(name, lb, ub)
  // with a dependency row on x_k adds in the reference (MheSrb.cpp:58-68, :217-270; never exercised there).  `a` is [count][9]
  // row-major over (p_s, v_s, accel bias).  Call BEFORE initialize(): the rows are handed to the handle when it is created.
  void addStateRows(const std::vector<double> &a, const std::vector<double> &lb, const std::vector<double> &ub) {
    if (lb.size() != ub.size() || a.size() != 9 * lb.size()) throw std::runtime_error("addStateRows: a must be [count][9]");
    rows_a_ = a;
    rows_lb_ = lb;
    rows_ub_ = ub;
  }
  // DecentralEst.hpp:103
  void reset() {
    if (h_) detail::check(dekf_reset(h_), h_, "dekf_reset");
    last_T_ = -1;
  }

  // results (DecentralEst.hpp:278-285), `[rows][n]`
  std::vector<double> R_sb_;            // [9][n] row-major 3x3 per instance
  std::vector<double> p_vo_accmulate_;  // [3][n]
  std::vector<double> x_MHE_;           // [ds][n]  p_s, v_s, accel bias (, foot positions if leg_odom_type_ == 1)
  std::vector<double> v_MHE_b_;         // [3][n]
  // KF alternative, est_type_ == 1 (DecentralEst.hpp:286-291): filled instead of x_MHE_ / v_MHE_b_
  std::vector<double> x_KF_;            // [9][n]
  std::vector<double> v_KF_b_;          // [3][n]
  std::vector<double> C_KF_() const {   // [81][n] row-major 9x9 per instance
    std::vector<double> c((size_t)ds_ * ds_ * n_);
    detail::check(dekf_get_host(h_, DEKF_GET_ARRIVAL_COV, c.data()), h_, "dekf_get_host");
    return c;
  }
  std::vector<int32_t> status_;         // [n] DEKF_ST_* bits of the last update

  // MHEproblem::M_p / n_p (MheSrb.hpp:86-87) of every instance
  struct MheQp {
    DecentralizedEstimation *o;
    std::vector<double> M_p() const {
      std::vector<double> m((size_t)o->ds_ * o->ds_ * o->n_);
      detail::check(dekf_get_host(o->h_, DEKF_GET_ARRIVAL_M, m.data()), o->h_, "dekf_get_host");
      return m;
    }
    std::vector<double> n_p() const {
      std::vector<double> v((size_t)o->ds_ * o->n_);
      detail::check(dekf_get_host(o->h_, DEKF_GET_ARRIVAL_N, v.data()), o->h_, "dekf_get_host");
      return v;
    }
    // the state blocks of MHEproblem::solution (MheSrb.hpp:58-112) of the last update(T), T >= 1: the smoothed window
    // [K][ds][n], K = min(T+1, N), row j = stage T-K+1+j, row K-1 == x_MHE_ (dekf_get_window; foot-state handles, ds = 9 + 3L:
    // dekf_get_foot_window; handles with state constraints: the window QP's optimum, dekf_get_constrained_window)
    std::vector<double> x_window() const {
      const size_t ds = (size_t)o->ds_;
      std::vector<double> w((size_t)o->N_ * ds * o->n_);
      const int32_t sel = o->constrained_ ? DEKF_GET_BOX_WINDOW_X : (ds != 9 ? DEKF_GET_FOOT_WINDOW_X : DEKF_GET_WINDOW_X);
      detail::check(dekf_get_host(o->h_, sel, w.data()), o->h_, "dekf_get_host");
      const int K = o->last_T_ + 1 < o->N_ ? o->last_T_ + 1 : o->N_;
      w.resize((size_t)K * ds * o->n_);
      return w;
    }
    // posterior covariance of each state of that window (dekf_get_window_cov; foot-state handles: dekf_get_foot_window; handles
    // with state constraints: active bounds as equalities, dekf_get_constrained_window): [K][ds * ds][n], block j = stage
    // T-K+1+j, row-major over the state components
    std::vector<double> P_window() const {
      const size_t ds = (size_t)o->ds_;
      std::vector<double> P((size_t)o->N_ * ds * ds * o->n_);
      const int32_t sel = o->constrained_ ? DEKF_GET_BOX_WINDOW_P : (ds != 9 ? DEKF_GET_FOOT_WINDOW_P : DEKF_GET_WINDOW_P);
      detail::check(dekf_get_host(o->h_, sel, P.data()), o->h_, "dekf_get_host");
      const int K = o->last_T_ + 1 < o->N_ ? o->last_T_ + 1 : o->N_;
      P.resize((size_t)K * ds * ds * o->n_);
      return P;
    }
    // lag-one cross-covariances of that window, any est_type 0 handle (dekf_get_window_cross_cov): [(K-1) * ds * ds][n],
    // block j = Cov(x_{T-K+1+j}, x_{T-K+2+j}), row-major with rows over the earlier state (not symmetric)
    std::vector<double> P_window_cross() const {
      const size_t ds = (size_t)o->ds_;
      std::vector<double> C((size_t)(o->N_ > 1 ? o->N_ - 1 : 1) * ds * ds * o->n_);
      detail::check(dekf_get_host(o->h_, DEKF_GET_WINDOW_C, C.data()), o->h_, "dekf_get_host");
      const int K = o->last_T_ + 1 < o->N_ ? o->last_T_ + 1 : o->N_;
      C.resize((size_t)(K - 1) * ds * ds * o->n_);
      return C;
    }
    // active bounds of each state of that window (handles with state constraints, dekf_get_constrained_window): [K][n], bit a =
    // lower bound of row a active, bit 9 + a = upper bound
    std::vector<uint32_t> active_window() const {
      std::vector<uint32_t> a((size_t)o->N_ * o->n_);
      detail::check(dekf_get_host(o->h_, DEKF_GET_BOX_WINDOW_ACTIVE, a.data()), o->h_, "dekf_get_host");
      const int K = o->last_T_ + 1 < o->N_ ? o->last_T_ + 1 : o->N_;
      a.resize((size_t)K * o->n_);
      return a;
    }
  } mhe_qp_{this};

  dekf_handle *handle() const { return h_; }
  int n_instances() const { return n_; }

 private:
  void step(int T) {
    robot_store &st = *robot_sub_ptr_;
    dekf_inputs in;
    std::memset(&in, 0, sizeof(in));
    in.gyro = st.angular_b_.data();
    in.accel = st.accel_b_.data();
    in.imu_time = st.imu_time_.data();
    in.joint_pos = st.joint_states_position_.data();
    in.joint_vel = st.joint_states_velocity_.data();
    in.foot_force = st.joint_states_position_.data() + (size_t)nq_ * n_;  // go1Sub.cpp:74
    in.quat = st.quaternion_.data();
    if (st.any_vo()) {
      in.vo_flag = st.vo_new_.data();
      in.vo_time_pre = st.vo_time_pre_.data();
      in.vo_time_now = st.vo_time_now_.data();
      in.vo_rel_p = st.vo_p_body_pre_2_body_.data();
    }
    dekf_outputs out;
    std::memset(&out, 0, sizeof(out));
    out.x = kf_ ? x_KF_.data() : x_MHE_.data();
    out.v_body = kf_ ? v_KF_b_.data() : v_MHE_b_.data();
    st.contact_.resize((size_t)nl_ * n_);
    out.contact = st.contact_.data();
    out.status = status_.data();
    detail::check(dekf_mhe_step_host(h_, T, &in, &out), h_, "dekf_mhe_step_host");
    last_T_ = T;
    std::fill(st.vo_new_.begin(), st.vo_new_.end(), (uint8_t)0);  // robot_sub_ptr_->vo_new_ = false (DecentralEst.cpp:891)
    detail::check(dekf_get_host(h_, DEKF_GET_R_SB, R_sb_.data()), h_, "dekf_get_host");
    detail::check(dekf_get_host(h_, DEKF_GET_P_VO, p_vo_accmulate_.data()), h_, "dekf_get_host");
  }

  std::shared_ptr<robot_store> robot_sub_ptr_;
  std::shared_ptr<robot_params> params_ptr_;
  const robot_params *prepared_for_ = nullptr;  // prepare()
  std::vector<double> rows_a_, rows_lb_, rows_ub_;  // addStateRows()
  dekf_handle *h_ = nullptr;
  int n_ = 0, nl_ = 0, nq_ = 0;
  int N_ = 0, last_T_ = -1;  // horizon, T of the last update (window length of mhe_qp_.x_window())
  bool kf_ = false;
  bool constrained_ = false;  // v_box_enable, x_box_mask or addStateRows: the window comes from dekf_get_constrained_window
  int ds_ = 9;
};

}  // namespace dekf
