// MATH-DEBUG HARNESS, NOT A PRODUCT PATH.
// The lag-one cross-covariances of the window (dekf_get_window_cross_cov) in the host build, for the three handle kinds: the
// ticks of hostsim.cpp (EKF tick, stage assembly and the kind's solve) followed after every update(T >= 1) by the serial
// form of the kind's backward covariance pass with the cross block switched on -- mhe_window_cov<T, true>
// (estimator_core.cuh), foot_window_smooth (footstate.cuh) and box_window_serial (box_window.cuh), the header functions
// the device runs.  The tick loops are those of window_cov_hostsim.cpp, foot_window_hostsim.cpp and box_window_hostsim.cpp.
// Built only by tests/hostsim/pywindowcrosssim.py into tests/hostsim/_build/.
#include "hostsim.cpp"
#include "../../decentralized_ekf_mhe_b200/csrc/box_window.cuh"

namespace {
// the inputs of tick s and the outputs the tick writes (x at x_out + s ds n)
void tick_io(int s, int n, int nq, int nl, int ds, const double *gyro, const double *accel, const double *imu_time,
             const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
             const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
             const double *quat_in, double *x_out, double *quat, double *vb, uint8_t *contact, Inputs &in, Outputs &out) {
  in.gyro = gyro + (size_t)s * 3 * n;
  in.accel = accel + (size_t)s * 3 * n;
  in.imu_time = imu_time + (size_t)s * n;
  in.joint_pos = joint_pos + (size_t)s * nq * n;
  in.joint_vel = joint_vel + (size_t)s * nq * n;
  in.foot_force = foot_force + (size_t)s * nl * n;
  in.vo_flag = vo_flag ? vo_flag + (size_t)s * n : nullptr;
  in.vo_quat = vo_quat + (size_t)s * 4 * n;
  in.vo_time_pre = vo_time_pre + (size_t)s * n;
  in.vo_time_now = vo_time_now + (size_t)s * n;
  in.vo_rel_p = vo_rel_p + (size_t)s * 3 * n;
  in.quat = quat_in ? quat_in + (size_t)s * 4 * n : nullptr;
  std::memset(&out, 0, sizeof(out));
  out.quat = quat;
  out.x = x_out + (size_t)s * ds * n;
  out.v_body = vb;
  out.contact = contact;
}

#define XS_IN gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat, vo_time_pre, vo_time_now, vo_rel_p
#define XS_PARAMS                                                                                                          \
  const double *gyro, const double *accel, const double *imu_time, const double *joint_pos, const double *joint_vel,     \
      const double *foot_force, const uint8_t *vo_flag, const double *vo_quat, const double *vo_time_pre,               \
      const double *vo_time_now, const double *vo_rel_p

// 9-state handles: cov_out [S][N][81][n], cross_out [S][N-1][81][n]
template <typename T, typename Model>
void run_nine(const dekf_config &cfg, int S, XS_PARAMS, double *x_out, double *cov_out, double *cross_out) {
  Sim<T> sim(cfg);
  const MheConst<double> mc64 = make_mhe_const<double>(cfg);
  const int n = cfg.n_instances, N = sim.dm.N;
  const int nq = Model::NLEG * Model::NJ, nl = Model::NLEG;
  std::vector<T> scr;
  if (sim.mc.window_solve == 0) scr.resize((size_t)N * 54 * sim.dm.ns);
  std::vector<double> quat(4 * (size_t)n), vb(3 * (size_t)n);
  std::vector<uint8_t> contact((size_t)nl * n);
  double sh[126];  // the kernel's per-thread shared-memory area, here at stride 1
  for (int s = 0; s < S; ++s) {
    Inputs in;
    Outputs out;
    tick_io(s, n, nq, nl, 9, XS_IN, nullptr, x_out, quat.data(), vb.data(), contact.data(), in, out);
    for (int i = 0; i < n; ++i) {
      ekf_tick<T>(sim.ec, sim.dm, sim.b, in, out, s, i);
      double q[4];
      for (int f = 0; f < 4; ++f) q[f] = (double)sim.b.ekf_q[(size_t)f * sim.dm.ns + i];
      mhe_assemble<T, Model>(sim.mc, sim.dm, sim.b, in, out, s, i, q);
      if (s >= 1 && sim.mc.window_solve == 1)
        mhe_solve_incr<T>(sim.mc, sim.dm, sim.b, in, out, s, i);
      else if (s >= 1)
        mhe_solve<T>(sim.mc, sim.dm, sim.b, in, out, s, i);
    }
    if (s < 1) continue;
    for (int i = 0; i < n; ++i)
      mhe_window_cov<T, true>(sim.mc, mc64, sim.dm, sim.b, scr.empty() ? nullptr : scr.data(), s, i,
                              cov_out + (size_t)s * N * 81 * n, (size_t)n, sh, 1, cross_out + (size_t)s * (N - 1) * 81 * n, N);
  }
}

// foot-state handles: cov_out [S][N][DS*DS][n], cross_out [S][N-1][DS*DS][n]
template <typename Model>
void run_foot(const dekf_config &cfg, int S, XS_PARAMS, double *x_out, double *cov_out, double *cross_out) {
  constexpr int L = Model::NLEG, DS = 9 + 3 * L;
  Sim<double> sim(cfg);
  const int n = cfg.n_instances, N = sim.dm.N;
  const int nq = Model::NLEG * Model::NJ;
  std::vector<double> rec((size_t)N * FootWin<L>::W);
  std::vector<double> quat(4 * (size_t)n), vb(3 * (size_t)n);
  std::vector<uint8_t> contact((size_t)L * n);
  for (int s = 0; s < S; ++s) {
    Inputs in;
    Outputs out;
    tick_io(s, n, nq, L, DS, XS_IN, nullptr, x_out, quat.data(), vb.data(), contact.data(), in, out);
    for (int i = 0; i < n; ++i) {
      ekf_tick<double>(sim.ec, sim.dm, sim.b, in, out, s, i);
      double q[4];
      for (int f = 0; f < 4; ++f) q[f] = sim.b.ekf_q[(size_t)f * sim.dm.ns + i];
      mhe_assemble<double, Model>(sim.mc, sim.dm, sim.b, in, out, s, i, q);
      if (s >= 1) foot_solve<double, L>(sim.fc, sim.dm, sim.b, sim.fb, in, out, s, i);
    }
    if (s < 1) continue;
    for (int i = 0; i < n; ++i)
      foot_window_smooth<double, L>(sim.fc, sim.dm, sim.b, sim.fb, s, i, rec.data(), nullptr,
                                    cov_out + (size_t)s * N * DS * DS * n + i, (size_t)n,
                                    cross_out + (size_t)s * (N - 1) * DS * DS * n + i);
  }
}

// state-constrained handles (serial solve): cov_out [S][N][81][n], act_out [S][N][n], capped_out [S][n],
// cross_out [S][N-1][81][n]
template <typename T, typename Model>
void run_box(const dekf_config &cfg, int S, XS_PARAMS, const double *quat_in, double *x_out, double *cov_out, uint32_t *act_out,
             uint8_t *capped_out, double *cross_out) {
  Sim<T> sim(cfg);
  const int n = cfg.n_instances, N = sim.dm.N;
  const int nq = Model::NLEG * Model::NJ, nl = Model::NLEG;
  std::vector<uint8_t> capped(sim.dm.ns, 0);
  sim.bb.capped = capped.data();
  std::vector<double> quat(4 * (size_t)n), vb(3 * (size_t)n);
  std::vector<uint8_t> contact((size_t)nl * n);
  const BwLayout<true> lay = {sim.bb.fac, (size_t)sim.dm.ns, N};
  for (int s = 0; s < S; ++s) {
    Inputs in;
    Outputs out;
    tick_io(s, n, nq, nl, 9, XS_IN, quat_in, x_out, quat.data(), vb.data(), contact.data(), in, out);
    for (int i = 0; i < n; ++i) {
      ekf_tick<T>(sim.ec, sim.dm, sim.b, in, out, s, i);
      double q[4];
      for (int f = 0; f < 4; ++f) q[f] = in.quat ? in.quat[(size_t)f * n + i] : (double)sim.b.ekf_q[(size_t)f * sim.dm.ns + i];
      mhe_assemble<T, Model>(sim.mc, sim.dm, sim.b, in, out, s, i, q);
      if (s >= 1) mhe_solve_box<T>(sim.mc, sim.bc, sim.dm, sim.b, sim.bb, in, out, s, i);
    }
    if (s < 1) continue;
    for (int i = 0; i < n; ++i) {
      box_window_serial<true>(sim.bc, sim.dm, sim.bb, lay, s, i, nullptr, cov_out + (size_t)s * N * 81 * n + i,
                              act_out + (size_t)s * N * n + i, (size_t)n, cross_out + (size_t)s * (N - 1) * 81 * n + i);
      capped_out[(size_t)s * n + i] = capped[i];
    }
  }
}
}  // namespace

extern "C" {
// Go1, est_type 0, leg_odom_type 0, no state bounds.  Blocks K and beyond (K-1 for cross_out), and tick 0, are left as they are.
int crosssim_run_nine(const dekf_config *cfg, int S, XS_PARAMS, double *x_out, double *cov_out, double *cross_out) {
  if (cfg->robot != DEKF_ROBOT_GO1 || cfg->est_type != 0 || cfg->leg_odom_type != 0 || cfg->v_box_enable || cfg->x_box_mask)
    return -1;
  if (cfg->precision == DEKF_FP32)
    run_nine<float, Go1Model<float>>(*cfg, S, XS_IN, x_out, cov_out, cross_out);
  else
    run_nine<double, Go1Model<double>>(*cfg, S, XS_IN, x_out, cov_out, cross_out);
  return 0;
}
// est_type 0, leg_odom_type 1, fp64
int crosssim_run_foot(const dekf_config *cfg, int S, XS_PARAMS, double *x_out, double *cov_out, double *cross_out) {
  if (cfg->est_type != 0 || cfg->leg_odom_type != 1 || cfg->precision != DEKF_FP64) return -1;
  switch (cfg->robot) {
    case DEKF_ROBOT_GO1: run_foot<Go1Model<double>>(*cfg, S, XS_IN, x_out, cov_out, cross_out); return 0;
    case DEKF_ROBOT_CASSIE: run_foot<CassieModel<double>>(*cfg, S, XS_IN, x_out, cov_out, cross_out); return 0;
    case DEKF_ROBOT_POGOX: run_foot<PogoXModel<double>>(*cfg, S, XS_IN, x_out, cov_out, cross_out); return 0;
  }
  return -1;
}
// est_type 0, leg_odom_type 0, a config with state constraints (or rows set by hostsim_set_rows)
int crosssim_run_box(const dekf_config *cfg, int S, XS_PARAMS, const double *quat_in, double *x_out, double *cov_out,
                     uint32_t *act_out, uint8_t *capped_out, double *cross_out) {
  if (cfg->est_type != 0 || cfg->leg_odom_type != 0) return -1;
  if (!make_box_const(*cfg).enable && g_rows == 0) return -1;
  const bool f32 = cfg->precision == DEKF_FP32;
#define XS_BOX(M)                                                                                                          \
  (f32 ? run_box<float, M<float>>(*cfg, S, XS_IN, quat_in, x_out, cov_out, act_out, capped_out, cross_out)                \
       : run_box<double, M<double>>(*cfg, S, XS_IN, quat_in, x_out, cov_out, act_out, capped_out, cross_out))
  switch (cfg->robot) {
    case DEKF_ROBOT_GO1: XS_BOX(Go1Model); return 0;
    case DEKF_ROBOT_CASSIE: XS_BOX(CassieModel); return 0;
    case DEKF_ROBOT_POGOX: XS_BOX(PogoXModel); return 0;
  }
  return -1;
}
}
