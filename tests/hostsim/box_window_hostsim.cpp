// MATH-DEBUG HARNESS, NOT A PRODUCT PATH.
// The window of a state-constrained handle (box_window_serial, csrc/box_window.cuh) in the host build: the constrained ticks
// of hostsim.cpp (EKF tick, stage assembly, mhe_solve_box; general rows through hostsim_set_rows) followed after every
// update(T >= 1) by what dekf_get_constrained_window computes from the serial solve's scratch.  Built only by
// tests/hostsim/pyboxwindowsim.py into tests/hostsim/_build/.
#include "hostsim.cpp"
#include "../../decentralized_ekf_mhe_b200/csrc/box_window.cuh"

namespace {
template <typename T, typename Model>
void run_box_window(const dekf_config &cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                    const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                    const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                    const double *quat_in, double *x_out, int32_t *status_out, double *win_out, double *cov_out,
                    uint32_t *act_out, uint8_t *capped_out) {
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
    Outputs out;
    std::memset(&out, 0, sizeof(out));
    out.quat = quat.data();
    out.x = x_out + (size_t)s * 9 * n;
    out.v_body = vb.data();
    out.contact = contact.data();
    for (int i = 0; i < n; ++i) {
      int st = ekf_tick<T>(sim.ec, sim.dm, sim.b, in, out, s, i);
      double q[4];
      for (int f = 0; f < 4; ++f) q[f] = in.quat ? in.quat[(size_t)f * n + i] : (double)sim.b.ekf_q[(size_t)f * sim.dm.ns + i];
      st |= mhe_assemble<T, Model>(sim.mc, sim.dm, sim.b, in, out, s, i, q);
      if (s >= 1) st |= mhe_solve_box<T>(sim.mc, sim.bc, sim.dm, sim.b, sim.bb, in, out, s, i);
      status_out[(size_t)s * n + i] = st;
    }
    if (s < 1) continue;
    for (int i = 0; i < n; ++i) {
      box_window_serial<true>(sim.bc, sim.dm, sim.bb, lay, s, i, win_out + (size_t)s * N * 9 * n + i,
                              cov_out + (size_t)s * N * 81 * n + i, act_out + (size_t)s * N * n + i, (size_t)n);
      capped_out[(size_t)s * n + i] = capped[i];
    }
  }
}
}  // namespace

extern "C" {
// est_type 0, leg_odom_type 0, a config with state constraints (or rows set by hostsim_set_rows).  x_out [S][9][n] (the step's
// x_T), status_out [S][n]; win_out [S][N][9][n], cov_out [S][N][81][n], act_out [S][N][n]: the window after every update (rows K
// and beyond, and tick 0, are left as they are); capped_out [S][n]: the solve's iteration-cap byte.
int boxwinsim_run(const dekf_config *cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                  const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                  const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                  const double *quat_in, double *x_out, int32_t *status_out, double *win_out, double *cov_out, uint32_t *act_out,
                  uint8_t *capped_out) {
  if (cfg->est_type != 0 || cfg->leg_odom_type != 0) return -1;
  if (!make_box_const(*cfg).enable && g_rows == 0) return -1;
#define BW_ARGS *cfg, S, gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat, vo_time_pre, vo_time_now, \
                vo_rel_p, quat_in, x_out, status_out, win_out, cov_out, act_out, capped_out
  const bool f32 = cfg->precision == DEKF_FP32;
  switch (cfg->robot) {
    case DEKF_ROBOT_GO1:
      if (f32) run_box_window<float, Go1Model<float>>(BW_ARGS); else run_box_window<double, Go1Model<double>>(BW_ARGS);
      return 0;
    case DEKF_ROBOT_CASSIE:
      if (f32) run_box_window<float, CassieModel<float>>(BW_ARGS); else run_box_window<double, CassieModel<double>>(BW_ARGS);
      return 0;
    case DEKF_ROBOT_POGOX:
      if (f32) run_box_window<float, PogoXModel<float>>(BW_ARGS); else run_box_window<double, PogoXModel<double>>(BW_ARGS);
      return 0;
  }
  return -1;
}
}
