// MATH-DEBUG HARNESS, NOT A PRODUCT PATH.
// The smoothed window (mhe_window_smooth, csrc/estimator_core.cuh) of the host build: the MHE ticks of hostsim.cpp (EKF tick,
// stage assembly, full or incremental window solve; est_type 0, leg_odom_type 0, no state bounds) followed after every
// update(T >= 1) by what dekf_get_window computes -- from the checkpoint ring (incremental) or from the getter's own forward
// sweep into a scratch ring (full re-sweep).  Built only by tests/hostsim/pywindowsim.py into tests/hostsim/_build/.
#include "hostsim.cpp"

namespace {
template <typename T, typename Model>
void run_window(const dekf_config &cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                double *x_out, double *win_out) {
  Sim<T> sim(cfg);
  const MheConst<double> mc64 = make_mhe_const<double>(cfg);
  const int n = cfg.n_instances, N = sim.dm.N;
  const int nq = Model::NLEG * Model::NJ, nl = Model::NLEG;
  std::vector<T> scr;
  if (sim.mc.window_solve == 0) scr.resize((size_t)N * 54 * sim.dm.ns);
  std::vector<double> quat(4 * (size_t)n), vb(3 * (size_t)n);
  std::vector<uint8_t> contact((size_t)nl * n);
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
    in.quat = nullptr;
    Outputs out;
    std::memset(&out, 0, sizeof(out));
    out.quat = quat.data();
    out.x = x_out + (size_t)s * 9 * n;
    out.v_body = vb.data();
    out.contact = contact.data();
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
    if (s >= 1)
      for (int i = 0; i < n; ++i)
        mhe_window_smooth<T>(sim.mc, mc64, sim.dm, sim.b, scr.empty() ? nullptr : scr.data(), s, i,
                             win_out + (size_t)s * N * 9 * n, (size_t)n);
  }
}
}  // namespace

extern "C" {
// x_out [S][9][n], win_out [S][N][9][n] (rows K = min(T+1, N) and beyond, and all of tick 0, are left as they are)
int windowsim_run(const dekf_config *cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                  const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                  const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                  double *x_out, double *win_out) {
  if (cfg->robot != DEKF_ROBOT_GO1 || cfg->est_type != 0 || cfg->leg_odom_type != 0 || cfg->v_box_enable || cfg->x_box_mask)
    return -1;
  if (cfg->precision == DEKF_FP32)
    run_window<float, Go1Model<float>>(*cfg, S, gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat,
                                       vo_time_pre, vo_time_now, vo_rel_p, x_out, win_out);
  else
    run_window<double, Go1Model<double>>(*cfg, S, gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat,
                                         vo_time_pre, vo_time_now, vo_rel_p, x_out, win_out);
  return 0;
}
}
