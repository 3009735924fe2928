// MATH-DEBUG HARNESS, NOT A PRODUCT PATH.
// The smoothed window of the foot-state model (foot_window_smooth, csrc/footstate.cuh) in the host build: the foot ticks of
// hostsim.cpp (EKF tick, stage assembly, foot_solve; est_type 0, leg_odom_type 1) followed after every update(T >= 1) by
// what dekf_get_foot_window computes, and by the information matrix M_T of that update (the forward sweep of foot_solve
// once more) so that block K-1 can be checked against M_T^-1.  Built only by tests/hostsim/pyfootwindowsim.py into
// tests/hostsim/_build/.
#include "hostsim.cpp"

namespace {
template <typename Model>
void run_foot_window(const dekf_config &cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                     const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                     const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                     double *x_out, double *win_out, double *cov_out, double *info_out) {
  constexpr int L = Model::NLEG, DS = 9 + 3 * L;
  Sim<double> sim(cfg);
  const int n = cfg.n_instances, N = sim.dm.N;
  const int nq = Model::NLEG * Model::NJ;
  std::vector<double> rec((size_t)N * FootWin<L>::W);
  std::vector<double> quat(4 * (size_t)n), vb(3 * (size_t)n);
  std::vector<uint8_t> contact((size_t)L * n);
  for (int s = 0; s < S; ++s) {
    Inputs in;
    in.gyro = gyro + (size_t)s * 3 * n;
    in.accel = accel + (size_t)s * 3 * n;
    in.imu_time = imu_time + (size_t)s * n;
    in.joint_pos = joint_pos + (size_t)s * nq * n;
    in.joint_vel = joint_vel + (size_t)s * nq * n;
    in.foot_force = foot_force + (size_t)s * L * n;
    in.vo_flag = vo_flag ? vo_flag + (size_t)s * n : nullptr;
    in.vo_quat = vo_quat + (size_t)s * 4 * n;
    in.vo_time_pre = vo_time_pre + (size_t)s * n;
    in.vo_time_now = vo_time_now + (size_t)s * n;
    in.vo_rel_p = vo_rel_p + (size_t)s * 3 * n;
    in.quat = nullptr;
    Outputs out;
    std::memset(&out, 0, sizeof(out));
    out.quat = quat.data();
    out.x = x_out + (size_t)s * DS * n;
    out.v_body = vb.data();
    out.contact = contact.data();
    for (int i = 0; i < n; ++i) {
      ekf_tick<double>(sim.ec, sim.dm, sim.b, in, out, s, i);
      double q[4];
      for (int f = 0; f < 4; ++f) q[f] = sim.b.ekf_q[(size_t)f * sim.dm.ns + i];
      mhe_assemble<double, Model>(sim.mc, sim.dm, sim.b, in, out, s, i, q);
      if (s >= 1) foot_solve<double, L>(sim.fc, sim.dm, sim.b, sim.fb, in, out, s, i);
    }
    if (s < 1) continue;
    for (int i = 0; i < n; ++i) {
      foot_window_smooth<double, L>(sim.fc, sim.dm, sim.b, sim.fb, s, i, rec.data(), win_out + (size_t)s * N * DS * n + i,
                                    cov_out + (size_t)s * N * DS * DS * n + i, (size_t)n);
      // M_T: the sweep of foot_solve from the same arrival cost
      const size_t ns = (size_t)sim.dm.ns;
      const int K = s + 1 < N ? s + 1 : N, k0 = s - K + 1;
      FootFilter<L> f;
      auto leg = [&](int k) { return sim.fb.leg + (size_t)(k % sim.dm.NW) * foot_rec_size(L) * ns + i; };
      double R[9], as[3], dlt[3];
      bool vo;
      if (s >= N)
        f.load(sim.fb, ns, i);
      else
        f.set_prior(sim.fc, leg(0), ns);
      for (int k = k0;; ++k) {
        f.meas_update(leg(k), ns);
        if (k == s) break;
        foot_common(sim.dm, sim.b, k, i, R, as, dlt, vo);
        f.propagate(sim.fc, R, as, (int)leg(k)[(size_t)(9 * L) * ns], vo, dlt);
      }
      for (int e = 0; e < DS * DS; ++e) info_out[((size_t)s * DS * DS + e) * n + i] = f.M[e];
    }
  }
}
}  // namespace

extern "C" {
// x_out [S][DS][n] (foot_solve's x_T); win_out [S][N][DS][n] and cov_out [S][N][DS*DS][n]: the window after every update (rows
// K and beyond, and tick 0, are left as they are); info_out [S][DS*DS][n]: the information matrix M_T of every update
int footwinsim_run(const dekf_config *cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                   const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                   const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                   double *x_out, double *win_out, double *cov_out, double *info_out) {
  if (cfg->est_type != 0 || cfg->leg_odom_type != 1 || cfg->precision != DEKF_FP64) return -1;
#define FW_ARGS *cfg, S, gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat, vo_time_pre, vo_time_now, \
                vo_rel_p, x_out, win_out, cov_out, info_out
  switch (cfg->robot) {
    case DEKF_ROBOT_GO1: run_foot_window<Go1Model<double>>(FW_ARGS); return 0;
    case DEKF_ROBOT_CASSIE: run_foot_window<CassieModel<double>>(FW_ARGS); return 0;
    case DEKF_ROBOT_POGOX: run_foot_window<PogoXModel<double>>(FW_ARGS); return 0;
  }
  return -1;
}
}
