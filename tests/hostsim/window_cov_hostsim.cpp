// MATH-DEBUG HARNESS, NOT A PRODUCT PATH.
// The smoothed covariances of the window (mhe_window_cov, csrc/estimator_core.cuh) of the host build: the MHE ticks of
// hostsim.cpp (EKF tick, stage assembly, full or incremental window solve; est_type 0, leg_odom_type 0, no state bounds)
// followed after every update(T >= 1) by what dekf_get_window_cov computes -- from the checkpoint ring (incremental) or from
// the getter's own forward sweep into a scratch ring (full re-sweep).  The companion of window_hostsim.cpp for the covariance
// half of the backward pass.  Built only by tests/hostsim/pywindowcovsim.py into tests/hostsim/_build/.
#include "hostsim.cpp"

namespace {
template <typename T, typename Model>
void run_window_cov(const dekf_config &cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                    const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                    const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                    double *x_out, double *cov_out, double *filt_out) {
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
    if (s < 1) continue;
    if (sim.mc.window_solve == 1)
      for (int i = 0; i < n; ++i) {  // filtered P_T as the incremental sweep left it in the checkpoint ring, widened
        Cov9<double> P;
        Vec9<double> x;
        load_state_as(sim.b.ckpt + (size_t)(s % sim.dm.NW) * 54 * sim.dm.ns + i, (size_t)sim.dm.ns, P, x);
        for (int e = 0; e < 81; ++e) filt_out[((size_t)s * 81 + e) * n + i] = cov_at(P, e / 9, e % 9);
      }
    for (int i = 0; i < n; ++i)
      mhe_window_cov<T>(sim.mc, mc64, sim.dm, sim.b, scr.empty() ? nullptr : scr.data(), s, i, cov_out + (size_t)s * N * 81 * n,
                        (size_t)n, sh, 1);
  }
}
}  // namespace

extern "C" {
// x_out [S][9][n]; cov_out [S][N][81][n]: the smoothed covariances after every update (blocks K and beyond, and tick 0, are
// left as they are); filt_out [S][81][n]: incremental handles only, the filtered P_T of every update read from the
// checkpoint ring
int windowcovsim_run(const dekf_config *cfg, int S, const double *gyro, const double *accel, const double *imu_time,
                     const double *joint_pos, const double *joint_vel, const double *foot_force, const uint8_t *vo_flag,
                     const double *vo_quat, const double *vo_time_pre, const double *vo_time_now, const double *vo_rel_p,
                     double *x_out, double *cov_out, double *filt_out) {
  if (cfg->robot != DEKF_ROBOT_GO1 || cfg->est_type != 0 || cfg->leg_odom_type != 0 || cfg->v_box_enable || cfg->x_box_mask)
    return -1;
  if (cfg->precision == DEKF_FP32)
    run_window_cov<float, Go1Model<float>>(*cfg, S, gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat,
                                           vo_time_pre, vo_time_now, vo_rel_p, x_out, cov_out, filt_out);
  else
    run_window_cov<double, Go1Model<double>>(*cfg, S, gyro, accel, imu_time, joint_pos, joint_vel, foot_force, vo_flag, vo_quat,
                                             vo_time_pre, vo_time_now, vo_rel_p, x_out, cov_out, filt_out);
  return 0;
}
}
