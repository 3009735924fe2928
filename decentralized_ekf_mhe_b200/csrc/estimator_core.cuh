// Per-instance estimator math: one estimator instance == one thread, all state in registers,
// every HBM array laid out SoA [field][instance] so that a warp touches full 256-byte lines.
//
// Reference path replaced (file:line under /root/reference/src):
//   orien_est/src/orien_ekf.cpp:77-89,108-228,270-357        -> ekf_tick()
//   go1_example/src/go1Sub.cpp:64-125 + Expressions/*.cc     -> mhe_assemble() (kinematics, contact)
//   decentral_legged_est/src/DecentralEst.cpp:353-583,864-985,987-1009, Spline/Bezier_simple.cpp
//                                                            -> mhe_assemble() (stage record, VO sync)
//   decentral_legged_est/src/MheSrb.cpp:272-349,475-723 (+OSQP) and DecentralEst.cpp:152-185
//                                                            -> mhe_solve() (marginalise + window solve)
//
// Algorithm of mhe_solve (DESIGN.md section 4): every row of the reference's QP is an equality with
// its own quadratically-penalised slack (or a free VO placeholder), so the QP is a linear-Gaussian
// smoothing problem and the only quantity read out is x_T (MheSrb.cpp:715-723).  x_T is therefore
// the mean of a forward Kalman sweep over the window started from the arrival cost; the arrival
// cost update (marginalizeQP) is exactly one stage of the same sweep.  The sweep is carried in
// COVARIANCE form (P, x) -- no 9x9 factorisation, only 3x3 inverses, and it stays accurate in fp32
// where the information form does not (SURVEY.md App. E).
#pragma once
#include <stdint.h>

#include "kinematics.cuh"
#include "smallmat.cuh"

namespace dekf {

// ------------------------------------------------------------------------------------------------
// layouts
// ------------------------------------------------------------------------------------------------
enum {
  REC_R = 0,     // 9  R_sb of the sample (row-major)
  REC_AS = 9,    // 3  a_s = R a_b + (0,0,-9.81)
  REC_LAM = 12,  // 6  Lambda = sum_i Q_meas,i (symmetric)          } sufficient statistic of the
  REC_ETA = 18,  // 3  eta    = sum_i Q_meas,i b_meas,i              } leg-odometry rows (H_i=[0 I 0])
  REC_DLT = 21,  // 3  VO displacement node_{k+1}-node_k (valid iff flag)
  REC_FLAG = 24, // 1  VO row of the stage is an equality (1) or still the free placeholder (0)
  REC_SIZE = 25  //    one record = one [25][128] TMA box per 128-instance tile
};
enum { EKF_HIST_FIELDS = 26 };  // gyro3 accel3 q4 P16 (time kept separately in double)

enum StatusBits {
  ST_EKF_VO_DROPPED = 1,     // "not storing enough imu info" (orien_ekf.cpp:178-183)
  ST_EKF_VO_NO_REPLAY = 2,   // rel <= 1: rollback without VO (orien_ekf.cpp:191, SURVEY.md fact 8)
  ST_EKF_HIST_OVERFLOW = 4,  // VO older than the device history ring (reference stacks are unbounded)
  ST_MHE_VO_DROPPED = 8,     // DecentralEst.cpp:898-904
  ST_MHE_VO_BOUNDED = 16,    // vo_to_be_processed_flag_ was set this step
  ST_NONFINITE = 32,
  ST_QP_MAXITER = 64         // constrained window solve: active set still changing at max_iter
};

template <typename T>
struct EkfConst {
  T dt;
  T Cg[3], Ca[3], Cvo[4];
  T g[3];
  T q0[4], P0[4];
};

template <typename T>
struct MheConst {
  T dt;
  T d1[3];   // dt^2 C_p + dt^4/4 C_accel       (pp block of Q_dyn^-1 before rotation)
  T d2[3];   // dt^3/2 C_accel                  (pv block)
  T d3[3];   // dt^2 C_accel                    (vv block)
  T cab[3];  // dt^2 C_accel_bias               (bb block)
  T cvo[3];  // vo_p_std^2                       (Q_cam^-1 before rotation)
  // the same four diagonals as (d[0], d[1]-d[0], d[2]-d[0]) for the two-term form R diag(d) R' = d0 I + e1 r1r1' + e2 r2r2'
  T n1[3], n2[3], n3[3], nvo[3];
  // version-4 sweep: C_accel and dt^2 C_p in the same (e0, e1-e0, e2-e0) form; the rotated noise blocks are
  // h^2, h dt, dt^2 times R C_accel R' (+ dt^2 R C_p R' on pp)
  T ae[3], pe[3];
  T cenc_v[8], cenc_p[8], cgy[3];
  T q_swing[3];
  T P0[9];   // prior covariance diag (p,v,b init std^2), prior mean 0
  T p_ib[3];
  T lever[3];  // p_imu_2_opti: v_body = R_sb (v_s + omega x lever), DecentralEst.cpp:181-185
  double thr;  // contact threshold, compared in double on the raw input (bit-exact)
  double dt_d;
  int N;
  int est_type;  // 0: MHE (DecentralEst.cpp:156-187), 1: KF alternative (:189-196, :592-861)
  int window_solve;  // 0: full window re-sweep every step (tier A), 1: incremental re-sweep from a checkpoint (tier B)
};

struct Dims {
  int n;   // number of instances == stride of every caller-owned (input / output) array
  int ns;  // stride of the handle-owned state arrays: n rounded up to the 128-instance tile of the TMA path
  int N;   // horizon
  int NW;  // window ring slots  = N + 1
  int HR;  // MHE history ring   = 4N + 1   (DecentralEst.cpp:963)
  int D;   // EKF history ring depth
  int tile0 = 0;  // first 128-instance tile of a k_solve_tma launch that covers only part of the batch (dekf_run)
};

template <typename T>
struct Buffers {
  // EKF state
  T *ekf_q;               // [4][n]
  T *ekf_P;               // [16][n]
  T *ekf_hist;            // [D][26][n]
  double *ekf_hist_time;  // [D][n]
  // MHE state
  T *arr_P;               // [45][n] arrival covariance (pp6 vv6 bb6 pv9 pb9 vb9)
  T *arr_x;               // [9][n]  arrival mean
  T *win;                 // [NW][25][ns]
  double *hist_time;      // [HR][n]
  double *hist_quat;      // [HR][4][n]
  double *wp;             // [12][n] last 4 accumulated-VO way points
  double *wp_time;        // [4][n]
  int32_t *wp_count;      // [n]
  double *p_vo;           // [3][n]
  uint8_t *pend_flag;     // [n]   VO message latched at T==0 (robot_store.vo_new_ stays true)
  double *pend;           // [5][n]
  int32_t *status;        // [n]
  // incremental window solve (window_solve == 1) only, else nullptr
  // leg_odom_type 1 (foot-position states, footstate.cuh) only, else nullptr
  double *foot_leg;       // [NW][9*legs+1][ns] per leg b_meas (3) + measurement covariance (6); contact bit mask
  T *ckpt;                // [NW][54][ns] filter state (P 45, x 9) of every window stage AFTER its leg-odometry update
  int32_t *resweep;       // [2][ns] earliest stage whose VO row changed at tick T (INT_MAX: none), slot = T & 1
};

// Per-tick scratch words are double-buffered by tick parity so that the assembly kernel of tick T+1 may run while the
// window solve of tick T is still in flight (dekf_run).
template <typename T>
DEKF_HD int32_t &tick_status(const Dims &dm, const Buffers<T> &b, int Tk, int i) { return b.status[(size_t)(Tk & 1) * dm.ns + i]; }
template <typename T>
DEKF_HD int32_t &tick_resweep(const Dims &dm, const Buffers<T> &b, int Tk, int i) { return b.resweep[(size_t)(Tk & 1) * dm.ns + i]; }

struct Inputs {
  const double *gyro, *accel, *imu_time, *joint_pos, *joint_vel, *foot_force;
  const uint8_t *vo_flag;
  const double *vo_quat, *vo_time_pre, *vo_time_now, *vo_rel_p;
  const double *quat;  // external orientation for the MHE ([4][n]); nullptr -> EKF state
};

struct Outputs {
  double *quat;      // [4][n]
  double *x;         // [9][n]
  double *v_body;    // [3][n]
  uint8_t *contact;  // [nlegs][n]
  // optional debug taps (may be nullptr)
  double *dbg_b_meas;  // [3*nlegs][n]
  double *dbg_Q_meas;  // [nlegs][6][n]  (symmetric 3x3 per leg)
  int32_t *dbg_vo;     // [8][n]: processed,i_pre,i_now,w0,i0,ins,num,disc0
  int32_t *dbg_ekf;    // [3][n]: cur, idx, nreplay
};

// ------------------------------------------------------------------------------------------------
// orientation EKF
// ------------------------------------------------------------------------------------------------
template <typename T>
struct EkfState {
  T q[4];
  T P[16];
};

// orien_ekf.cpp:108-123 (+ :214-228 Ohm, :270-294 W with its indexing bug, :353-357)
template <typename T>
DEKF_HD void ekf_predict(const EkfConst<T> &c, EkfState<T> &s, const T w[3]) {
  const T h = c.dt / T(2);
  // F = I + dt/2 * Ohm
  T F[16];
  F[0] = T(1);  F[1] = -h * w[0]; F[2] = -h * w[1]; F[3] = -h * w[2];
  F[4] = h * w[0];  F[5] = T(1);  F[6] = h * w[2];  F[7] = -h * w[1];
  F[8] = h * w[1];  F[9] = -h * w[2]; F[10] = T(1); F[11] = h * w[0];
  F[12] = h * w[2]; F[13] = h * w[1]; F[14] = -h * w[0]; F[15] = T(1);
  // W from the UN-propagated quaternion; rows 2/3 as the reference computes them:
  // row2 = (z, x, w), row3 = (-y, 0, 0)
  const T k = T(0.5) * c.dt;
  const T qw = s.q[0], qx = s.q[1], qy = s.q[2], qz = s.q[3];
  T W[12];
  W[0] = -k * qx; W[1] = -k * qy; W[2] = -k * qz;
  W[3] = k * qw;  W[4] = -k * qz; W[5] = k * qy;
  W[6] = k * qz;  W[7] = k * qx;  W[8] = k * qw;
  W[9] = -k * qy; W[10] = T(0);   W[11] = T(0);
  T qn[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) qn[r] = F[r * 4 + 0] * qw + F[r * 4 + 1] * qx + F[r * 4 + 2] * qy + F[r * 4 + 3] * qz;
  T FP[16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
      FP[r * 4 + cc] = F[r * 4 + 0] * s.P[0 * 4 + cc] + F[r * 4 + 1] * s.P[1 * 4 + cc] + F[r * 4 + 2] * s.P[2 * 4 + cc] +
                       F[r * 4 + 3] * s.P[3 * 4 + cc];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      T v = FP[r * 4 + 0] * F[cc * 4 + 0] + FP[r * 4 + 1] * F[cc * 4 + 1] + FP[r * 4 + 2] * F[cc * 4 + 2] +
            FP[r * 4 + 3] * F[cc * 4 + 3];
      v += W[r * 3 + 0] * c.Cg[0] * W[cc * 3 + 0] + W[r * 3 + 1] * c.Cg[1] * W[cc * 3 + 1] +
           W[r * 3 + 2] * c.Cg[2] * W[cc * 3 + 2];
      s.P[r * 4 + cc] = v;
    }
  const T nrm = sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
#pragma unroll
  for (int r = 0; r < 4; ++r) s.q[r] = qn[r] / nrm;
}

// orien_ekf.cpp:125-142 (+ :296-329)
template <typename T>
DEKF_HD void ekf_correct(const EkfConst<T> &c, EkfState<T> &s, const T a[3]) {
  const T w = s.q[0], x = s.q[1], y = s.q[2], z = s.q[3];
  const M3<T> R = quat_to_rot<T>(w, x, y, z);
  const V3<T> g = v3<T>(c.g[0], c.g[1], c.g[2]);
  const V3<T> a_hat = mul_t(R, g);
  T H[12];
  H[0] = g[0] * w + g[1] * z - g[2] * y;
  H[1] = g[0] * x + g[1] * y + g[2] * z;
  H[2] = -g[0] * y + g[1] * x - g[2] * w;
  H[3] = -g[0] * z + g[1] * w + g[2] * x;
  H[4] = -g[0] * z + g[1] * w + g[2] * x;
  H[5] = g[0] * y - g[1] * x + g[2] * w;
  H[6] = g[0] * x + g[1] * y + g[2] * z;
  H[7] = -g[0] * w - g[1] * z + g[2] * y;
  H[8] = g[0] * y - g[1] * x + g[2] * w;
  H[9] = g[0] * z - g[1] * w - g[2] * x;
  H[10] = g[0] * w + g[1] * z - g[2] * y;
  H[11] = g[0] * x + g[1] * y + g[2] * z;
#pragma unroll
  for (int i = 0; i < 12; ++i) H[i] = T(2) * H[i];
  const T rel = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]) / sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]);
  T PHt[12];  // 4x3
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc)
      PHt[r * 3 + cc] = s.P[r * 4 + 0] * H[cc * 4 + 0] + s.P[r * 4 + 1] * H[cc * 4 + 1] + s.P[r * 4 + 2] * H[cc * 4 + 2] +
                        s.P[r * 4 + 3] * H[cc * 4 + 3];
  M3<T> S;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      T v = H[r * 4 + 0] * PHt[0 * 3 + cc] + H[r * 4 + 1] * PHt[1 * 3 + cc] + H[r * 4 + 2] * PHt[2 * 3 + cc] +
            H[r * 4 + 3] * PHt[3 * 3 + cc];
      if (r == cc) v += rel * rel * c.Ca[r];
      S(r, cc) = v;
    }
  const M3<T> Si = inverse(S);
  T K[12];  // 4x3
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc)
      K[r * 3 + cc] = PHt[r * 3 + 0] * Si(0, cc) + PHt[r * 3 + 1] * Si(1, cc) + PHt[r * 3 + 2] * Si(2, cc);
  const T in0 = a[0] - a_hat[0], in1 = a[1] - a_hat[1], in2 = a[2] - a_hat[2];
  T qn[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) qn[r] = s.q[r] + (K[r * 3 + 0] * in0 + K[r * 3 + 1] * in1 + K[r * 3 + 2] * in2);
  T IKH[16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
      IKH[r * 4 + cc] = ((r == cc) ? T(1) : T(0)) -
                        (K[r * 3 + 0] * H[0 * 4 + cc] + K[r * 3 + 1] * H[1 * 4 + cc] + K[r * 3 + 2] * H[2 * 4 + cc]);
  T Pn[16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
      Pn[r * 4 + cc] = IKH[r * 4 + 0] * s.P[0 * 4 + cc] + IKH[r * 4 + 1] * s.P[1 * 4 + cc] + IKH[r * 4 + 2] * s.P[2 * 4 + cc] +
                       IKH[r * 4 + 3] * s.P[3 * 4 + cc];
#pragma unroll
  for (int i = 0; i < 16; ++i) s.P[i] = Pn[i];
  const T nrm = sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
#pragma unroll
  for (int r = 0; r < 4; ++r) s.q[r] = qn[r] / nrm;
}

// orien_ekf.cpp:144-154 (H = I4).  (P + C_vo) is SPD: K = P (P + C_vo)^-1 through an unrolled
// Cholesky instead of the reference's pivoted LU.
template <typename T>
DEKF_HD void ekf_vo_correct(const EkfConst<T> &c, EkfState<T> &s, const T qv[4]) {
  T L[16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) L[r * 4 + cc] = T(0.5) * (s.P[r * 4 + cc] + s.P[cc * 4 + r]) + ((r == cc) ? c.Cvo[r] : T(0));
  // in-place lower Cholesky
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    T d = L[j * 4 + j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= L[j * 4 + k] * L[j * 4 + k];
    d = sqrt(d);
    L[j * 4 + j] = d;
    const T id = T(1) / d;
#pragma unroll
    for (int i = j + 1; i < 4; ++i) {
      T v = L[i * 4 + j];
#pragma unroll
      for (int k = 0; k < j; ++k) v -= L[i * 4 + k] * L[j * 4 + k];
      L[i * 4 + j] = v * id;
    }
  }
  // K^T = S^-1 P^T : solve for each row r of P (as a column of P^T): K[r][:] = (S^-1 P[r][:]^T)^T
  T K[16];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    T y[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      T v = s.P[r * 4 + i];
#pragma unroll
      for (int k = 0; k < i; ++k) v -= L[i * 4 + k] * y[k];
      y[i] = v / L[i * 4 + i];
    }
#pragma unroll
    for (int i = 3; i >= 0; --i) {
      T v = y[i];
#pragma unroll
      for (int k = i + 1; k < 4; ++k) v -= L[k * 4 + i] * y[k];
      y[i] = v / L[i * 4 + i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) K[r * 4 + i] = y[i];
  }
  T in[4], qn[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) in[i] = qv[i] - s.q[i];
#pragma unroll
  for (int r = 0; r < 4; ++r) qn[r] = s.q[r] + (K[r * 4 + 0] * in[0] + K[r * 4 + 1] * in[1] + K[r * 4 + 2] * in[2] + K[r * 4 + 3] * in[3]);
  T Pn[16];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      T v = T(0);
#pragma unroll
      for (int k = 0; k < 4; ++k) v += (((r == k) ? T(1) : T(0)) - K[r * 4 + k]) * s.P[k * 4 + cc];
      Pn[r * 4 + cc] = v;
    }
#pragma unroll
  for (int i = 0; i < 16; ++i) s.P[i] = Pn[i];
  const T nrm = sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
#pragma unroll
  for (int r = 0; r < 4; ++r) s.q[r] = qn[r] / nrm;
}

// std::upper_bound over a ring of doubles: logical index j in [0,size) lives at slot
// ((first + j) mod ring); returns the first j whose time is > v.
DEKF_HD int ring_upper_bound(const double *times, int n, int i, int first, int size, int ring, double v) {
  int lo = 0, len = size;
  while (len > 0) {
    const int half = len >> 1;
    const int mid = lo + half;
    const double t = times[(size_t)((first + mid) % ring) * n + i];
    if (!(v < t)) {
      lo = mid + 1;
      len = len - half - 1;
    } else {
      len = half;
    }
  }
  return lo;
}

// One EKF timer tick for instance i at discrete time k (orien_ekf.cpp:77-89 + get_measurement
// :156-212).  Returns status bits.
// PART selects which half of the tick runs:
//   EKF_ALL     the whole tick
//   EKF_REPLAY  instance i HAS a VO pose: history push, rewind, VO correction, replay; the state goes back to ekf_q / ekf_P
//   EKF_UPDATE  history push unless the instance has a VO pose (EKF_REPLAY pushed it), then this tick's predict / correct.
//               On a tick without any VO pose (in.vo_flag == nullptr) this IS the whole tick, compiled without the replay code
//               (no spill frame): what dekf_run launches for large batches on such ticks.
// REPLAY + UPDATE perform the operations of EKF_ALL on the same operands (the state makes one round trip through memory); they
// serve the opt-in compaction of ragged VO arrival (DEKF_VO_COMPACT=1, DESIGN.md).
enum { EKF_ALL = 0, EKF_REPLAY = 1, EKF_UPDATE = 2 };
template <typename T, int PART = EKF_ALL>
DEKF_HD int ekf_tick(const EkfConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                     int k, int i) {
  const int n = dm.n, ns = dm.ns, D = dm.D;
  int status = 0;
  EkfState<T> s;
#pragma unroll
  for (int f = 0; f < 4; ++f) s.q[f] = b.ekf_q[(size_t)f * ns + i];
#pragma unroll
  for (int f = 0; f < 16; ++f) s.P[f] = b.ekf_P[(size_t)f * ns + i];
  T w[3], a[3];
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    w[f] = (T)in.gyro[(size_t)f * n + i];
    a[f] = (T)in.accel[(size_t)f * n + i];
  }
  const double t_imu = in.imu_time[i];
  const bool has_vo = in.vo_flag != nullptr && in.vo_flag[i];
  // push (state BEFORE this tick's update), :158-163
  if (PART != EKF_UPDATE || !has_vo) {
    T *h = b.ekf_hist + (size_t)(k % D) * EKF_HIST_FIELDS * ns + i;
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      h[(size_t)f * ns] = w[f];
      h[(size_t)(3 + f) * ns] = a[f];
    }
#pragma unroll
    for (int f = 0; f < 4; ++f) h[(size_t)(6 + f) * ns] = s.q[f];
#pragma unroll
    for (int f = 0; f < 16; ++f) h[(size_t)(10 + f) * ns] = s.P[f];
    b.ekf_hist_time[(size_t)(k % D) * ns + i] = t_imu;
  }
  int dbg_cur = -2, dbg_idx = -2, dbg_nr = -2;
  if (PART != EKF_UPDATE && has_vo) {
    const double vt = in.vo_time_now[i];
    T qv[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) qv[f] = (T)in.vo_quat[(size_t)f * n + i];
    const int size = (k + 1 < D) ? (k + 1) : D;
    const int first = k + 1 - size;  // discrete time of logical index 0
    const int ub = ring_upper_bound(b.ekf_hist_time, ns, i, first, size, D, vt);
    dbg_cur = k;
    dbg_nr = 0;
    if (ub == 0) {
      dbg_idx = -1;
      status |= (first > 0) ? ST_EKF_HIST_OVERFLOW : ST_EKF_VO_DROPPED;
    } else {
      const int idx = first + ub - 1;  // :186
      const int rel = k - idx;         // :187
      dbg_idx = idx;
      {
        const T *h = b.ekf_hist + (size_t)(idx % D) * EKF_HIST_FIELDS * ns + i;
#pragma unroll
        for (int f = 0; f < 4; ++f) s.q[f] = h[(size_t)(6 + f) * ns];
#pragma unroll
        for (int f = 0; f < 16; ++f) s.P[f] = h[(size_t)(10 + f) * ns];
      }
      if (rel <= 1) status |= ST_EKF_VO_NO_REPLAY;
      for (int j = 0; j < rel - 1; ++j) {  // :191
        const T *h = b.ekf_hist + (size_t)((idx + j) % D) * EKF_HIST_FIELDS * ns + i;
        T wj[3], aj[3];
#pragma unroll
        for (int f = 0; f < 3; ++f) {
          wj[f] = h[(size_t)f * ns];
          aj[f] = h[(size_t)(3 + f) * ns];
        }
        ekf_predict(c, s, wj);
        ekf_correct(c, s, aj);
        if (j == 0) ekf_vo_correct(c, s, qv);  // :197-202
        dbg_nr++;
      }
    }
  }
  if (PART != EKF_REPLAY) {
    ekf_predict(c, s, w);  // :82
    ekf_correct(c, s, a);  // :83
  }
#pragma unroll
  for (int f = 0; f < 4; ++f) b.ekf_q[(size_t)f * ns + i] = s.q[f];
#pragma unroll
  for (int f = 0; f < 16; ++f) b.ekf_P[(size_t)f * ns + i] = s.P[f];
  if (PART != EKF_REPLAY && out.quat != nullptr) {
#pragma unroll
    for (int f = 0; f < 4; ++f) out.quat[(size_t)f * n + i] = (double)s.q[f];
  }
  if (out.dbg_ekf != nullptr) {
    out.dbg_ekf[(size_t)0 * n + i] = dbg_cur;
    out.dbg_ekf[(size_t)1 * n + i] = dbg_idx;
    out.dbg_ekf[(size_t)2 * n + i] = dbg_nr;
  }
  return status;
}

// ------------------------------------------------------------------------------------------------
// MHE: stage assembly (kinematics, contact, measurement statistic, VO synchronisation)
// ------------------------------------------------------------------------------------------------
// Bezier_simple.cpp:73-82, evaluation order kept
DEKF_HD void bezier_point(double out[3], double u, const double *P0, const double *P1, const double *P2, const double *P3) {
#pragma unroll
  for (int cdx = 0; cdx < 3; ++cdx) {
    double point = u * u * u * ((-1) * P0[cdx] + 3 * P1[cdx] - 3 * P2[cdx] + P3[cdx]);
    point += u * u * (3 * P0[cdx] - 6 * P1[cdx] + 3 * P2[cdx]);
    point += u * ((-3) * P0[cdx] + 3 * P1[cdx]);
    point += P0[cdx];
    out[cdx] = point;
  }
}

// stage data of the foot-state model (leg_odom_type 1, footstate.cuh) written by the assembly kernel:
// b_i = R p_i, Q_i = R (J_i C_enc_pos J_i')^-1 R' (DecentralEst.cpp:550-564), always double
template <typename T, int NJ>
DEKF_HD void foot_leg_record(const T *cenc_p, const M3<T> &R, const V3<T> &p, const T *J /*3 x NJ*/, double *rec /*stride ns*/,
                             size_t ns, int leg) {
  double Rd[9], pd[3], JC[3 * NJ];
  for (int f = 0; f < 9; ++f) Rd[f] = (double)R.a[f];
  for (int f = 0; f < 3; ++f) pd[f] = (double)p[f];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < NJ; ++c) JC[r * NJ + c] = (double)J[r * NJ + c] * (double)cenc_p[c];
  S3<double> JCJ;
  for (int r = 0; r < 3; ++r)
    for (int c = r; c < 3; ++c) {
      double v = 0.0;
      for (int k = 0; k < NJ; ++k) v += JC[r * NJ + k] * (double)J[c * NJ + k];
      JCJ.a[S3<double>::idx(r, c)] = v;
    }
  const S3<double> Qb = inverse(JCJ);
  M3<double> Rm;
  for (int f = 0; f < 9; ++f) Rm.a[f] = Rd[f];
  const S3<double> Qw = rsrt(Rm, Qb);
  double *o = rec + (size_t)(9 * leg) * ns;
  for (int r = 0; r < 3; ++r) o[(size_t)r * ns] = Rd[r * 3 + 0] * pd[0] + Rd[r * 3 + 1] * pd[1] + Rd[r * 3 + 2] * pd[2];
  for (int f = 0; f < 6; ++f) o[(size_t)(3 + f) * ns] = Qw.a[f];
}

// GetMeasurement(T) + the Measurement_T / Dynamic_T / VO_T data of UpdateMHE (DecentralEst.cpp:
// 374-424, 474-478, 496-572, 864-985) + UpdateVOConstraints (:987-1009) for instance i.
// q_ext: orientation to use ([w,x,y,z]); written to the history ring un-normalised like the reference
// stores R of the normalised quaternion.
// GetMeasurement(T), VO half (DecentralEst.cpp:883-945) + UpdateVOConstraints (:987-1009) for instance i: time synchronisation of
// the VO message against the history BEFORE this tick's sample is pushed, p_vo_accmulate_, the Bezier way points and the VO rows of
// the window stages the message bounds.  Touches nothing the orientation EKF or the leg kinematics of this tick produce -- except
// in the KF alternative at T == 0, which sees this tick's own sample (qd; may be null when est_type == 0).
template <typename T>
DEKF_HD int mhe_vo_sync(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out, int Tk, int i,
                        const double *qd) {
  const int n = dm.n, ns = dm.ns, N = dm.N, NW = dm.NW, HR = dm.HR;
  int status = 0;
  if (b.resweep != nullptr) tick_resweep(dm, b, Tk, i) = 0x7fffffff;

  // ---- VO synchronisation against the history BEFORE this sample is pushed (:883-945)
  int vo_new = (in.vo_flag != nullptr) ? (int)in.vo_flag[i] : 0;
  double t_pre = 0.0, t_now = 0.0, relp[3] = {0.0, 0.0, 0.0};
  if (vo_new) {
    t_pre = in.vo_time_pre[i];
    t_now = in.vo_time_now[i];
#pragma unroll
    for (int f = 0; f < 3; ++f) relp[f] = in.vo_rel_p[(size_t)f * n + i];
  }
  const bool kf = c.est_type == 1;
  if (kf) {
    // KF alternative: initialize() runs InitializeKF + UpdateKF (DecentralEst.cpp:139-141), i.e. GetMeasurement(0)
    // twice at T==0: the first call sees an empty stack (message stays latched, :884), the second one sees
    // [sample 0] and consumes it.  Every later call is GetMeasurement(0) too (:787), so w0 == stack size and no
    // VO bound is ever inserted; only p_vo_accmulate_ and the way points advance.
    if (Tk == 0) {
      b.hist_time[i] = in.imu_time[i];
#pragma unroll
      for (int f = 0; f < 4; ++f) b.hist_quat[(size_t)f * ns + i] = qd[f];
    }
  } else if (Tk == 0) {
    // stack is empty: the message stays latched in robot_store (vo_new_ remains true)
    b.pend_flag[i] = (uint8_t)vo_new;
    if (vo_new) {
      b.pend[(size_t)0 * ns + i] = t_pre;
      b.pend[(size_t)1 * ns + i] = t_now;
#pragma unroll
      for (int f = 0; f < 3; ++f) b.pend[(size_t)(2 + f) * ns + i] = relp[f];
    }
    vo_new = 0;
  } else if (Tk == 1 && !vo_new && b.pend_flag[i]) {
    vo_new = 1;
    t_pre = b.pend[(size_t)0 * ns + i];
    t_now = b.pend[(size_t)1 * ns + i];
#pragma unroll
    for (int f = 0; f < 3; ++f) relp[f] = b.pend[(size_t)(2 + f) * ns + i];
  }
  int dbg[8] = {-2, -2, -2, -2, -2, -2, -2, -2};
  if (vo_new) {
    // samples held: discrete times Tk-size .. Tk-1 (KF alternative at T==0: sample 0 itself, see above)
    const int size = (kf && Tk == 0) ? 1 : ((Tk < HR) ? Tk : HR);
    const int first = (kf && Tk == 0) ? 0 : Tk - size;
    dbg[0] = 0;
    const int ub = ring_upper_bound(b.hist_time, ns, i, first, size, HR, t_pre);  // :895
    if (ub == 0) {
      status |= ST_MHE_VO_DROPPED;  // :898-904
      dbg[1] = -1;
    } else {
      const int i_pre = ub - 1;  // :907
      const int i_now = ring_upper_bound(b.hist_time, ns, i, first, size, HR, t_now) - 1;  // :911-913
      // R_vo_sb_pre_ = R_input_rotation_stack_[i_pre]  (:909)
      const double *hq = b.hist_quat + (size_t)((first + i_pre) % HR) * 4 * ns + i;
      const M3<double> Rp = quat_to_rot<double>(hq[0], hq[(size_t)ns], hq[(size_t)2 * ns], hq[(size_t)3 * ns]);
      double pv[3];
#pragma unroll
      for (int f = 0; f < 3; ++f) {
        pv[f] = b.p_vo[(size_t)f * ns + i] + (Rp(f, 0) * relp[0] + Rp(f, 1) * relp[1] + Rp(f, 2) * relp[2]);  // :915
        b.p_vo[(size_t)f * ns + i] = pv[f];
      }
      const int w0 = kf ? size : size - ((N < Tk) ? N : Tk);  // :917 (KF alternative: GetMeasurement(0) -> min(N,0))
      const int i0 = (w0 > i_pre) ? w0 : i_pre;               // :918
      // :919 (the reference reads one past the end here in the KF alternative; the value is unused then)
      const double t_start = (i0 < size) ? b.hist_time[(size_t)((first + i0) % HR) * ns + i] : 0.0;
      const int disc0 = first + i0;                                             // :920
      // add_way_point (Bezier_simple.cpp:12-27): keep the last four
      int cnt = b.wp_count[i];
      double wp[4][3], wt[4];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        wt[p] = b.wp_time[(size_t)p * ns + i];
#pragma unroll
        for (int f = 0; f < 3; ++f) wp[p][f] = b.wp[(size_t)(p * 3 + f) * ns + i];
      }
      if (cnt < 4) {
#pragma unroll
        for (int p = 0; p < 4; ++p)
          if (p == cnt) {
            wt[p] = t_now;
#pragma unroll
            for (int f = 0; f < 3; ++f) wp[p][f] = pv[f];
          }
        cnt++;
      } else {
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          wt[p] = wt[p + 1];
#pragma unroll
          for (int f = 0; f < 3; ++f) wp[p][f] = wp[p + 1][f];
        }
        wt[3] = t_now;
#pragma unroll
        for (int f = 0; f < 3; ++f) wp[3][f] = pv[f];
      }
      b.wp_count[i] = cnt;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        b.wp_time[(size_t)p * ns + i] = wt[p];
#pragma unroll
        for (int f = 0; f < 3; ++f) b.wp[(size_t)(p * 3 + f) * ns + i] = wp[p][f];
      }
      dbg[0] = 1;
      dbg[1] = i_pre;
      dbg[2] = i_now;
      dbg[3] = w0;
      dbg[4] = i0;
      if (i_now > w0 && cnt >= 4) {  // :925
        const int ins = i0 - w0;         // :927
        const int num = i_now - i0 + 1;  // :928
        dbg[5] = ins;
        dbg[6] = num;
        dbg[7] = disc0;
        status |= ST_MHE_VO_BOUNDED;
        if (b.resweep != nullptr) tick_resweep(dm, b, Tk, i) = disc0;
        // set_interval + interpolate_waypoint (Bezier_simple.cpp:29-71) + UpdateVOConstraints
        const double t_interval = wt[3] - wt[0];
        const double u_inc = c.dt_d / t_interval;
        const double u0 = (t_start - wt[0]) / t_interval;
        double node_pre[3];
        bezier_point(node_pre, u0 + u_inc * 0.0, wp[0], wp[1], wp[2], wp[3]);
        for (int j = 1; j < num; ++j) {
          double node[3];
          bezier_point(node, u0 + u_inc * (double)j, wp[0], wp[1], wp[2], wp[3]);
          const int d = disc0 + j - 1;  // VO_measurement_{disc0 + (j-1)}  (:1004)
          T *rec = b.win + (size_t)(d % NW) * REC_SIZE * ns + i;
#pragma unroll
          for (int f = 0; f < 3; ++f) {
            rec[(size_t)(REC_DLT + f) * ns] = (T)(node[f] - node_pre[f]);
            node_pre[f] = node[f];
          }
          rec[(size_t)REC_FLAG * ns] = T(1);
        }
      }
    }
  }
  if (out.dbg_vo != nullptr) {
#pragma unroll
    for (int f = 0; f < 8; ++f) out.dbg_vo[(size_t)f * n + i] = dbg[f];
  }

  return status;
}

// Per-leg statistic of the leg-odometry rows (go1Sub.cpp:64-125 kinematics, DecentralEst.cpp:509-546): foot position p in the IMU
// frame, Jacobian J, beta = -(J dq + omega x p) (b_meas = R beta), Qb = (G C G')^-1 in the body frame and Qb beta.
template <typename T, typename Model>
DEKF_HD void leg_statistic(const MheConst<T> &c, int leg, const T *q, const T *dq, const V3<T> &om, V3<T> &p, T *J /*3 x NJ*/,
                           V3<T> &beta, S3<T> &Qb, V3<T> &Qbeta) {
  constexpr int NJ = Model::NJ;
  Model::leg_fk(leg, q, p, J);
  p[0] += c.p_ib[0];
  p[1] += c.p_ib[1];
  p[2] += c.p_ib[2];
  // beta = -(J dq + omega x p)   (b_meas = R beta, :515-516)
  V3<T> Jdq = v3<T>(T(0), T(0), T(0));
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    Jdq[0] += J[0 * NJ + j] * dq[j];
    Jdq[1] += J[1 * NJ + j] * dq[j];
    Jdq[2] += J[2 * NJ + j] * dq[j];
  }
  const V3<T> wxp = cross(om, p);
  beta = v3<T>(-(Jdq[0] + wxp[0]), -(Jdq[1] + wxp[1]), -(Jdq[2] + wxp[2]));
  // C_b = G C G', G = [-J, -omega^x J, p^x], C = blkdiag(C_enc_vel, C_enc_pos, C_gyro) (:523-543)
  S3<T> Cb;
#pragma unroll
  for (int f = 0; f < 6; ++f) Cb.a[f] = T(0);
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const V3<T> col = v3<T>(J[0 * NJ + j], J[1 * NJ + j], J[2 * NJ + j]);
    const V3<T> wc = cross(om, col);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc)
        Cb.a[S3<T>::idx(r, cc)] += c.cenc_v[j] * col[r] * col[cc] + c.cenc_p[j] * wc[r] * wc[cc];
  }
  {
    const M3<T> ps = skew(p);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc)
        Cb.a[S3<T>::idx(r, cc)] += c.cgy[0] * ps(r, 0) * ps(cc, 0) + c.cgy[1] * ps(r, 1) * ps(cc, 1) + c.cgy[2] * ps(r, 2) * ps(cc, 2);
  }
  Qb = inverse(Cb);
  Qbeta = mul(Qb, beta);
}

// Tail of GetMeasurement(T) + the Measurement_T / Dynamic_T data of UpdateMHE (DecentralEst.cpp:374-424, 474-478, 949-975): the
// leg sums become (Lambda, eta), the sample is pushed to the history ring and the stage record of discrete time Tk is written.
template <typename T>
DEKF_HD void mhe_push_sample(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, int Tk, int i, const double qd[4],
                             const M3<T> &R, const V3<T> &as, const S3<T> &Qb_sum, const V3<T> &Qbeta_sum, const V3<T> &beta_swing,
                             int n_swing, int contact_mask, int NL) {
  const int ns = dm.ns, NW = dm.NW, HR = dm.HR;
  // Lambda = R Qb_sum R' + n_swing diag(q_swing);  eta = R Qbeta_sum + diag(q_swing) R beta_swing
  S3<T> Lam = rsrt(R, Qb_sum);
  Lam.a[0] += (T)n_swing * c.q_swing[0];
  Lam.a[3] += (T)n_swing * c.q_swing[1];
  Lam.a[5] += (T)n_swing * c.q_swing[2];
  V3<T> eta = mul(R, Qbeta_sum);
  {
    const V3<T> Rb = mul(R, beta_swing);
    eta[0] += c.q_swing[0] * Rb[0];
    eta[1] += c.q_swing[1] * Rb[1];
    eta[2] += c.q_swing[2] * Rb[2];
  }

  if (b.foot_leg != nullptr) b.foot_leg[((size_t)(Tk % NW) * (9 * NL + 1) + 9 * NL) * ns + i] = (double)contact_mask;
  // ---- push (:949-975): history ring + stage record of discrete time Tk
  b.hist_time[(size_t)(Tk % HR) * ns + i] = in.imu_time[i];
#pragma unroll
  for (int f = 0; f < 4; ++f) b.hist_quat[((size_t)(Tk % HR) * 4 + f) * ns + i] = qd[f];
  {
    T *rec = b.win + (size_t)(Tk % NW) * REC_SIZE * ns + i;
#pragma unroll
    for (int f = 0; f < 9; ++f) rec[(size_t)(REC_R + f) * ns] = R.a[f];
#pragma unroll
    for (int f = 0; f < 3; ++f) rec[(size_t)(REC_AS + f) * ns] = as[f];
#pragma unroll
    for (int f = 0; f < 6; ++f) rec[(size_t)(REC_LAM + f) * ns] = Lam.a[f];
#pragma unroll
    for (int f = 0; f < 3; ++f) rec[(size_t)(REC_ETA + f) * ns] = eta[f];
#pragma unroll
    for (int f = 0; f < 3; ++f) rec[(size_t)(REC_DLT + f) * ns] = T(0);
    rec[(size_t)REC_FLAG * ns] = T(0);  // VO row of stage Tk starts as a free placeholder (:474-481)
  }
}

// HOIST: contact detection and the legs' joint samples are requested ahead of their use (k_assemble, large batches: 99.4 -> 98.6 us
// per tick at 65,536 instances); the single-warp fused tick is faster without it (53.1 vs 56.7 us), so k_fused passes false.
// VOSPLIT: the VO synchronisation of the instances that carry a message ran as its own launch over the compacted list of those
// instances (k_vo_sync; it left its status bits in the vo_stat scratch): here a flagged instance only picks those bits up, an
// unflagged one marks "no re-sweep" -- exactly what mhe_vo_sync does for it at T >= 2.
template <typename T, typename Model, bool HOIST = true, bool VOSPLIT = false>
DEKF_HD int mhe_assemble(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in,
                         const Outputs &out, int Tk, int i, const double qd[4], const int32_t *vo_stat = nullptr) {
  constexpr int NL = Model::NLEG, NJ = Model::NJ;
  const int n = dm.n, ns = dm.ns, NW = dm.NW;
  int status = 0;

  // ---- contact detection (go1Sub.cpp:74, exact) and the first leg's joint sample: requested up front so that the loads are in
  // flight during the VO synchronisation instead of stalling every pass of the (rolled) leg loop below
  int contact_mask = 0;
  T q_next[NJ], dq_next[NJ];
  if constexpr (HOIST) {
#pragma unroll
    for (int leg = 0; leg < NL; ++leg) {
      const bool contact = (in.foot_force[(size_t)leg * n + i] >= c.thr);
      if (out.contact != nullptr) out.contact[(size_t)leg * n + i] = contact ? 1 : 0;
      contact_mask |= (contact ? 1 : 0) << leg;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      q_next[j] = (T)in.joint_pos[(size_t)j * n + i];
      dq_next[j] = (T)in.joint_vel[(size_t)j * n + i];
    }
  }

  if constexpr (VOSPLIT) {
    if (in.vo_flag != nullptr && in.vo_flag[i])
      status |= vo_stat[i];
    else if (b.resweep != nullptr)
      tick_resweep(dm, b, Tk, i) = 0x7fffffff;
  } else {
    status |= mhe_vo_sync<T>(c, dm, b, in, out, Tk, i, qd);
  }

  // ---- current sample (:867-879)
  const M3<T> R = quat_to_rot<T>((T)qd[0], (T)qd[1], (T)qd[2], (T)qd[3]);
  V3<T> ab, om;
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    ab[f] = (T)in.accel[(size_t)f * n + i];
    om[f] = (T)in.gyro[(size_t)f * n + i];
  }
  V3<T> as = mul(R, ab);
  as[2] += T(-9.81);

  // ---- legs: contact, kinematics, leg-odometry statistic (go1Sub.cpp:64-125, DecentralEst.cpp:509-546)
  S3<T> Qb_sum;  // sum over stance legs of (G C G')^-1, body frame
#pragma unroll
  for (int f = 0; f < 6; ++f) Qb_sum.a[f] = T(0);
  V3<T> Qbeta_sum = v3<T>(T(0), T(0), T(0));  // sum over stance legs of (G C G')^-1 beta_i
  V3<T> beta_swing = v3<T>(T(0), T(0), T(0));  // sum over swing legs of beta_i
  int n_swing = 0;
  // The leg loop stays ROLLED: one copy of the kinematics / covariance code in the instruction stream instead of NL
  // (k_assemble<double, Go1>: 20.6 -> 18.8 us per launch, spill frame 104 -> 56 B; profiles/r02_tune_solve.md).
  // -DDEKF_LEG_UNROLLED restores the unrolled form.
#if defined(DEKF_LEG_UNROLLED)
#pragma unroll
#else
#pragma unroll 1
#endif
  for (int leg = 0; leg < NL; ++leg) {
    bool contact;
    T q[NJ], dq[NJ];
    if constexpr (HOIST) {
      contact = ((contact_mask >> leg) & 1) != 0;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        q[j] = q_next[j];
        dq[j] = dq_next[j];
      }
      if (leg + 1 < NL) {  // the next leg's joint sample travels while this leg is computed
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          q_next[j] = (T)in.joint_pos[(size_t)((leg + 1) * NJ + j) * n + i];
          dq_next[j] = (T)in.joint_vel[(size_t)((leg + 1) * NJ + j) * n + i];
        }
      }
    } else {
      contact = (in.foot_force[(size_t)leg * n + i] >= c.thr);  // go1Sub.cpp:74, exact
      if (out.contact != nullptr) out.contact[(size_t)leg * n + i] = contact ? 1 : 0;
      contact_mask |= (contact ? 1 : 0) << leg;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        q[j] = (T)in.joint_pos[(size_t)(leg * NJ + j) * n + i];
        dq[j] = (T)in.joint_vel[(size_t)(leg * NJ + j) * n + i];
      }
    }
    V3<T> p, beta, Qbeta;
    T J[3 * NJ];
    S3<T> Qb;
    leg_statistic<T, Model>(c, leg, q, dq, om, p, J, beta, Qb, Qbeta);
    if (b.foot_leg != nullptr)  // leg_odom_type 1: b_meas = R p, C_meas = R J C_enc_pos J' R' (:550-564)
      foot_leg_record<T, NJ>(c.cenc_p, R, p, J, b.foot_leg + (size_t)(Tk % NW) * (9 * NL + 1) * ns + i, (size_t)ns, leg);
    if (contact) {
#pragma unroll
      for (int f = 0; f < 6; ++f) Qb_sum.a[f] += Qb.a[f];
      Qbeta_sum = add(Qbeta_sum, Qbeta);
    } else {
      beta_swing = add(beta_swing, beta);
      n_swing++;
    }
    if (out.dbg_b_meas != nullptr) {
      const V3<T> bm = mul(R, beta);
#pragma unroll
      for (int f = 0; f < 3; ++f) out.dbg_b_meas[(size_t)(leg * 3 + f) * n + i] = (double)bm[f];
    }
    if (out.dbg_Q_meas != nullptr) {
      S3<T> Qw = rsrt(R, Qb);
      if (!contact) {
        Qw.a[0] = c.q_swing[0];
        Qw.a[1] = T(0);
        Qw.a[2] = T(0);
        Qw.a[3] = c.q_swing[1];
        Qw.a[4] = T(0);
        Qw.a[5] = c.q_swing[2];
      }
#pragma unroll
      for (int f = 0; f < 6; ++f) out.dbg_Q_meas[(size_t)(leg * 6 + f) * n + i] = (double)Qw.a[f];
    }
  }
  mhe_push_sample<T>(c, dm, b, in, Tk, i, qd, R, as, Qb_sum, Qbeta_sum, beta_swing, n_swing, contact_mask, NL);
  return status;
}

// ------------------------------------------------------------------------------------------------
// MHE: covariance-form window sweep
// ------------------------------------------------------------------------------------------------
template <typename T>
struct Cov9 {
  S3<T> pp, vv, bb;
  M3<T> pv, pb, vb;
};
template <typename T>
struct Vec9 {
  V3<T> p, v, b;
};

// The same 9-vector kept outside the register file (k_solve_tma's XS variant: one column of a [9][STRIDE] shared-memory
// array per thread).  Same member syntax as Vec9 (x.p[r], x.v[r], x.b[r]); every access is a shared-memory access.
template <typename T, int STRIDE>
struct MemV3 {
  T *q;
  DEKF_HD T &operator[](int i) { return q[i * STRIDE]; }
  DEKF_HD const T &operator[](int i) const { return q[i * STRIDE]; }
};
template <typename T, int STRIDE>
struct MemVec9 {
  MemV3<T, STRIDE> p, v, b;
  DEKF_HD explicit MemVec9(T *base) : p{base}, v{base + 3 * STRIDE}, b{base + 6 * STRIDE} {}
};

template <typename T>
DEKF_HD void load_cov(const T *base, int n, int i, Cov9<T> &P) {
#pragma unroll
  for (int f = 0; f < 6; ++f) {
    P.pp.a[f] = base[(size_t)f * n + i];
    P.vv.a[f] = base[(size_t)(6 + f) * n + i];
    P.bb.a[f] = base[(size_t)(12 + f) * n + i];
  }
#pragma unroll
  for (int f = 0; f < 9; ++f) {
    P.pv.a[f] = base[(size_t)(18 + f) * n + i];
    P.pb.a[f] = base[(size_t)(27 + f) * n + i];
    P.vb.a[f] = base[(size_t)(36 + f) * n + i];
  }
}
template <typename T>
DEKF_HD void store_cov(T *base, int n, int i, const Cov9<T> &P) {
#pragma unroll
  for (int f = 0; f < 6; ++f) {
    base[(size_t)f * n + i] = P.pp.a[f];
    base[(size_t)(6 + f) * n + i] = P.vv.a[f];
    base[(size_t)(12 + f) * n + i] = P.bb.a[f];
  }
#pragma unroll
  for (int f = 0; f < 9; ++f) {
    base[(size_t)(18 + f) * n + i] = P.pv.a[f];
    base[(size_t)(27 + f) * n + i] = P.pb.a[f];
    base[(size_t)(36 + f) * n + i] = P.vb.a[f];
  }
}

// Leg-odometry update of stage k: rows A_meas x_k - v_k = b_meas, cost 1/2 v' Q_meas v with
// A_meas = [0 I 0] per leg (DecentralEst.cpp:95-98, :575-581) == one 3-dim measurement of v_s with
// information Lambda and information vector eta.  P <- P - P_v W P_v', W = (Lambda^-1 + P_vv)^-1
// = (I + Lambda P_vv)^-1 Lambda  (never inverts Lambda: swing legs carry 1e-14).
template <typename T>
DEKF_HD void meas_update(Cov9<T> &P, Vec9<T> &x, const S3<T> &Lam, const V3<T> &eta) {
  const M3<T> Pvv = to_m3(P.vv);
  const M3<T> LamM = to_m3(Lam);
  M3<T> Z = mul(LamM, Pvv);
  Z(0, 0) += T(1);
  Z(1, 1) += T(1);
  Z(2, 2) += T(1);
  const M3<T> Zi = inverse(Z);
  const M3<T> W = mul(Zi, LamM);  // symmetric
  const V3<T> r = sub(eta, mul(Lam, x.v));
  const V3<T> t = mul(Zi, r);
  const M3<T> Kp = mul(P.pv, W);
  const M3<T> Kv = mul(Pvv, W);
  const M3<T> Kb = mul_tn(P.vb, W);
  x.p = add(x.p, mul(P.pv, t));
  x.v = add(x.v, mul(Pvv, t));
  x.b = add(x.b, mul_t(P.vb, t));
  // P -= K P_v'
  const S3<T> dpp = mul_nt_sym(Kp, P.pv);
  const M3<T> dpv = mul(Kp, Pvv);
  const M3<T> dpb = mul(Kp, P.vb);
  const M3<T> dvv = mul(Kv, Pvv);
  const M3<T> dvb = mul(Kv, P.vb);
  const M3<T> dbb = mul(Kb, P.vb);
#pragma unroll
  for (int f = 0; f < 6; ++f) P.pp.a[f] -= dpp.a[f];
#pragma unroll
  for (int f = 0; f < 9; ++f) {
    P.pv.a[f] -= dpv.a[f];
    P.pb.a[f] -= dpb.a[f];
    P.vb.a[f] -= dvb.a[f];
  }
  const S3<T> dvvs = upper(dvv), dbbs = upper(dbb);
#pragma unroll
  for (int f = 0; f < 6; ++f) {
    P.vv.a[f] -= dvvs.a[f];
    P.bb.a[f] -= dbbs.a[f];
  }
}

// Dynamics k -> k+1: rows A_k x_k - x_{k+1} - w_k = b_k with cost 1/2 w' Q_dyn w
// (DecentralEst.cpp:387-424, Q_dyn^-1 = blkdiag(G C G', dt^2 C_ab) in closed form, no 6x6 inverse)
// and, when the VO row of the stage has been made an equality (:1004-1005), the relative-position
// measurement  p_{k+1} - p_k = Delta_k + vcam,  cov(vcam) = R diag(vo_p_std^2) R' (:477).
template <typename T>
DEKF_HD void propagate(const MheConst<T> &c, Cov9<T> &P, Vec9<T> &x, const M3<T> &R, const V3<T> &as, bool vo,
                       const V3<T> &dlt) {
  const T dt = c.dt, h = T(0.5) * c.dt * c.dt;
  const S3<T> C1 = rdrt(R, v3<T>(c.d1[0], c.d1[1], c.d1[2]));
  const S3<T> C2 = rdrt(R, v3<T>(c.d2[0], c.d2[1], c.d2[2]));
  const S3<T> C3 = rdrt(R, v3<T>(c.d3[0], c.d3[1], c.d3[2]));
  const M3<T> RPbp = mul_nt(R, P.pb);  // R * P_bp
  const M3<T> RPbv = mul_nt(R, P.vb);  // R * P_bv
  const M3<T> RPbb = mul(R, P.bb);
  const V3<T> Rxb = mul(R, x.b);
  // mean shift of the position difference h(x) = p+ - p = dt v - h R b + h a_s
  const V3<T> hmean = v3<T>(dt * x.v[0] - h * Rxb[0] + h * as[0], dt * x.v[1] - h * Rxb[1] + h * as[1],
                            dt * x.v[2] - h * Rxb[2] + h * as[2]);
  M3<T> Up, Uv, Ub;
  S3<T> Sinn;
  if (vo) {
    // P L' with L = [0, dt I, -h R]
    const M3<T> Ep = mul_nt(P.pb, R);
    const M3<T> Ev = mul_nt(P.vb, R);
    const M3<T> Pvv = to_m3(P.vv);
    M3<T> PLp, PLv, PLb;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        PLp(r, cc) = dt * P.pv(r, cc) - h * Ep(r, cc);
        PLv(r, cc) = dt * Pvv(r, cc) - h * Ev(r, cc);
        PLb(r, cc) = dt * P.vb(cc, r) - h * RPbb(cc, r);
      }
    const M3<T> RPLb = mul(R, PLb);
    const M3<T> C1m = to_m3(C1), C2m = to_m3(C2);
    M3<T> Vh;
#pragma unroll
    for (int f = 0; f < 9; ++f) {
      Vh.a[f] = dt * PLv.a[f] - h * RPLb.a[f];
      Up.a[f] = PLp.a[f] + Vh.a[f] + C1m.a[f];
      Uv.a[f] = PLv.a[f] - dt * RPLb.a[f] + C2m.a[f];
      Ub.a[f] = PLb.a[f];
    }
    Sinn = add(add(upper(Vh), C1), rdrt(R, v3<T>(c.cvo[0], c.cvo[1], c.cvo[2])));
  }
  // time update P+ = A P A' + Q_dyn^-1, A = [[I, dt I, -h R],[0, I, -dt R],[0,0,I]]
  {
    const M3<T> Ppp = to_m3(P.pp), Pvv = to_m3(P.vv);
    M3<T> APpp, APpv, APpb, APvv, APvb;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        APpp(r, cc) = Ppp(r, cc) + dt * P.pv(cc, r) - h * RPbp(r, cc);
        APpv(r, cc) = P.pv(r, cc) + dt * Pvv(r, cc) - h * RPbv(r, cc);
        APpb(r, cc) = P.pb(r, cc) + dt * P.vb(r, cc) - h * RPbb(r, cc);
        APvv(r, cc) = Pvv(r, cc) - dt * RPbv(r, cc);
        APvb(r, cc) = P.vb(r, cc) - dt * RPbb(r, cc);
      }
    const M3<T> X = mul_nt(APpb, R);
    const M3<T> Y = mul_nt(APvb, R);
    M3<T> npp, nvv;
#pragma unroll
    for (int f = 0; f < 9; ++f) {
      npp.a[f] = APpp.a[f] + dt * APpv.a[f] - h * X.a[f];
      nvv.a[f] = APvv.a[f] - dt * Y.a[f];
    }
    const M3<T> C2m = to_m3(C2);
    P.pp = add(upper(npp), C1);
    P.vv = add(upper(nvv), C3);
#pragma unroll
    for (int f = 0; f < 9; ++f) {
      P.pv.a[f] = APpv.a[f] - dt * X.a[f] + C2m.a[f];
      P.pb.a[f] = APpb.a[f];
      P.vb.a[f] = APvb.a[f];
    }
    P.bb.a[0] += c.cab[0];
    P.bb.a[3] += c.cab[1];
    P.bb.a[5] += c.cab[2];
  }
  x.p = add(x.p, hmean);
  x.v = v3<T>(x.v[0] - dt * Rxb[0] + dt * as[0], x.v[1] - dt * Rxb[1] + dt * as[1], x.v[2] - dt * Rxb[2] + dt * as[2]);
  if (vo) {
    const S3<T> Si = inverse(Sinn);
    const M3<T> Kp = mul(Up, Si), Kv = mul(Uv, Si), Kb = mul(Ub, Si);
    const V3<T> nu = sub(dlt, hmean);
    x.p = add(x.p, mul(Kp, nu));
    x.v = add(x.v, mul(Kv, nu));
    x.b = add(x.b, mul(Kb, nu));
    const S3<T> dpp = mul_nt_sym(Kp, Up), dvv = mul_nt_sym(Kv, Uv), dbb = mul_nt_sym(Kb, Ub);
    const M3<T> dpv = mul_nt(Kp, Uv), dpb = mul_nt(Kp, Ub), dvb = mul_nt(Kv, Ub);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
      P.pp.a[f] -= dpp.a[f];
      P.vv.a[f] -= dvv.a[f];
      P.bb.a[f] -= dbb.a[f];
    }
#pragma unroll
    for (int f = 0; f < 9; ++f) {
      P.pv.a[f] -= dpv.a[f];
      P.pb.a[f] -= dpb.a[f];
      P.vb.a[f] -= dvb.a[f];
    }
  }
}

// ---- version 2 of the two sweep stages: same algebra as meas_update / propagate above, organised as in-place
// accumulations (every product term is one FMA on its destination block, short-lived temporaries only) --------------
template <typename T>
DEKF_HD void meas_update2(Cov9<T> &P, Vec9<T> &x, const S3<T> &Lam, const V3<T> &eta) {
  const M3<T> Pvv = to_m3(P.vv);
  M3<T> Z;  // I + Lam P_vv
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      T v = (r == c) ? T(1) : T(0);
      v += Lam(r, 0) * Pvv(0, c);
      v += Lam(r, 1) * Pvv(1, c);
      v += Lam(r, 2) * Pvv(2, c);
      Z(r, c) = v;
    }
  const M3<T> Zi = inverse(Z);
  M3<T> W;  // (Lam^-1 + P_vv)^-1 = Zi Lam, symmetric: upper triangle computed, mirrored
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = r; c < 3; ++c) {
      const T v = Zi(r, 0) * Lam(0, c) + Zi(r, 1) * Lam(1, c) + Zi(r, 2) * Lam(2, c);
      W(r, c) = v;
      W(c, r) = v;
    }
  V3<T> rr = eta;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    T v = rr[r];
    v -= Lam(r, 0) * x.v[0];
    v -= Lam(r, 1) * x.v[1];
    v -= Lam(r, 2) * x.v[2];
    rr[r] = v;
  }
  const V3<T> t = mul(Zi, rr);
  add_mul(x.p, P.pv, t);
  add_mul(x.v, Pvv, t);
  add_mul_t(x.b, P.vb, t);
  // P -= P_v W P_v',  P_v = [P_pv; P_vv; P_vb']  -- block rows in an order that lets every block be updated in place
  {
    const M3<T> Kp = mul(P.pv, W);
    sub_mul_nt_sym(P.pp, Kp, P.pv);
    sub_mul(P.pb, Kp, P.vb);
    sub_mul(P.pv, Kp, Pvv);
  }
  {
    const M3<T> G = mul(W, P.vb);
    sub_mul_tn_sym(P.bb, P.vb, G);
    sub_mul(P.vb, Pvv, G);
  }
  {
    const M3<T> Kv = mul(Pvv, W);
    sub_mul_sym(P.vv, Kv, Pvv);
  }
}

template <typename T>
DEKF_HD void propagate2(const MheConst<T> &c, Cov9<T> &P, Vec9<T> &x, const M3<T> &R, const V3<T> &as, bool vo,
                        const V3<T> &dlt) {
  const T dt = c.dt, h = T(0.5) * c.dt * c.dt;
  // mean: p+ = p + dt v + h (a_s - R b),  v+ = v + dt (a_s - R b)
  const V3<T> Rxb = mul(R, x.b);
  const V3<T> acc = sub(as, Rxb);
  const V3<T> hmean = v3<T>(dt * x.v[0] + h * acc[0], dt * x.v[1] + h * acc[1], dt * x.v[2] + h * acc[2]);
  // products with the bias blocks shared by the time update and the VO row
  const M3<T> Cv = mul_nt(P.vb, R);      // P_vb R'
  const M3<T> B = mul(R, to_m3(P.bb));   // R P_bb
  const S3<T> BR = mul_nt_sym(B, R);     // R P_bb R'
  M3<T> Cp = mul_nt(P.pb, R);            // P_pb R'  (old P_pb)
  const RotOuter<T> ro = rot_outer(R);
  const S3<T> C1 = rdrt2(ro, c.n1), C2 = rdrt2(ro, c.n2);
  M3<T> Up, Uv, Ub;
  S3<T> Sinn;
  if (vo) {
    // d = p+ - p = L x + (noise),  L = [0, dt I, -h R];  U = Cov(x+, d),  Sinn = Cov(d) + R diag(vo_p_std^2) R'
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        const T plp = dt * P.pv(r, cc) - h * Cp(r, cc);
        const T plv = dt * P.vv(r, cc) - h * Cv(r, cc);
        const T plb = dt * P.vb(cc, r) - h * B(cc, r);
        const T rplb = dt * Cv(cc, r) - h * BR(r, cc);  // (R PL_b)(r,cc)
        const T vh = dt * plv - h * rplb;
        Up(r, cc) = plp + vh + C1(r, cc);
        Uv(r, cc) = plv - dt * rplb + C2(r, cc);
        Ub(r, cc) = plb;
        if (r <= cc) Sinn.a[S3<T>::idx(r, cc)] = vh + C1(r, cc);
      }
    const S3<T> Cvo = rdrt2(ro, c.nvo);
#pragma unroll
    for (int f = 0; f < 6; ++f) Sinn.a[f] += Cvo.a[f];
  }
  // time update in place: A = A1 A2, A2: p += dt v, A1: p -= h R b, v -= dt R b
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = r; cc < 3; ++cc) {
      // P_pp += dt (P_pv' + P_pv_new),  P_pv_new = P_pv + dt P_vv
      const T s = P.pv(cc, r) + (P.pv(r, cc) + dt * P.vv(r, cc));
      P.pp.a[S3<T>::idx(r, cc)] += dt * s;
    }
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      P.pv(r, cc) += dt * P.vv(r, cc);
      P.pb(r, cc) += dt * P.vb(r, cc);
      Cp(r, cc) += dt * Cv(r, cc);  // (P_pb + dt P_vb) R'
    }
  const T hh = h * h, hdt = h * dt, dt2 = dt * dt;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = r; cc < 3; ++cc) {
      const int k = S3<T>::idx(r, cc);
      P.pp.a[k] += hh * BR.a[k] - h * (Cp(r, cc) + Cp(cc, r)) + C1.a[k];
      P.vv.a[k] += dt2 * BR.a[k] - dt * (Cv(r, cc) + Cv(cc, r));
    }
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      P.pv(r, cc) += hdt * BR(r, cc) - dt * Cp(r, cc) - h * Cv(cc, r) + C2(r, cc);
      P.pb(r, cc) -= h * B(r, cc);
      P.vb(r, cc) -= dt * B(r, cc);
    }
  {
    const S3<T> C3 = rdrt2(ro, c.n3);
#pragma unroll
    for (int f = 0; f < 6; ++f) P.vv.a[f] += C3.a[f];
  }
  P.bb.a[0] += c.cab[0];
  P.bb.a[3] += c.cab[1];
  P.bb.a[5] += c.cab[2];
  x.p = add(x.p, hmean);
  x.v = v3<T>(x.v[0] + dt * acc[0], x.v[1] + dt * acc[1], x.v[2] + dt * acc[2]);
  if (vo) {
    const S3<T> Si = inverse(Sinn);
    const M3<T> Sim = to_m3(Si);
    const V3<T> nu = sub(dlt, hmean);
    const V3<T> t = mul(Si, nu);
    add_mul(x.p, Up, t);
    add_mul(x.v, Uv, t);
    add_mul(x.b, Ub, t);
    {
      const M3<T> Kp = mul(Up, Sim);
      sub_mul_nt_sym(P.pp, Kp, Up);
      sub_mul_nt(P.pv, Kp, Uv);
      sub_mul_nt(P.pb, Kp, Ub);
    }
    {
      const M3<T> Kv = mul(Uv, Sim);
      sub_mul_nt_sym(P.vv, Kv, Uv);
      sub_mul_nt(P.vb, Kv, Ub);
    }
    {
      const M3<T> Kb = mul(Ub, Sim);
      sub_mul_nt_sym(P.bb, Kb, Ub);
    }
  }
}

// ---- version 3: version 1 with the determinant reciprocal taken off the critical path (products on the adjugate) ----
template <typename T>
DEKF_HD void meas_update3(Cov9<T> &P, Vec9<T> &x, const S3<T> &Lam, const V3<T> &eta) {
  const M3<T> Pvv = to_m3(P.vv);
  const M3<T> LamM = to_m3(Lam);
  M3<T> Z = mul(LamM, Pvv);
  Z(0, 0) += T(1);
  Z(1, 1) += T(1);
  Z(2, 2) += T(1);
  T det;
  const M3<T> Za = adjugate(Z, det);
  const T id = T(1) / det;
  const M3<T> Wu = mul(Za, LamM);
  const V3<T> r = sub(eta, mul(Lam, x.v));
  const V3<T> tu = mul(Za, r);
  const M3<T> W = scale(id, Wu);
  const V3<T> t = scale(id, tu);
  const M3<T> Kp = mul(P.pv, W);
  const M3<T> Kv = mul(Pvv, W);
  const M3<T> Kb = mul_tn(P.vb, W);
  x.p = add(x.p, mul(P.pv, t));
  x.v = add(x.v, mul(Pvv, t));
  x.b = add(x.b, mul_t(P.vb, t));
  const S3<T> dpp = mul_nt_sym(Kp, P.pv);
  const M3<T> dpv = mul(Kp, Pvv);
  const M3<T> dpb = mul(Kp, P.vb);
  const M3<T> dvv = mul(Kv, Pvv);
  const M3<T> dvb = mul(Kv, P.vb);
  const M3<T> dbb = mul(Kb, P.vb);
#pragma unroll
  for (int f = 0; f < 6; ++f) P.pp.a[f] -= dpp.a[f];
#pragma unroll
  for (int f = 0; f < 9; ++f) {
    P.pv.a[f] -= dpv.a[f];
    P.pb.a[f] -= dpb.a[f];
    P.vb.a[f] -= dvb.a[f];
  }
  const S3<T> dvvs = upper(dvv), dbbs = upper(dbb);
#pragma unroll
  for (int f = 0; f < 6; ++f) {
    P.vv.a[f] -= dvvs.a[f];
    P.bb.a[f] -= dbbs.a[f];
  }
}

// ---- version 4 (round 2): the sweep stages re-derived for the fewest FP64 instructions ----------------------------------
// Every multiply-add is an explicit fma (deterministic contraction: the full re-sweep, the incremental sweep and the host
// build of this header perform bit-identical operations).  Differences to versions 1-3:
//  * leg-odometry update through Z^-1 = (I + Lam P_vv)^-1 only:  P_vv+ = P_vv Z^-1,  P_vb+ = Z^-T P_vb,  P_pv+ = P_pv Z^-1,
//    P_pb+ = P_pb - P_pv G,  P_bb+ = P_bb - P_vb' G  with  G = Z^-1 (Lam P_vb)  -- no gain matrices K_v, K_b;
//    (Lam P_vb) and adj(Z) r do not depend on 1/det(Z) and overlap its latency.
//  * the accelerometer noise R C_a R' enters the time update only as an addend of R P_bb R' (Q_dyn^-1 = G C G' with
//    G = [h R; dt R], DecentralEst.cpp:409-418), so the three rotated noise blocks C1, C2, C3 cost one.
//  * the VO row re-uses the blocks of the time update: U_v = (P_pv+ - P_pv + dt P_pb R')', U_b = (P_pb+ - P_pb)',
//    U_p - PL_p = Cov(d) - C_vo = the increment of P_pp+.
//  * PP = false leaves P_pp untouched.  P_pp feeds nothing but itself (p is observed only through differences
//    p_{k+1} - p_k, whose statistics involve P_pv, P_pb alone), so the full re-sweep carries it through the first stage only,
//    where the arrival cost of the next tick is produced (marginalizeQP, MheSrb.cpp:475-713).
template <typename T>
DEKF_HD T fm(T a, T b, T c) { return a * b + c; }
#if defined(__CUDA_ARCH__)
template <>
DEKF_HD double fm<double>(double a, double b, double c) { return fma(a, b, c); }
template <>
DEKF_HD float fm<float>(float a, float b, float c) { return fmaf(a, b, c); }
#else
template <>
DEKF_HD double fm<double>(double a, double b, double c) { return ::fma(a, b, c); }
template <>
DEKF_HD float fm<float>(float a, float b, float c) { return ::fmaf(a, b, c); }
#endif

// R diag(e0, e0+e1, e0+e2) R' = e0 I + e1 r1 r1' + e2 r2 r2' added onto S (r1, r2: 2nd / 3rd column of R); branch-free
template <typename T>
DEKF_HD void add_rot_diag(S3<T> &S, const M3<T> &R, const T e[3]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const T s1 = e[1] * R(r, 1), s2 = e[2] * R(r, 2);
#pragma unroll
    for (int cc = r; cc < 3; ++cc)
      S.a[S3<T>::idx(r, cc)] = fm(s2, R(cc, 2), fm(s1, R(cc, 1), S.a[S3<T>::idx(r, cc)] + ((r == cc) ? e[0] : T(0))));
  }
}

// PPM selects how P_pp is carried: 0 not at all, 1 in P.pp (registers), 2 read-modify-written at ppm[f * pps] (f = 0..5)
// when ppm != nullptr (the first stage of the full re-sweep works directly on the arrival cost in HBM).
template <typename T>
DEKF_HD void pp_load(S3<T> &pp, const T *ppm, size_t pps) {
#pragma unroll
  for (int f = 0; f < 6; ++f) pp.a[f] = ppm[f * pps];
}
template <typename T>
DEKF_HD void pp_store(const S3<T> &pp, T *ppm, size_t pps) {
#pragma unroll
  for (int f = 0; f < 6; ++f) ppm[f * pps] = pp.a[f];
}

template <int PPM, typename T, typename X>
DEKF_HD void meas_update4(Cov9<T> &P, X &x, const S3<T> &Lam, const V3<T> &eta, T *ppm = nullptr, size_t pps = 0) {
  M3<T> Z;  // I + Lam P_vv
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c)
      Z(r, c) = fm(Lam(r, 2), P.vv(2, c), fm(Lam(r, 1), P.vv(1, c), fm(Lam(r, 0), P.vv(0, c), (r == c) ? T(1) : T(0))));
  T det;
  M3<T> Zi = adjugate(Z, det);
  const T id = T(1) / det;
  V3<T> rr;  // eta - Lam v
#pragma unroll
  for (int r = 0; r < 3; ++r) rr[r] = fm(-Lam(r, 2), x.v[2], fm(-Lam(r, 1), x.v[1], fm(-Lam(r, 0), x.v[0], eta[r])));
  M3<T> LP;  // Lam P_vb
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) LP(r, c) = fm(Lam(r, 2), P.vb(2, c), fm(Lam(r, 1), P.vb(1, c), Lam(r, 0) * P.vb(0, c)));
  V3<T> t;  // Z^-1 (eta - Lam v)
#pragma unroll
  for (int r = 0; r < 3; ++r) t[r] = fm(Zi(r, 2), rr[2], fm(Zi(r, 1), rr[1], Zi(r, 0) * rr[0]));
#pragma unroll
  for (int f = 0; f < 9; ++f) Zi.a[f] *= id;
#pragma unroll
  for (int r = 0; r < 3; ++r) t[r] *= id;
  M3<T> G;  // Z^-1 Lam P_vb = W P_vb
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) G(r, c) = fm(Zi(r, 2), LP(2, c), fm(Zi(r, 1), LP(1, c), Zi(r, 0) * LP(0, c)));
  // mean
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    x.p[r] = fm(P.pv(r, 2), t[2], fm(P.pv(r, 1), t[1], fm(P.pv(r, 0), t[0], x.p[r])));
    x.b[r] = fm(P.vb(2, r), t[2], fm(P.vb(1, r), t[1], fm(P.vb(0, r), t[0], x.b[r])));
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) x.v[r] = fm(P.vv(r, 2), t[2], fm(P.vv(r, 1), t[1], fm(P.vv(r, 0), t[0], x.v[r])));
  if (PPM == 1 || (PPM == 2 && ppm != nullptr)) {
    // P_pp -= (P_pv W) P_pv',  W = Z^-1 Lam (symmetric)
    S3<T> pp;
    if constexpr (PPM == 1) pp = P.pp; else pp_load(pp, ppm, pps);
    S3<T> W;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = r; c < 3; ++c) W.a[S3<T>::idx(r, c)] = fm(Zi(r, 2), Lam(2, c), fm(Zi(r, 1), Lam(1, c), Zi(r, 0) * Lam(0, c)));
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      T kp[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) kp[c] = fm(P.pv(r, 2), W(2, c), fm(P.pv(r, 1), W(1, c), P.pv(r, 0) * W(0, c)));
#pragma unroll
      for (int c = r; c < 3; ++c)
        pp.a[S3<T>::idx(r, c)] = fm(-kp[2], P.pv(c, 2), fm(-kp[1], P.pv(c, 1), fm(-kp[0], P.pv(c, 0), pp.a[S3<T>::idx(r, c)])));
    }
    if constexpr (PPM == 1) P.pp = pp; else pp_store(pp, ppm, pps);
  }
  // blocks that read the OLD P_pv / P_vb first
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) P.pb(r, c) = fm(-P.pv(r, 2), G(2, c), fm(-P.pv(r, 1), G(1, c), fm(-P.pv(r, 0), G(0, c), P.pb(r, c))));
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = r; c < 3; ++c)
      P.bb.a[S3<T>::idx(r, c)] =
          fm(-P.vb(2, r), G(2, c), fm(-P.vb(1, r), G(1, c), fm(-P.vb(0, r), G(0, c), P.bb.a[S3<T>::idx(r, c)])));
  {
    M3<T> n;  // P_pv Z^-1
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) n(r, c) = fm(P.pv(r, 2), Zi(2, c), fm(P.pv(r, 1), Zi(1, c), P.pv(r, 0) * Zi(0, c)));
    P.pv = n;
  }
  {
    M3<T> n;  // Z^-T P_vb
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) n(r, c) = fm(Zi(2, r), P.vb(2, c), fm(Zi(1, r), P.vb(1, c), Zi(0, r) * P.vb(0, c)));
    P.vb = n;
  }
  {
    S3<T> n;  // P_vv Z^-1 (symmetric)
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = r; c < 3; ++c) n.a[S3<T>::idx(r, c)] = fm(P.vv(r, 2), Zi(2, c), fm(P.vv(r, 1), Zi(1, c), P.vv(r, 0) * Zi(0, c)));
    P.vv = n;
  }
}

template <int PPM, typename T, typename X>
DEKF_HD void propagate4(const MheConst<T> &c, Cov9<T> &P, X &x, const M3<T> &R, const V3<T> &as, bool vo,
                        const V3<T> &dlt, T *ppm = nullptr, size_t pps = 0) {
  const bool pp_on = PPM == 1 || (PPM == 2 && ppm != nullptr);
  const T dt = c.dt, h = T(0.5) * c.dt * c.dt;
  const T dt2 = dt * dt, hdt = h * dt, hh = h * h;
  // mean: acc = a_s - R b,  d = p+ - p = dt v + h acc,  v+ = v + dt acc
  V3<T> hmean;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const T acc = fm(-R(r, 2), x.b[2], fm(-R(r, 1), x.b[1], fm(-R(r, 0), x.b[0], as[r])));
    hmean[r] = fm(h, acc, dt * x.v[r]);
    x.p[r] += hmean[r];
    x.v[r] = fm(dt, acc, x.v[r]);
  }
  // position rows first: Ep = P_pb R' is only needed for P_pv (and PL_p = Cov(p, d) = dt P_pv - h Ep)
  M3<T> PLp;
  {
    M3<T> Ep;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) Ep(r, cc) = fm(P.pb(r, 2), R(cc, 2), fm(P.pb(r, 1), R(cc, 1), P.pb(r, 0) * R(cc, 0)));
    if (pp_on || vo) {
#pragma unroll
      for (int f = 0; f < 9; ++f) PLp.a[f] = fm(-h, Ep.a[f], dt * P.pv.a[f]);
    }
#pragma unroll
    for (int f = 0; f < 9; ++f) P.pv.a[f] = fm(-dt, Ep.a[f], P.pv.a[f]);
  }
  // B = R P_bb,  Ev = P_vb R',  BRn = R P_bb R' + R C_a R'
  M3<T> B, Ev;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      B(r, cc) = fm(R(r, 2), P.bb(2, cc), fm(R(r, 1), P.bb(1, cc), R(r, 0) * P.bb(0, cc)));
      Ev(r, cc) = fm(P.vb(r, 2), R(cc, 2), fm(P.vb(r, 1), R(cc, 1), P.vb(r, 0) * R(cc, 0)));
    }
  S3<T> BRn;
#pragma unroll
  for (int f = 0; f < 6; ++f) BRn.a[f] = T(0);
  add_rot_diag(BRn, R, c.ae);
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = r; cc < 3; ++cc)
      BRn.a[S3<T>::idx(r, cc)] = fm(B(r, 2), R(cc, 2), fm(B(r, 1), R(cc, 1), fm(B(r, 0), R(cc, 0), BRn.a[S3<T>::idx(r, cc)])));
  P.bb.a[0] += c.cab[0];
  P.bb.a[3] += c.cab[1];
  P.bb.a[5] += c.cab[2];
  // U_v = Cov(v+, d) = dt P_vv - h Ev - dt^2 Ev' + h dt BRn (old P_vv);  P_pv+ = P_pv - dt Ep + U_v'
  M3<T> Uv;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) Uv(r, cc) = fm(hdt, BRn(r, cc), fm(-dt2, Ev(cc, r), fm(-h, Ev(r, cc), dt * P.vv(r, cc))));
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) P.pv(r, cc) += Uv(cc, r);
  // Cov(d) without the camera noise: Vn = dt^2 P_vv - h dt (Ev + Ev') + h^2 BRn + dt^2 R C_p R'
  S3<T> Vn;
  if (pp_on || vo) {
#pragma unroll
    for (int f = 0; f < 6; ++f) Vn.a[f] = T(0);
    add_rot_diag(Vn, R, c.pe);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc) {
        const int k = S3<T>::idx(r, cc);
        Vn.a[k] = fm(dt2, P.vv.a[k], fm(-hdt, Ev(r, cc) + Ev(cc, r), fm(hh, BRn.a[k], Vn.a[k])));
      }
  }
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = r; cc < 3; ++cc) {
      const int k = S3<T>::idx(r, cc);
      P.vv.a[k] = fm(dt2, BRn.a[k], fm(-dt, Ev(r, cc) + Ev(cc, r), P.vv.a[k]));
    }
  M3<T> Xb;  // dt P_vb - h B = P_pb+ - P_pb = U_b'
#pragma unroll
  for (int f = 0; f < 9; ++f) {
    Xb.a[f] = fm(-h, B.a[f], dt * P.vb.a[f]);
    P.pb.a[f] += Xb.a[f];
    P.vb.a[f] = fm(-dt, B.a[f], P.vb.a[f]);
  }
  S3<T> pp;
  if (pp_on) {
    if constexpr (PPM == 1) pp = P.pp; else pp_load(pp, ppm, pps);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc) {
        const int k = S3<T>::idx(r, cc);
        pp.a[k] += (PLp(r, cc) + PLp(cc, r)) + Vn.a[k];
      }
    if (!vo) {
      if constexpr (PPM == 1) P.pp = pp; else pp_store(pp, ppm, pps);
    }
  }
  if (vo) {
    // p_{k+1} - p_k = Delta + vcam, cov(vcam) = R diag(vo_p_std^2) R' (DecentralEst.cpp:477, :1004-1005)
    S3<T> Si;
    T id;
    {
      S3<T> Sinn = Vn;
      add_rot_diag(Sinn, R, c.nvo);
      T det;
      Si = adjugate(Sinn, det);
      id = T(1) / det;
    }
    // U_p = PL_p + Vn,  U_b = Xb'
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) PLp(r, cc) += Vn(r, cc);
    V3<T> t;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      // innovation Delta - (predicted d); hmean was already added to x.p
      t[r] = dlt[r] - hmean[r];
    }
    {
      const V3<T> nu = t;
#pragma unroll
      for (int r = 0; r < 3; ++r) t[r] = fm(Si(r, 2), nu[2], fm(Si(r, 1), nu[1], Si(r, 0) * nu[0]));
    }
#pragma unroll
    for (int f = 0; f < 6; ++f) Si.a[f] *= id;
#pragma unroll
    for (int r = 0; r < 3; ++r) t[r] *= id;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      x.p[r] = fm(PLp(r, 2), t[2], fm(PLp(r, 1), t[1], fm(PLp(r, 0), t[0], x.p[r])));
      x.v[r] = fm(Uv(r, 2), t[2], fm(Uv(r, 1), t[1], fm(Uv(r, 0), t[0], x.v[r])));
      x.b[r] = fm(Xb(2, r), t[2], fm(Xb(1, r), t[1], fm(Xb(0, r), t[0], x.b[r])));
    }
    // P -= U S^-1 U', one row of K = U S^-1 at a time
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      T k[3];
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) k[cc] = fm(PLp(r, 2), Si(2, cc), fm(PLp(r, 1), Si(1, cc), PLp(r, 0) * Si(0, cc)));
      if (pp_on) {
#pragma unroll
        for (int cc = r; cc < 3; ++cc)
          pp.a[S3<T>::idx(r, cc)] = fm(-k[2], PLp(cc, 2), fm(-k[1], PLp(cc, 1), fm(-k[0], PLp(cc, 0), pp.a[S3<T>::idx(r, cc)])));
      }
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        P.pv(r, cc) = fm(-k[2], Uv(cc, 2), fm(-k[1], Uv(cc, 1), fm(-k[0], Uv(cc, 0), P.pv(r, cc))));
        P.pb(r, cc) = fm(-k[2], Xb(2, cc), fm(-k[1], Xb(1, cc), fm(-k[0], Xb(0, cc), P.pb(r, cc))));
      }
    }
    if (pp_on) {
      if constexpr (PPM == 1) P.pp = pp; else pp_store(pp, ppm, pps);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      T k[3];
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) k[cc] = fm(Uv(r, 2), Si(2, cc), fm(Uv(r, 1), Si(1, cc), Uv(r, 0) * Si(0, cc)));
#pragma unroll
      for (int cc = r; cc < 3; ++cc)
        P.vv.a[S3<T>::idx(r, cc)] =
            fm(-k[2], Uv(cc, 2), fm(-k[1], Uv(cc, 1), fm(-k[0], Uv(cc, 0), P.vv.a[S3<T>::idx(r, cc)])));
#pragma unroll
      for (int cc = 0; cc < 3; ++cc)
        P.vb(r, cc) = fm(-k[2], Xb(2, cc), fm(-k[1], Xb(1, cc), fm(-k[0], Xb(0, cc), P.vb(r, cc))));
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      T k[3];
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) k[cc] = fm(Xb(2, r), Si(2, cc), fm(Xb(1, r), Si(1, cc), Xb(0, r) * Si(0, cc)));
#pragma unroll
      for (int cc = r; cc < 3; ++cc)
        P.bb.a[S3<T>::idx(r, cc)] =
            fm(-k[2], Xb(2, cc), fm(-k[1], Xb(1, cc), fm(-k[0], Xb(0, cc), P.bb.a[S3<T>::idx(r, cc)])));
    }
  }
}

// ---- version 5 of the propagation: stages WITHOUT a VO row take an in-place path with the shortest live ranges
// (A = T1 T2 with T2: p += dt v and T1: p -= h R b, v -= dt R b; each rotated product is consumed right after it is formed);
// stages WITH a VO row need Cov(x+, p+ - p) from the pre-update blocks and take the version-4 path.  Which path a stage takes
// depends only on its own VO flag, so the full re-sweep, the incremental sweep and the KF alternative stay bit-identical.
template <int PPM, typename T, typename X>
DEKF_HD void propagate5(const MheConst<T> &c, Cov9<T> &P, X &x, const M3<T> &R, const V3<T> &as, bool vo, const V3<T> &dlt,
                        T *ppm = nullptr, size_t pps = 0) {
  if (vo) {
    propagate4<PPM>(c, P, x, R, as, true, dlt, ppm, pps);
    return;
  }
  const bool pp_on = PPM == 1 || (PPM == 2 && ppm != nullptr);
  const T dt = c.dt, h = T(0.5) * c.dt * c.dt;
  const T dt2 = dt * dt, hdt = h * dt, hh = h * h;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const T acc = fm(-R(r, 2), x.b[2], fm(-R(r, 1), x.b[1], fm(-R(r, 0), x.b[0], as[r])));
    x.p[r] += fm(h, acc, dt * x.v[r]);
    x.v[r] = fm(dt, acc, x.v[r]);
  }
  S3<T> pp;
  if (pp_on) {
    if constexpr (PPM == 1) pp = P.pp; else pp_load(pp, ppm, pps);
    // T2 on P_pp: += dt (P_pv + P_pv') + dt^2 P_vv;  noise dt^2 R C_p R'
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc) {
        const int k = S3<T>::idx(r, cc);
        pp.a[k] = fm(dt, P.pv(r, cc) + P.pv(cc, r), fm(dt2, P.vv.a[k], pp.a[k]));
      }
    add_rot_diag(pp, R, c.pe);
  }
  // T2: P_pv += dt P_vv, P_pb += dt P_vb
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      P.pv(r, cc) = fm(dt, P.vv(r, cc), P.pv(r, cc));
      P.pb(r, cc) = fm(dt, P.vb(r, cc), P.pb(r, cc));
    }
  // T1, position rows: Ep = P_pb R';  P_pv -= dt Ep  (P_pp -= h (Ep + Ep'))
  {
    M3<T> Ep;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        Ep(r, cc) = fm(P.pb(r, 2), R(cc, 2), fm(P.pb(r, 1), R(cc, 1), P.pb(r, 0) * R(cc, 0)));
        P.pv(r, cc) = fm(-dt, Ep(r, cc), P.pv(r, cc));
      }
    if (pp_on) {
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = r; cc < 3; ++cc) pp.a[S3<T>::idx(r, cc)] = fm(-h, Ep(r, cc) + Ep(cc, r), pp.a[S3<T>::idx(r, cc)]);
    }
  }
  // T1, velocity rows: Ev = P_vb R';  P_pv -= h Ev',  P_vv -= dt (Ev + Ev')
  {
    M3<T> Ev;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        Ev(r, cc) = fm(P.vb(r, 2), R(cc, 2), fm(P.vb(r, 1), R(cc, 1), P.vb(r, 0) * R(cc, 0)));
        P.pv(cc, r) = fm(-h, Ev(r, cc), P.pv(cc, r));
      }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc) P.vv.a[S3<T>::idx(r, cc)] = fm(-dt, Ev(r, cc) + Ev(cc, r), P.vv.a[S3<T>::idx(r, cc)]);
  }
  // T1, bias column: B = R P_bb;  P_pb -= h B,  P_vb -= dt B;  BRn = B R' + R C_a R' enters P_pv, P_vv (and P_pp)
  {
    M3<T> B;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        B(r, cc) = fm(R(r, 2), P.bb(2, cc), fm(R(r, 1), P.bb(1, cc), R(r, 0) * P.bb(0, cc)));
        P.pb(r, cc) = fm(-h, B(r, cc), P.pb(r, cc));
        P.vb(r, cc) = fm(-dt, B(r, cc), P.vb(r, cc));
      }
    S3<T> BRn;
#pragma unroll
    for (int f = 0; f < 6; ++f) BRn.a[f] = T(0);
    add_rot_diag(BRn, R, c.ae);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = r; cc < 3; ++cc) {
        const int k = S3<T>::idx(r, cc);
        BRn.a[k] = fm(B(r, 2), R(cc, 2), fm(B(r, 1), R(cc, 1), fm(B(r, 0), R(cc, 0), BRn.a[k])));
        P.vv.a[k] = fm(dt2, BRn.a[k], P.vv.a[k]);
        if (pp_on) pp.a[k] = fm(hh, BRn.a[k], pp.a[k]);
      }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) P.pv(r, cc) = fm(hdt, BRn(r, cc), P.pv(r, cc));
  }
  P.bb.a[0] += c.cab[0];
  P.bb.a[3] += c.cab[1];
  P.bb.a[5] += c.cab[2];
  if (pp_on) {
    if constexpr (PPM == 1) P.pp = pp; else pp_store(pp, ppm, pps);
  }
}

// Math policy of the sweep: MV / PV select the version of the measurement / propagation stage.
template <int MV, int PV>
struct MathSel {
  // PPM (version 4 only; versions 1-3 always carry P_pp in P.pp): see meas_update4
  template <int PPM = 1, typename T, typename X>
  DEKF_HD static void meas(Cov9<T> &P, X &x, const S3<T> &Lam, const V3<T> &eta, T *ppm = nullptr, size_t pps = 0) {
    if constexpr (MV == 1)
      meas_update(P, x, Lam, eta);
    else if constexpr (MV == 2)
      meas_update2(P, x, Lam, eta);
    else if constexpr (MV == 3)
      meas_update3(P, x, Lam, eta);
    else
      meas_update4<PPM>(P, x, Lam, eta, ppm, pps);
  }
  template <int PPM = 1, typename T, typename X>
  DEKF_HD static void prop(const MheConst<T> &c, Cov9<T> &P, X &x, const M3<T> &R, const V3<T> &as, bool vo,
                           const V3<T> &dlt, T *ppm = nullptr, size_t pps = 0) {
    if constexpr (PV == 1)
      propagate(c, P, x, R, as, vo, dlt);
    else if constexpr (PV == 2)
      propagate2(c, P, x, R, as, vo, dlt);
    else if constexpr (PV == 4)
      propagate4<PPM>(c, P, x, R, as, vo, dlt, ppm, pps);
    else
      propagate5<PPM>(c, P, x, R, as, vo, dlt, ppm, pps);
  }
  static constexpr bool kLazyPP = (MV == 4 && PV >= 4);
};
// Measured on B200 (tools/tune_solve.cu, profiles/r01_tune_solve.md): fp64 is register-bound at 255 registers, the
// in-place propagation of version 2 spills more there (139 vs 121 us/launch); fp32 has registers to spare and takes
// the version with the fewest instructions (67.7 vs 77.4 us/launch).
template <typename T>
struct DefaultMath : MathSel<4, 5> {};

template <typename T>
struct StageRec {
  M3<T> R;
  V3<T> as;
  S3<T> Lam;
  V3<T> eta, dlt;
  bool vo;
};

// Stage records straight from the HBM window ring (fused small-batch kernel, host debug harness).
template <typename T>
struct GlobalStageSource {
  const Dims &dm;
  const Buffers<T> &b;
  int i;
  // small batches (k_fused: a handful of warps on the whole device, nothing to hide a load behind): ask for the record of
  // stage k + 2 while stage k is being processed, so that its loads hit L1 instead of paying an L2 round trip per stage
  bool prefetch = false;
  DEKF_HD GlobalStageSource(const Dims &dm_, const Buffers<T> &b_, int i_, bool pf = false) : dm(dm_), b(b_), i(i_), prefetch(pf) {}
  DEKF_HD void acquire(int /*ordinal*/) const {}
  DEKF_HD void release(int /*ordinal*/) const {}
  DEKF_HD const T *rec(int k) const { return b.win + (size_t)(k % dm.NW) * REC_SIZE * dm.ns + i; }
  DEKF_HD void meas(int, int k, S3<T> &Lam, V3<T> &eta) const {
    const T *r = rec(k);
    const size_t ns = (size_t)dm.ns;
#if defined(__CUDA_ARCH__)
    if (prefetch) {
      const T *q = rec(k + 2);
#pragma unroll
      for (int f = 0; f < REC_SIZE; ++f) asm volatile("prefetch.global.L1 [%0];" ::"l"(q + f * ns));
    }
#endif
#pragma unroll
    for (int f = 0; f < 6; ++f) Lam.a[f] = r[(REC_LAM + f) * ns];
#pragma unroll
    for (int f = 0; f < 3; ++f) eta[f] = r[(REC_ETA + f) * ns];
  }
  DEKF_HD void rot(int, int k, M3<T> &R) const {
    const T *r = rec(k);
    const size_t ns = (size_t)dm.ns;
#pragma unroll
    for (int f = 0; f < 9; ++f) R.a[f] = r[(REC_R + f) * ns];
  }
  DEKF_HD void dyn(int, int k, V3<T> &as, V3<T> &dlt, bool &vo) const {
    const T *r = rec(k);
    const size_t ns = (size_t)dm.ns;
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      as[f] = r[(REC_AS + f) * ns];
      dlt[f] = r[(REC_DLT + f) * ns];
    }
    vo = r[REC_FLAG * ns] != T(0);
  }
};

// update(T) after UpdateMHE/UpdateVOConstraints: marginalizeQP(T-N) if T >= N, solve, read x_T,
// v_MHE_b (DecentralEst.cpp:167-185).  Tier A: the whole window is re-swept every step, like the
// reference re-solves the whole QP every step.  `src` hands out the stage records: ordinal j = 0.. is
// the position in the sweep (stage k0 + j), acquire/release bracket the use of one record (the TMA
// path maps them onto the full/empty mbarriers of its shared-memory ring).
// Start of the sweep of update(T): the prior at stage 0 while the window is still growing, else the arrival cost at stage
// T-N.  Returns the first stage k0.  Separate from the sweep so that the TMA kernel can issue these loads before it sets
// up its barriers and tiles.
template <typename T, typename X>
DEKF_HD int mhe_solve_start(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, int Tk, int i, Cov9<T> &P, X &x) {
  const int ns = dm.ns, N = dm.N;
  if (Tk < N) {
    // Prior_0: Q_prior = blkdiag(Q_p0, Q_v0, Q_b0), x_prior = 0 (DecentralEst.cpp:232-253)
#pragma unroll
    for (int f = 0; f < 6; ++f) P.pp.a[f] = P.vv.a[f] = P.bb.a[f] = T(0);
#pragma unroll
    for (int f = 0; f < 9; ++f) P.pv.a[f] = P.pb.a[f] = P.vb.a[f] = T(0);
    P.pp.a[0] = c.P0[0];
    P.pp.a[3] = c.P0[1];
    P.pp.a[5] = c.P0[2];
    P.vv.a[0] = c.P0[3];
    P.vv.a[3] = c.P0[4];
    P.vv.a[5] = c.P0[5];
    P.bb.a[0] = c.P0[6];
    P.bb.a[3] = c.P0[7];
    P.bb.a[5] = c.P0[8];
#pragma unroll
    for (int f = 0; f < 3; ++f) x.p[f] = x.v[f] = x.b[f] = T(0);
    return 0;
  }
  load_cov(b.arr_P, ns, i, P);
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    x.p[f] = b.arr_x[(size_t)f * ns + i];
    x.v[f] = b.arr_x[(size_t)(3 + f) * ns + i];
    x.b[f] = b.arr_x[(size_t)(6 + f) * ns + i];
  }
  return Tk - N;
}

template <typename T, typename Source, typename Math = DefaultMath<T>, typename X = Vec9<T>>
DEKF_HD int mhe_solve_sweep(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                            int Tk, int i, Source &src, Cov9<T> &P, X &x, const int k0) {
  const int n = dm.n, ns = dm.ns, N = dm.N;
  // Version-4 math: P_pp is only needed where the arrival cost of the next tick is produced, i.e. in stage T-N.  That
  // stage is peeled off (it carries P_pp in registers); the loop over the remaining stages does not carry P_pp at all.
  // Otherwise: one copy of the stage body in the instruction stream (the loop is ~2k instructions; the I-cache matters).
  constexpr bool LZ = Math::kLazyPP;
  constexpr int PPM = LZ ? 0 : 1;
  M3<T> RT;
  V3<T> om = v3<T>(T(0), T(0), T(0));
  int k = k0;
  if (LZ && Tk >= N) {
    src.acquire(0);
    {
      S3<T> Lam;
      V3<T> eta;
      src.meas(0, k, Lam, eta);
      Math::template meas<1>(P, x, Lam, eta);
    }
    src.rot(0, k, RT);
    {
      V3<T> as, dlt;
      bool vo;
      src.dyn(0, k, as, dlt, vo);
      src.release(0);
      Math::template prop<1>(c, P, x, RT, as, vo, dlt);
    }
    // marginalizeQP(T-N): the arrival cost moves to x_{T-N+1} (MheSrb.cpp:475-713)
    store_cov(b.arr_P, ns, i, P);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      b.arr_x[(size_t)f * ns + i] = x.p[f];
      b.arr_x[(size_t)(3 + f) * ns + i] = x.v[f];
      b.arr_x[(size_t)(6 + f) * ns + i] = x.b[f];
    }
    if (k == Tk - 1) {
#pragma unroll
      for (int f = 0; f < 3; ++f) om[f] = (T)in.gyro[(size_t)f * n + i];
    }
    ++k;
  }
  for (;; ++k) {
    const int j = k - k0;
    src.acquire(j);
    {
      S3<T> Lam;
      V3<T> eta;
      src.meas(j, k, Lam, eta);
      Math::template meas<PPM>(P, x, Lam, eta);
    }
    src.rot(j, k, RT);
    if (k == Tk) {
      src.release(j);
      break;
    }
    {
      V3<T> as, dlt;
      bool vo;
      src.dyn(j, k, as, dlt, vo);
      src.release(j);
      Math::template prop<PPM>(c, P, x, RT, as, vo, dlt);
    }
    if (k == Tk - 1) {
      // angular velocity of the newest sample for the read-out below: fetched one stage ahead of its use
#pragma unroll
      for (int f = 0; f < 3; ++f) om[f] = (T)in.gyro[(size_t)f * n + i];
    }
    if (!LZ && k == Tk - N) {
      store_cov(b.arr_P, ns, i, P);
#pragma unroll
      for (int f = 0; f < 3; ++f) {
        b.arr_x[(size_t)f * ns + i] = x.p[f];
        b.arr_x[(size_t)(3 + f) * ns + i] = x.v[f];
        b.arr_x[(size_t)(6 + f) * ns + i] = x.b[f];
      }
    }
  }
  // getsolution(T) + v_MHE_b = R_sb (v + omega x p_imu_2_opti) (DecentralEst.cpp:181-185)
  if (k0 == Tk) {  // (not reachable from update(T >= 1); keeps the read-out defined)
#pragma unroll
    for (int f = 0; f < 3; ++f) om[f] = (T)in.gyro[(size_t)f * n + i];
  }
  const V3<T> lever = v3<T>(c.lever[0], c.lever[1], c.lever[2]);
  Vec9<T> xr;
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    xr.p[f] = x.p[f];
    xr.v[f] = x.v[f];
    xr.b[f] = x.b[f];
  }
  const V3<T> vb = mul(RT, add(xr.v, cross(om, lever)));
  int status = 0;
  const T chk = xr.p[0] + xr.p[1] + xr.p[2] + xr.v[0] + xr.v[1] + xr.v[2] + xr.b[0] + xr.b[1] + xr.b[2];
  if (!(chk == chk) || !(chk - chk == T(0))) status |= ST_NONFINITE;
  if (out.x != nullptr) {
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      out.x[(size_t)f * n + i] = (double)xr.p[f];
      out.x[(size_t)(3 + f) * n + i] = (double)xr.v[f];
      out.x[(size_t)(6 + f) * n + i] = (double)xr.b[f];
    }
  }
  if (out.v_body != nullptr) {
#pragma unroll
    for (int f = 0; f < 3; ++f) out.v_body[(size_t)f * n + i] = (double)vb[f];
  }
  return status;
}

template <typename T, typename Source, typename Math = DefaultMath<T>>
DEKF_HD int mhe_solve(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                      int Tk, int i, Source &src) {
  Cov9<T> P;
  Vec9<T> x;
  const int k0 = mhe_solve_start(c, dm, b, Tk, i, P, x);
  return mhe_solve_sweep<T, Source, Math>(c, dm, b, in, out, Tk, i, src, P, x, k0);
}

template <typename T>
DEKF_HD int mhe_solve(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                      int Tk, int i, bool prefetch = false) {
  GlobalStageSource<T> src(dm, b, i, prefetch);
  return mhe_solve<T>(c, dm, b, in, out, Tk, i, src);
}

// Incremental window solve (tier B of SURVEY.md 8d; legal because no row of the shipped QP is an inequality and only
// x_T is read out).  The forward sweep of update(T) over the window differs from the sweep of update(T-1) only (a) by
// the new stage T and (b) from the first stage whose VO row was turned into an equality this tick
// (UpdateVOConstraints, DecentralEst.cpp:987-1009) onwards.  The filter state after the leg-odometry update of every
// window stage is kept in a ring (`ckpt`), so update(T) restarts at stage ks = min(T-1, first changed stage) and runs
// the SAME operations on the SAME operands as the full sweep would from there on: the results are bit-identical to
// the full re-sweep (tests/test_gpu_parity.py::test_incremental_equals_full_resweep).  marginalizeQP(T-N) is not
// needed on the step path any more: the arrival cost (M_p, n_p) is the time update of checkpoint T-N and is computed
// when a getter asks for it (arrival_from_checkpoint).
template <typename T>
DEKF_HD void load_ckpt(const Dims &dm, const Buffers<T> &b, int k, int i, Cov9<T> &P, Vec9<T> &x) {
  const T *base = b.ckpt + (size_t)(k % dm.NW) * 54 * dm.ns;
  load_cov(base, dm.ns, i, P);
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    x.p[f] = base[(size_t)(45 + f) * dm.ns + i];
    x.v[f] = base[(size_t)(48 + f) * dm.ns + i];
    x.b[f] = base[(size_t)(51 + f) * dm.ns + i];
  }
}
template <typename T>
DEKF_HD void store_ckpt(const Dims &dm, const Buffers<T> &b, int k, int i, const Cov9<T> &P, const Vec9<T> &x) {
  T *base = b.ckpt + (size_t)(k % dm.NW) * 54 * dm.ns;
  store_cov(base, dm.ns, i, P);
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    base[(size_t)(45 + f) * dm.ns + i] = x.p[f];
    base[(size_t)(48 + f) * dm.ns + i] = x.v[f];
    base[(size_t)(51 + f) * dm.ns + i] = x.b[f];
  }
}

// `ks`: restart stage (its checkpoint must be valid; any stage <= the instance's own first changed stage and >= the
// window start will do, so a CTA may agree on a common one).  `src` as in mhe_solve; ordinal j is stage ks + j.
template <typename T, typename Source, typename Math = DefaultMath<T>>
DEKF_HD int mhe_solve_incr(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                           int Tk, int i, Source &src, int ks) {
  const int n = dm.n;
  Cov9<T> P;
  Vec9<T> x;
  if (Tk == 1) {
    // Prior_0 (DecentralEst.cpp:232-253); the leg-odometry rows of stage 0 follow in the loop (j == 0 below)
#pragma unroll
    for (int f = 0; f < 6; ++f) P.pp.a[f] = P.vv.a[f] = P.bb.a[f] = T(0);
#pragma unroll
    for (int f = 0; f < 9; ++f) P.pv.a[f] = P.pb.a[f] = P.vb.a[f] = T(0);
    P.pp.a[0] = c.P0[0];
    P.pp.a[3] = c.P0[1];
    P.pp.a[5] = c.P0[2];
    P.vv.a[0] = c.P0[3];
    P.vv.a[3] = c.P0[4];
    P.vv.a[5] = c.P0[5];
    P.bb.a[0] = c.P0[6];
    P.bb.a[3] = c.P0[7];
    P.bb.a[5] = c.P0[8];
    x.p = x.v = x.b = v3<T>(T(0), T(0), T(0));
  } else {
    load_ckpt(dm, b, ks, i, P, x);
  }
  M3<T> RT;
  for (int k = ks;; ++k) {
    const int j = k - ks;
    src.acquire(j);
    if (j > 0 || Tk == 1) {  // the restart checkpoint already holds the leg-odometry update of stage ks
      S3<T> Lam;
      V3<T> eta;
      src.meas(j, k, Lam, eta);
      Math::meas(P, x, Lam, eta);
      store_ckpt(dm, b, k, i, P, x);
    }
    src.rot(j, k, RT);
    if (k == Tk) {
      src.release(j);
      break;
    }
    {
      V3<T> as, dlt;
      bool vo;
      src.dyn(j, k, as, dlt, vo);
      src.release(j);
      Math::prop(c, P, x, RT, as, vo, dlt);
    }
  }
  V3<T> om;
#pragma unroll
  for (int f = 0; f < 3; ++f) om[f] = (T)in.gyro[(size_t)f * n + i];
  const V3<T> lever = v3<T>(c.lever[0], c.lever[1], c.lever[2]);
  const V3<T> vb = mul(RT, add(x.v, cross(om, lever)));
  int status = 0;
  const T chk = x.p[0] + x.p[1] + x.p[2] + x.v[0] + x.v[1] + x.v[2] + x.b[0] + x.b[1] + x.b[2];
  if (!(chk == chk) || !(chk - chk == T(0))) status |= ST_NONFINITE;
  if (out.x != nullptr) {
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      out.x[(size_t)f * n + i] = (double)x.p[f];
      out.x[(size_t)(3 + f) * n + i] = (double)x.v[f];
      out.x[(size_t)(6 + f) * n + i] = (double)x.b[f];
    }
  }
  if (out.v_body != nullptr) {
#pragma unroll
    for (int f = 0; f < 3; ++f) out.v_body[(size_t)f * n + i] = (double)vb[f];
  }
  return status;
}

// restart stage of instance i at tick Tk: T-1, or the first stage whose VO row changed this tick
template <typename T>
DEKF_HD int incr_restart_stage(const Dims &dm, const Buffers<T> &b, int Tk, int i) {
  if (Tk == 1) return 0;
  int ks = Tk - 1;
  const int rs = tick_resweep(dm, b, Tk, i);
  if (rs < ks) ks = rs;
  const int kmin = (Tk >= dm.N) ? Tk - dm.N : 0;  // VO bounds never reach below the window start (DecentralEst.cpp:917-918)
  return ks < kmin ? kmin : ks;
}

template <typename T>
DEKF_HD int mhe_solve_incr(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                           int Tk, int i, bool prefetch = false) {
  GlobalStageSource<T> src(dm, b, i, prefetch);
  return mhe_solve_incr<T>(c, dm, b, in, out, Tk, i, src, incr_restart_stage(dm, b, Tk, i));
}

// marginalizeQP(T-N) on demand for the incremental solve: arrival cost on x_{T-N+1} = time update (dynamics + VO row
// of stage T-N as it stands now) of checkpoint T-N; written to arr_P / arr_x where the getters read it.
template <typename T, typename Math = DefaultMath<T>>
DEKF_HD void arrival_from_checkpoint(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, int Tk, int i) {
  if (Tk < dm.N) return;  // still the initial prior (k_init_state)
  GlobalStageSource<T> src(dm, b, i);
  Cov9<T> P;
  Vec9<T> x;
  load_ckpt(dm, b, Tk - dm.N, i, P, x);
  M3<T> R;
  V3<T> as, dlt;
  bool vo;
  src.rot(0, Tk - dm.N, R);
  src.dyn(0, Tk - dm.N, as, dlt, vo);
  Math::prop(c, P, x, R, as, vo, dlt);
  store_cov(b.arr_P, dm.ns, i, P);
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    b.arr_x[(size_t)f * dm.ns + i] = x.p[f];
    b.arr_x[(size_t)(3 + f) * dm.ns + i] = x.v[f];
    b.arr_x[(size_t)(6 + f) * dm.ns + i] = x.b[f];
  }
}

// KF alternative, est_type_ == 1 (DecentralEst.cpp:592-861 InitializeKF / UpdateKF, :189-196 output): the same
// linear-Gaussian model filtered one sample at a time, (x_KF_, C_KF_) kept in arr_x / arr_P.  T == 0 is
// InitializeKF + UpdateKF on the same sample (DecentralEst.cpp:139-141): prior -> correct(0) -> predict with
// (R_0, a_s,0) -> correct(0) again.  T >= 1: predict with the previous sample's (R, a_s) (:706-707 read the
// stack back BEFORE GetMeasurement), correct with the new sample (:787-860).  The correction uses the
// sufficient statistic (Lambda, eta) of the leg-odometry rows like the MHE sweep; C_KF_ stays symmetric.
template <typename T, typename Math = DefaultMath<T>>
DEKF_HD int kf_update(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, const Inputs &in, const Outputs &out,
                      int Tk, int i) {
  const int n = dm.n, ns = dm.ns;
  GlobalStageSource<T> src(dm, b, i);
  Cov9<T> P;
  Vec9<T> x;
  S3<T> Lam;
  V3<T> eta, as, dlt;
  M3<T> R;
  bool vo;
  if (Tk == 0) {
#pragma unroll
    for (int f = 0; f < 6; ++f) P.pp.a[f] = P.vv.a[f] = P.bb.a[f] = T(0);
#pragma unroll
    for (int f = 0; f < 9; ++f) P.pv.a[f] = P.pb.a[f] = P.vb.a[f] = T(0);
    P.pp.a[0] = c.P0[0];
    P.pp.a[3] = c.P0[1];
    P.pp.a[5] = c.P0[2];
    P.vv.a[0] = c.P0[3];
    P.vv.a[3] = c.P0[4];
    P.vv.a[5] = c.P0[5];
    P.bb.a[0] = c.P0[6];
    P.bb.a[3] = c.P0[7];
    P.bb.a[5] = c.P0[8];
    x.p = x.v = x.b = v3<T>(T(0), T(0), T(0));
    src.meas(0, 0, Lam, eta);
    Math::meas(P, x, Lam, eta);  // :697-699
  } else {
    load_cov(b.arr_P, ns, i, P);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      x.p[f] = b.arr_x[(size_t)f * ns + i];
      x.v[f] = b.arr_x[(size_t)(3 + f) * ns + i];
      x.b[f] = b.arr_x[(size_t)(6 + f) * ns + i];
    }
  }
  const int kp = (Tk == 0) ? 0 : Tk - 1;
  src.rot(0, kp, R);
  src.dyn(0, kp, as, dlt, vo);
  Math::prop(c, P, x, R, as, false, dlt);  // :783-785 (the KF alternative has no VO rows)
  src.meas(0, Tk, Lam, eta);
  Math::meas(P, x, Lam, eta);  // :858-860
  src.rot(0, Tk, R);
  store_cov(b.arr_P, ns, i, P);
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    b.arr_x[(size_t)f * ns + i] = x.p[f];
    b.arr_x[(size_t)(3 + f) * ns + i] = x.v[f];
    b.arr_x[(size_t)(6 + f) * ns + i] = x.b[f];
  }
  // v_KF_b_ = R_sb (v + omega x p_imu_2_opti) (:192-194)
  V3<T> om;
#pragma unroll
  for (int f = 0; f < 3; ++f) om[f] = (T)in.gyro[(size_t)f * n + i];
  const V3<T> lever = v3<T>(c.lever[0], c.lever[1], c.lever[2]);
  const V3<T> vb = mul(R, add(x.v, cross(om, lever)));
  int status = 0;
  const T chk = x.p[0] + x.p[1] + x.p[2] + x.v[0] + x.v[1] + x.v[2] + x.b[0] + x.b[1] + x.b[2];
  if (!(chk == chk) || !(chk - chk == T(0))) status |= ST_NONFINITE;
  if (out.x != nullptr) {
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      out.x[(size_t)f * n + i] = (double)x.p[f];
      out.x[(size_t)(3 + f) * n + i] = (double)x.v[f];
      out.x[(size_t)(6 + f) * n + i] = (double)x.b[f];
    }
  }
  if (out.v_body != nullptr) {
#pragma unroll
    for (int f = 0; f < 3; ++f) out.v_body[(size_t)f * n + i] = (double)vb[f];
  }
  return status;
}

// ------------------------------------------------------------------------------------------------
// Smoothed window (dekf_get_window): every state block of MHEproblem::solution (MheSrb.hpp:58-112), not only x_T.
// The window QP of update(T) holds K = min(T+1, N) states, stages T-K+1 .. T, with the arrival cost on the first.  Its
// optimum is the Rauch-Tung-Striebel smoother of the forward sweep: x_T^s = m_T and, for k = T-1 down to T-K+1,
//   x_k^s = m'_k + C' Sigma^-1 (x_{k+1}^s - mu)
// where (m_k, P_k) is the filtered state of stage k (after its leg-odometry rows), mu / Sigma the prediction of x_{k+1}
// (dynamics, then the VO row p_{k+1} - p_k = Delta_k if it is an equality: exactly the forward sweep's time update) and
// m'_k, C' = Cov(x_k, x_{k+1}) are conditioned on that VO row.  Exact, because the leg rows of stage k+1 and everything after
// them see x_k only through x_{k+1}.  With A the transition, L = [0, dt I, -h R] (p_{k+1} - p_k = L x_k + h a_s + w_p),
// U = Cov(x_{k+1}, d) = A P L' + [C1; C2; 0], S = L P L' + C1 + R C_vo R' and nu = Delta - (L m + h a_s):
//   m'_k + C' z = m_k + P_k g,   g = A' z + L' S^-1 (nu - U' z),   U' z = L P A' z + C1 z_p + C2 z_v,   z = Sigma^-1 (x^s - mu)
// (no VO row: g = A' z).  Only Sigma is factorised (9x9 Cholesky); C' is never formed.  The arithmetic is D (double) for
// both handle precisions; every multiply-add is an explicit fm so that the host build performs the same operations.
// ------------------------------------------------------------------------------------------------
template <typename D, typename T>
DEKF_HD void load_state_as(const T *base, size_t ns, Cov9<D> &P, Vec9<D> &x) {
#pragma unroll
  for (int f = 0; f < 6; ++f) {
    P.pp.a[f] = (D)base[f * ns];
    P.vv.a[f] = (D)base[(6 + f) * ns];
    P.bb.a[f] = (D)base[(12 + f) * ns];
  }
#pragma unroll
  for (int f = 0; f < 9; ++f) {
    P.pv.a[f] = (D)base[(18 + f) * ns];
    P.pb.a[f] = (D)base[(27 + f) * ns];
    P.vb.a[f] = (D)base[(36 + f) * ns];
  }
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    x.p[f] = (D)base[(45 + f) * ns];
    x.v[f] = (D)base[(48 + f) * ns];
    x.b[f] = (D)base[(51 + f) * ns];
  }
}

// entry (r, c) of the dense 9x9 matrix held by a Cov9 (indices are compile-time constants after unrolling)
template <typename D>
DEKF_HD D cov_at(const Cov9<D> &P, int r, int c) {
  if (r > c) {
    const int t = r;
    r = c;
    c = t;
  }
  const int br = r / 3, bc = c / 3, rr = r % 3, cc = c % 3;
  if (br == bc) return br == 0 ? P.pp(rr, cc) : (br == 1 ? P.vv(rr, cc) : P.bb(rr, cc));
  if (br == 0) return bc == 1 ? P.pv(rr, cc) : P.pb(rr, cc);
  return P.vb(rr, cc);
}

// y += P a (P symmetric 9x9 in blocks)
template <typename D>
DEKF_HD void cov_mul_add(const Cov9<D> &P, const V3<D> &ap, const V3<D> &av, const V3<D> &ab, Vec9<D> &y) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    D sp = y.p[r], sv = y.v[r], sb = y.b[r];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      sp = fm(P.pp(r, k), ap[k], sp);
      sp = fm(P.pv(r, k), av[k], sp);
      sp = fm(P.pb(r, k), ab[k], sp);
      sv = fm(P.pv(k, r), ap[k], sv);
      sv = fm(P.vv(r, k), av[k], sv);
      sv = fm(P.vb(r, k), ab[k], sv);
      sb = fm(P.pb(k, r), ap[k], sb);
      sb = fm(P.vb(k, r), av[k], sb);
      sb = fm(P.bb(r, k), ab[k], sb);
    }
    y.p[r] = sp;
    y.v[r] = sv;
    y.b[r] = sb;
  }
}

template <typename D, typename T>
DEKF_HD void load_rec_dyn(const T *rec, size_t ns, M3<D> &R, V3<D> &as, V3<D> &dlt) {
#pragma unroll
  for (int f = 0; f < 9; ++f) R.a[f] = (D)rec[(REC_R + f) * ns];
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    as[f] = (D)rec[(REC_AS + f) * ns];
    dlt[f] = (D)rec[(REC_DLT + f) * ns];
  }
}

// One backward stage: reads x_{k+1}^s at xnext, writes x_k^s at xout (both [9] at stride n_out).  `ck` = filtered state of
// stage k ([54] at stride ns: P 45 incl. P_pp, x 9), `rec` = stage record k (stride ns); both already offset to the instance.
// Register budget: only z crosses from the factorisation phase to the product phase; P_k, the record and x_{k+1}^s are
// re-read where they are needed instead of being kept live.
template <typename D, typename T>
DEKF_HD void window_back_stage(const MheConst<D> &c, const T *ck, const T *rec, size_t ns, const double *xnext, double *xout,
                               size_t n_out) {
  const bool vo = rec[REC_FLAG * ns] != T(0);
  // z = Sigma^-1 (x^s_{k+1} - mu): (mu, Sigma) is the forward sweep's time update (+ VO row) of stage k, in D
  D z[9];
  {
    Cov9<D> Sg;
    Vec9<D> mu;
    {
      M3<D> R;
      V3<D> as, dlt;
      load_rec_dyn(rec, ns, R, as, dlt);
      load_state_as(ck, ns, Sg, mu);
      DefaultMath<D>::template prop<1>(c, Sg, mu, R, as, vo, dlt);
    }
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      z[f] = (D)xnext[f * n_out] - mu.p[f];
      z[3 + f] = (D)xnext[(3 + f) * n_out] - mu.v[f];
      z[6 + f] = (D)xnext[(6 + f) * n_out] - mu.b[f];
    }
    D Lc[45], dinv[9];  // packed lower Cholesky factor, row r at r (r + 1) / 2; reciprocal diagonal
#pragma unroll
    for (int r = 0; r < 9; ++r) {
#pragma unroll
      for (int cc = 0; cc <= r; ++cc) {
        D v = cov_at(Sg, r, cc);
#pragma unroll
        for (int k = 0; k < cc; ++k) v = fm(-Lc[r * (r + 1) / 2 + k], Lc[cc * (cc + 1) / 2 + k], v);
        if (cc == r) {
          const D d = sqrt(v);
          Lc[r * (r + 1) / 2 + r] = d;
          dinv[r] = D(1) / d;
        } else {
          Lc[r * (r + 1) / 2 + cc] = v * dinv[cc];
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 9; ++r) {
      D v = z[r];
#pragma unroll
      for (int k = 0; k < r; ++k) v = fm(-Lc[r * (r + 1) / 2 + k], z[k], v);
      z[r] = v * dinv[r];
    }
#pragma unroll
    for (int r = 8; r >= 0; --r) {
      D v = z[r];
#pragma unroll
      for (int k = r + 1; k < 9; ++k) v = fm(-Lc[k * (k + 1) / 2 + r], z[k], v);
      z[r] = v * dinv[r];
    }
  }
#if defined(__CUDA_ARCH__)
  asm volatile("" ::: "memory");  // a real re-read: keeps the compiler from holding the first loads live across the factorisation
#endif
  const D dt = c.dt, h = D(0.5) * c.dt * c.dt;
  M3<D> R;
  V3<D> as, dlt;
  load_rec_dyn(rec, ns, R, as, dlt);
  Cov9<D> P;
  Vec9<D> m;
  load_state_as(ck, ns, P, m);
  // a = A' z = [z_p;  dt z_p + z_v;  z_b - R' (h z_p + dt z_v)]
  V3<D> ap, av, ab;
  {
    V3<D> t;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      ap[r] = z[r];
      av[r] = fm(dt, z[r], z[3 + r]);
      t[r] = fm(h, z[r], dt * z[3 + r]);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) ab[r] = fm(-R(2, r), t[2], fm(-R(1, r), t[1], fm(-R(0, r), t[0], z[6 + r])));
  }
  Vec9<D> w = m;
  cov_mul_add(P, ap, av, ab, w);  // w = m + P A' z
  if (vo) {
    // rhs = nu - U' z = Delta - (L m + h a_s) - L (P A' z) - C1 z_p - C2 z_v;  L y = dt y_v - h R y_b
    S3<D> C1, C2, Sm;
#pragma unroll
    for (int f = 0; f < 6; ++f) C1.a[f] = C2.a[f] = Sm.a[f] = D(0);
    add_rot_diag(C1, R, c.n1);
    add_rot_diag(C2, R, c.n2);
    add_rot_diag(Sm, R, c.nvo);
    V3<D> rhs;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      // w - m = P A' z, so L m + L P A' z = L w
      const D Rwb = fm(R(r, 2), w.b[2], fm(R(r, 1), w.b[1], R(r, 0) * w.b[0]));
      D v = dlt[r] - fm(-h, Rwb, fm(h, as[r], dt * w.v[r]));
#pragma unroll
      for (int k = 0; k < 3; ++k) v = fm(-C2(r, k), z[3 + k], fm(-C1(r, k), z[k], v));
      rhs[r] = v;
    }
    // S = L P L' + C1 + R C_vo R' = dt^2 P_vv - h dt (E + E') + h^2 R P_bb R' + C1 + R C_vo R',  E = P_vb R'
    {
      M3<D> E, B;
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) {
          E(r, cc) = fm(P.vb(r, 2), R(cc, 2), fm(P.vb(r, 1), R(cc, 1), P.vb(r, 0) * R(cc, 0)));
          B(r, cc) = fm(R(r, 2), P.bb(2, cc), fm(R(r, 1), P.bb(1, cc), R(r, 0) * P.bb(0, cc)));
        }
      const D dt2 = dt * dt, hdt = h * dt, hh = h * h;
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = r; cc < 3; ++cc) {
          const int k = S3<D>::idx(r, cc);
          const D BR = fm(B(r, 2), R(cc, 2), fm(B(r, 1), R(cc, 1), B(r, 0) * R(cc, 0)));
          Sm.a[k] = fm(hh, BR, fm(-hdt, E(r, cc) + E(cc, r), fm(dt2, P.vv.a[k], Sm.a[k] + C1.a[k])));
        }
    }
    // q = S^-1 rhs (3x3 Cholesky)
    V3<D> q;
    {
      const D l00 = sqrt(Sm.a[0]), i0 = D(1) / l00;
      const D l10 = Sm.a[1] * i0, l20 = Sm.a[2] * i0;
      const D l11 = sqrt(fm(-l10, l10, Sm.a[3])), i1 = D(1) / l11;
      const D l21 = fm(-l20, l10, Sm.a[4]) * i1;
      const D l22 = sqrt(fm(-l21, l21, fm(-l20, l20, Sm.a[5]))), i2 = D(1) / l22;
      const D y0 = rhs[0] * i0;
      const D y1 = fm(-l10, y0, rhs[1]) * i1;
      const D y2 = fm(-l21, y1, fm(-l20, y0, rhs[2])) * i2;
      q[2] = y2 * i2;
      q[1] = fm(-l21, q[2], y1) * i1;
      q[0] = fm(-l20, q[2], fm(-l10, q[1], y0)) * i0;
    }
    // w += P L' q,  L' q = [0;  dt q;  -h R' q]
    V3<D> e0, ev, eb;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      e0[r] = D(0);
      ev[r] = dt * q[r];
      eb[r] = -h * fm(R(2, r), q[2], fm(R(1, r), q[1], R(0, r) * q[0]));
    }
    cov_mul_add(P, e0, ev, eb, w);
  }
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    xout[f * n_out] = (double)w.p[f];
    xout[(3 + f) * n_out] = (double)w.v[f];
    xout[(6 + f) * n_out] = (double)w.b[f];
  }
}

// FULL mode source of the filtered states: the forward sweep of update(T) from the arrival cost of its window (arr_P / arr_x
// after update(T) is the prior of x_{T-N+1}; Prior_0 while T < N), with the operations of mhe_solve_incr (P_pp carried), each
// stage's (P, x) stored into scr[k % N] ([N][54][ns]).  Bit-identical to the checkpoints of the incremental solve.
template <typename T, typename Math = DefaultMath<T>>
DEKF_HD void window_forward(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, int Tk, int i, T *scr) {
  GlobalStageSource<T> src(dm, b, i);
  Cov9<T> P;
  Vec9<T> x;
  mhe_solve_start(c, dm, b, Tk, i, P, x);
  const int k0 = Tk < dm.N ? 0 : Tk - dm.N + 1;
  const size_t ns = (size_t)dm.ns;
  for (int k = k0;; ++k) {
    S3<T> Lam;
    V3<T> eta;
    src.meas(0, k, Lam, eta);
    Math::meas(P, x, Lam, eta);
    T *base = scr + (size_t)(k % dm.N) * 54 * ns;
    store_cov(base, dm.ns, i, P);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      base[(45 + f) * ns + i] = x.p[f];
      base[(48 + f) * ns + i] = x.v[f];
      base[(51 + f) * ns + i] = x.b[f];
    }
    if (k == Tk) break;
    M3<T> R;
    V3<T> as, dlt;
    bool vo;
    src.rot(0, k, R);
    src.dyn(0, k, as, dlt, vo);
    Math::prop(c, P, x, R, as, vo, dlt);
  }
}

// Backward pass over the filtered states of stages Tk-K+1 .. Tk held in `ring` (slot k % slots, [slots][54][ns]).
template <typename T>
DEKF_HD void window_backward(const MheConst<double> &c64, const Dims &dm, const Buffers<T> &b, const T *ring, int slots, int Tk,
                             int i, double *xout, size_t n_out) {
  const int N = dm.N, K = Tk + 1 < N ? Tk + 1 : N, k0 = Tk - K + 1;
  const size_t ns = (size_t)dm.ns;
  {
    const T *top = ring + (size_t)(Tk % slots) * 54 * ns + i;  // x_T^s = m_T
    double *o = xout + (size_t)(Tk - k0) * 9 * n_out + i;
#pragma unroll
    for (int f = 0; f < 9; ++f) o[f * n_out] = (double)top[(45 + f) * ns];
  }
  for (int k = Tk - 1; k >= k0; --k) {
    double *o = xout + (size_t)(k - k0) * 9 * n_out + i;
    window_back_stage<double, T>(c64, ring + (size_t)(k % slots) * 54 * ns + i, b.win + (size_t)(k % dm.NW) * REC_SIZE * ns + i, ns,
                                 o + 9 * n_out, o, n_out);
  }
}

// Smoothed window of update(Tk) (Tk >= 1) for instance i: xout [K][9][n_out], row j = stage Tk-K+1+j, K = min(Tk+1, N).
// scr == nullptr: the filtered states are the checkpoint ring of the incremental solve (window_solve 1); otherwise the
// forward sweep above writes them into scr first (window_solve 0).  c: the handle's constants, c64: the same in double.
template <typename T>
DEKF_HD void mhe_window_smooth(const MheConst<T> &c, const MheConst<double> &c64, const Dims &dm, const Buffers<T> &b, T *scr,
                               int Tk, int i, double *xout, size_t n_out) {
  if (scr == nullptr) {
    window_backward<T>(c64, dm, b, b.ckpt, dm.NW, Tk, i, xout, n_out);
    return;
  }
  window_forward<T>(c, dm, b, Tk, i, scr);
#if defined(__CUDA_ARCH__)
  asm volatile("" ::: "memory");  // the backward pass reads the ring back; nothing of the forward sweep stays live
#endif
  window_backward<T>(c64, dm, b, scr, dm.N, Tk, i, xout, n_out);
}

// ------------------------------------------------------------------------------------------------
// Smoothed covariances (dekf_get_window_cov): for every window state the 9x9 block of the window QP's posterior covariance
// (the x_k block of the inverse of its KKT matrix over the equality rows, in the 1/2 z'Hz scaling under which M_p = P^-1).
// The covariance half of the RTS pass above, with its notation (P = P_k filtered, (mu, Sigma) the time update of stage k
// incl. the VO row when it is an equality, L = [0, dt I, -h R], S = L P L' + C1 + R C_vo R'):
//   P'_k = P - P L' S^-1 L P                        x_k conditioned on the VO row
//   C'   = P (A' - L' S^-1 U') = P'_k A' - P L' S^-1 [C1 C2 0]    Cov(x_k, x_{k+1}) conditioned on the VO row
//   G    = C' Sigma^-1,    P_k^s = P'_k - G (Sigma - P_{k+1}^s) G'
// (no VO row: P' = P, C' = P A'), P_T^s = P_T.  Row r of P' needs P L' S^-1 only through its own row q_r = S^-1 (L P)_{:,r},
// so P' is formed one row at a time and C' row r right after it.  Arithmetic in double, every multiply-add an explicit fm.
// Each output entry is written to (r, c) and (c, r) from one value, so every block is exactly symmetric.
// ------------------------------------------------------------------------------------------------
// packed upper triangle of a symmetric 9x9, row-major: (r, c), r <= c
DEKF_HD constexpr int sym9(int r, int c) { return r <= c ? r * (17 - r) / 2 + c : c * (17 - c) / 2 + r; }

// field of entry (r, c) of the dense 9x9 matrix in the stored layout of a Cov9 (store_cov: pp, vv, bb, pv, pb, vb)
DEKF_HD constexpr int cov_slot(int r, int c) {
  return r > c ? cov_slot(c, r)
               : (r / 3 == c / 3 ? 6 * (r / 3) + (r % 3 == 0 ? c % 3 : (r % 3 == 1 ? 2 + c % 3 : 5))
                                 : 18 + 9 * (r / 3 + c / 3 - 1) + 3 * (r % 3) + c % 3);
}

// One backward covariance stage: reads P_{k+1}^s at pnext, writes P_k^s at pout (both [81] row-major at stride n_out).  `ck`,
// `rec` as in window_back_stage.  `sh`: per-thread work area of 126 doubles at stride ss, G (row-major, [81]) then
// Sigma - P_{k+1}^s (sym9, [45]).  P'_k is parked in the upper triangle of pout between the first and the last phase.
// CROSS: also the lag-one cross-covariance Cov^s(x_k, x_{k+1}) = G P_{k+1}^s into cout ([81] row-major at stride n_out, rows
// over x_k): the smoothed x_k given x_{k+1} is x'_k + G (x_{k+1} - mu), so its covariance with x_{k+1} is G P_{k+1}^s.
template <typename D, typename T, bool CROSS = false>
DEKF_HD void window_cov_stage(const MheConst<D> &c, const T *ck, const T *rec, size_t ns, const double *pnext, double *pout,
                              size_t n_out, double *sh, size_t ss, double *cout = nullptr) {
  const bool vo = rec[REC_FLAG * ns] != T(0);
  const D dt = c.dt, h = D(0.5) * c.dt * c.dt;
  double *Gs = sh, *Ds = sh + 81 * ss;
  // phase 1: P' (upper triangle into pout) and C' (into G), one row at a time; P is read row by row from ck, the finished
  // entries left of the diagonal back from pout.  With a VO row, P L' is staged first in the Sigma - P^s area (free until
  // phase 2): PLs[(m * 3 + j) * ss] = dt P(m, v_j) - h (P_{m,b} R')_j
  {
    M3<D> R;
#pragma unroll
    for (int f = 0; f < 9; ++f) R.a[f] = (D)rec[(REC_R + f) * ns];
    S3<D> C1, C2;
#pragma unroll
    for (int f = 0; f < 6; ++f) C1.a[f] = C2.a[f] = D(0);
    double *PLs = Ds;
    D l00 = D(0), l10 = D(0), l20 = D(0), l11 = D(0), l21 = D(0), l22 = D(0), i0 = D(0), i1 = D(0), i2 = D(0);
    if (vo) {
      add_rot_diag(C1, R, c.n1);
      add_rot_diag(C2, R, c.n2);
#pragma unroll
      for (int r = 0; r < 9; ++r) {
        D pb[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) pb[k] = (D)ck[cov_slot(r, 6 + k) * ns];
#pragma unroll
        for (int j = 0; j < 3; ++j)
          PLs[(r * 3 + j) * ss] = (double)fm(-h, fm(pb[2], R(j, 2), fm(pb[1], R(j, 1), pb[0] * R(j, 0))), dt * (D)ck[cov_slot(r, 3 + j) * ns]);
      }
      // S = L (P L') + C1 + R C_vo R',  (L y)_r = dt y_{v,r} - h (R y_b)_r
      S3<D> Sm;
#pragma unroll
      for (int f = 0; f < 6; ++f) Sm.a[f] = D(0);
      add_rot_diag(Sm, R, c.nvo);
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int j = r; j < 3; ++j) {
          const D RPb = fm(R(r, 2), (D)PLs[(8 * 3 + j) * ss], fm(R(r, 1), (D)PLs[(7 * 3 + j) * ss], R(r, 0) * (D)PLs[(6 * 3 + j) * ss]));
          const int k = S3<D>::idx(r, j);
          Sm.a[k] = fm(-h, RPb, fm(dt, (D)PLs[((3 + r) * 3 + j) * ss], Sm.a[k] + C1.a[k]));
        }
      l00 = sqrt(Sm.a[0]);
      i0 = D(1) / l00;
      l10 = Sm.a[1] * i0;
      l20 = Sm.a[2] * i0;
      l11 = sqrt(fm(-l10, l10, Sm.a[3]));
      i1 = D(1) / l11;
      l21 = fm(-l20, l10, Sm.a[4]) * i1;
      l22 = sqrt(fm(-l21, l21, fm(-l20, l20, Sm.a[5])));
      i2 = D(1) / l22;
    }
#pragma unroll
    for (int r = 0; r < 9; ++r) {
#if defined(__CUDA_ARCH__)
      asm volatile("" ::: "memory");  // the entries of the earlier rows are re-read from pout, not kept in registers
#endif
      D y[9];  // row r of P'
#pragma unroll
      for (int cc = r; cc < 9; ++cc) y[cc] = (D)ck[cov_slot(r, cc) * ns];
      D q[3] = {D(0), D(0), D(0)};  // S^-1 (L P)_{:,r}
      if (vo) {
        const D y0 = (D)PLs[(r * 3 + 0) * ss] * i0;
        const D y1 = fm(-l10, y0, (D)PLs[(r * 3 + 1) * ss]) * i1;
        const D y2 = fm(-l21, y1, fm(-l20, y0, (D)PLs[(r * 3 + 2) * ss])) * i2;
        q[2] = y2 * i2;
        q[1] = fm(-l21, q[2], y1) * i1;
        q[0] = fm(-l20, q[2], fm(-l10, q[1], y0)) * i0;
#pragma unroll
        for (int cc = r; cc < 9; ++cc)
          y[cc] = fm(-q[2], (D)PLs[(cc * 3 + 2) * ss], fm(-q[1], (D)PLs[(cc * 3 + 1) * ss], fm(-q[0], (D)PLs[(cc * 3 + 0) * ss], y[cc])));
      }
#pragma unroll
      for (int cc = r; cc < 9; ++cc) pout[(r * 9 + cc) * n_out] = (double)y[cc];
#pragma unroll
      for (int cc = 0; cc < r; ++cc) y[cc] = (D)pout[(cc * 9 + r) * n_out];
      // C' row r = A P'_{:,r} - [C1 q; C2 q; 0],  A y = [y_p + dt y_v - h R y_b;  y_v - dt R y_b;  y_b]
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const D Rb = fm(R(j, 2), y[8], fm(R(j, 1), y[7], R(j, 0) * y[6]));
        D cp = fm(-h, Rb, fm(dt, y[3 + j], y[j]));
        D cv = fm(-dt, Rb, y[3 + j]);
        if (vo) {
          cp = fm(-C1(j, 2), q[2], fm(-C1(j, 1), q[1], fm(-C1(j, 0), q[0], cp)));
          cv = fm(-C2(j, 2), q[2], fm(-C2(j, 1), q[1], fm(-C2(j, 0), q[0], cv)));
        }
        Gs[(r * 9 + j) * ss] = (double)cp;
        Gs[(r * 9 + 3 + j) * ss] = (double)cv;
        Gs[(r * 9 + 6 + j) * ss] = (double)y[6 + j];
      }
    }
  }
#if defined(__CUDA_ARCH__)
  asm volatile("" ::: "memory");  // P' and C' are in memory; nothing of phase 1 stays live across the factorisation
#endif
  // phase 2: Sigma (the forward time update of stage k, in D), Sigma - P_{k+1}^s into Ds, Cholesky of Sigma in registers
  D Lc[45], dinv[9];  // packed lower factor, row r at r (r + 1) / 2; reciprocal diagonal
  {
    Cov9<D> Sg;
    Vec9<D> mu;
    {
      M3<D> R;
      V3<D> as, dlt;
      load_rec_dyn(rec, ns, R, as, dlt);
      load_state_as(ck, ns, Sg, mu);
      DefaultMath<D>::template prop<1>(c, Sg, mu, R, as, vo, dlt);
    }
#pragma unroll
    for (int r = 0; r < 9; ++r)
#pragma unroll
      for (int cc = r; cc < 9; ++cc) Ds[sym9(r, cc) * ss] = (double)(cov_at(Sg, r, cc) - (D)pnext[(r * 9 + cc) * n_out]);
#pragma unroll
    for (int r = 0; r < 9; ++r) {
#pragma unroll
      for (int cc = 0; cc <= r; ++cc) {
        D v = cov_at(Sg, r, cc);
#pragma unroll
        for (int k = 0; k < cc; ++k) v = fm(-Lc[r * (r + 1) / 2 + k], Lc[cc * (cc + 1) / 2 + k], v);
        if (cc == r) {
          const D d = sqrt(v);
          Lc[r * (r + 1) / 2 + r] = d;
          dinv[r] = D(1) / d;
        } else {
          Lc[r * (r + 1) / 2 + cc] = v * dinv[cc];
        }
      }
    }
  }
  // phase 3: G row j = Sigma^-1 C'_{j,:}' (Sigma symmetric), in place
#pragma unroll 1
  for (int j = 0; j < 9; ++j) {
    double *g = Gs + (size_t)j * 9 * ss;
    D z[9];
#pragma unroll
    for (int r = 0; r < 9; ++r) {
      D v = (D)g[r * ss];
#pragma unroll
      for (int k = 0; k < r; ++k) v = fm(-Lc[r * (r + 1) / 2 + k], z[k], v);
      z[r] = v * dinv[r];
    }
#pragma unroll
    for (int r = 8; r >= 0; --r) {
      D v = z[r];
#pragma unroll
      for (int k = r + 1; k < 9; ++k) v = fm(-Lc[k * (k + 1) / 2 + r], z[k], v);
      z[r] = v * dinv[r];
    }
#pragma unroll
    for (int r = 0; r < 9; ++r) g[r * ss] = (double)z[r];
  }
#if defined(__CUDA_ARCH__)
  asm volatile("" ::: "memory");
#endif
  // phase 4: P_k^s = P' - G (Sigma - P_{k+1}^s) G', one row of G (Sigma - P^s) at a time, upper triangle mirrored
  D Dm[45];
#pragma unroll
  for (int f = 0; f < 45; ++f) Dm[f] = (D)Ds[f * ss];
#pragma unroll 1
  for (int r = 0; r < 9; ++r) {
    D u[9];
    {
      D g[9];
#pragma unroll
      for (int l = 0; l < 9; ++l) g[l] = (D)Gs[(r * 9 + l) * ss];
#pragma unroll
      for (int mm = 0; mm < 9; ++mm) {
        D v = Dm[sym9(mm, 0)] * g[0];
#pragma unroll
        for (int l = 1; l < 9; ++l) v = fm(Dm[sym9(mm, l)], g[l], v);
        u[mm] = v;
      }
    }
#pragma unroll 1
    for (int cc = r; cc < 9; ++cc) {
      D v = (D)pout[(r * 9 + cc) * n_out];
#pragma unroll
      for (int l = 0; l < 9; ++l) v = fm(-(D)Gs[(cc * 9 + l) * ss], u[l], v);
      pout[(r * 9 + cc) * n_out] = (double)v;
      pout[(cc * 9 + r) * n_out] = (double)v;
    }
  }
  if constexpr (CROSS) {
    // phase 5: C_k = G P_{k+1}^s, one column of P_{k+1}^s in registers at a time, G re-read from the work area
#pragma unroll 1
    for (int cc = 0; cc < 9; ++cc) {
      D p[9];
#pragma unroll
      for (int l = 0; l < 9; ++l) p[l] = (D)pnext[(l * 9 + cc) * n_out];
#pragma unroll
      for (int r = 0; r < 9; ++r) {
        D v = (D)Gs[(r * 9) * ss] * p[0];
#pragma unroll
        for (int l = 1; l < 9; ++l) v = fm((D)Gs[(r * 9 + l) * ss], p[l], v);
        cout[(r * 9 + cc) * n_out] = (double)v;
      }
    }
  }
}

// Backward covariance pass over the filtered states of stages Tk-K+1 .. Tk in `ring` (as window_backward); pout [K][81][n_out].
// CROSS: also the lag-one blocks, cout [K-1][81][n_out] (block j = Cov(x_{Tk-K+1+j}, x_{Tk-K+2+j})), and block j of pout sits
// at slot j % pslots (pslots >= K: the whole window; 2: a two-block ring for a caller that wants the cross blocks only).
template <typename T, bool CROSS = false>
DEKF_HD void window_cov_backward(const MheConst<double> &c64, const Dims &dm, const Buffers<T> &b, const T *ring, int slots, int Tk,
                                 int i, double *pout, size_t n_out, double *sh, size_t ss, double *cout = nullptr, int pslots = 0) {
  const int N = dm.N, K = Tk + 1 < N ? Tk + 1 : N, k0 = Tk - K + 1;
  const size_t ns = (size_t)dm.ns;
  auto pblk = [&](int j) { return pout + (size_t)(CROSS ? j % pslots : j) * 81 * n_out + i; };
  {
    Cov9<double> P;  // P_T^s = P_T, widened
    Vec9<double> x;
    load_state_as(ring + (size_t)(Tk % slots) * 54 * ns + i, ns, P, x);
    double *o = pblk(Tk - k0);
#pragma unroll
    for (int r = 0; r < 9; ++r)
#pragma unroll
      for (int cc = 0; cc < 9; ++cc) o[(r * 9 + cc) * n_out] = cov_at(P, r, cc);
  }
  for (int k = Tk - 1; k >= k0; --k) {
    double *o = pblk(k - k0);
    window_cov_stage<double, T, CROSS>(c64, ring + (size_t)(k % slots) * 54 * ns + i,
                                       b.win + (size_t)(k % dm.NW) * REC_SIZE * ns + i, ns, pblk(k - k0 + 1), o, n_out, sh, ss,
                                       CROSS ? cout + (size_t)(k - k0) * 81 * n_out + i : nullptr);
  }
}

// Smoothed covariances of update(Tk) (Tk >= 1) for instance i: pout [K][81][n_out], block j = stage Tk-K+1+j, row-major over
// (p_s, v_s, accel bias).  Sources of the filtered states as in mhe_window_smooth; sh / ss: see window_cov_stage; CROSS,
// cout, pslots: see window_cov_backward.
template <typename T, bool CROSS = false>
DEKF_HD void mhe_window_cov(const MheConst<T> &c, const MheConst<double> &c64, const Dims &dm, const Buffers<T> &b, T *scr, int Tk,
                            int i, double *pout, size_t n_out, double *sh, size_t ss, double *cout = nullptr, int pslots = 0) {
  if (scr == nullptr) {
    window_cov_backward<T, CROSS>(c64, dm, b, b.ckpt, dm.NW, Tk, i, pout, n_out, sh, ss, cout, pslots);
    return;
  }
  window_forward<T>(c, dm, b, Tk, i, scr);
#if defined(__CUDA_ARCH__)
  asm volatile("" ::: "memory");
#endif
  window_cov_backward<T, CROSS>(c64, dm, b, scr, dm.N, Tk, i, pout, n_out, sh, ss, cout, pslots);
}

}  // namespace dekf
