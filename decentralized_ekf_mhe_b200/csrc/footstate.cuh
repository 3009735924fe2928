// leg_odom_type_ == 1: foot positions are part of the state (SURVEY.md 8f rank 2).
//
// Reference (decentral_legged_est/src/DecentralEst.cpp): dim_state_ = 9 + 3 * num_legs (:20), x = [p, v, b_a,
// p_foot_1 .. p_foot_L]; measurement rows  p_foot_i - p - v_i = R_sb fk_i  (A_meas = [-I 0 0 .. I ..], :101-111) with
// Q_meas,i = R (J_i C_enc_pos J_i')^-1 R' (:310-325, :550-564); the feet follow a random walk whose weight is
// R Q_foot_slide R' / dt^2 in stance and R Q_foot_swing R' / dt^2 in swing (:432-452); prior on the feet =
// first measurement with Q_foot_init (:316-323).  The KF alternative uses the same model (:676-683, :759-776,
// :845-853).
//
// Same reasoning as the 9-state path (estimator_core.cuh): the QP is a linear-Gaussian smoothing problem and only
// x_T is read, so update(T) is ONE forward sweep over the window from the arrival cost.  Here the sweep is carried in
// INFORMATION form (M, m) -- the swing-foot process variance dt^2 * (1e7)^2 = 2.5e9 next to 1e-6 position variances
// costs the covariance form its last six digits (measured: 2e-6 against the oracle), while the information form
// only ever adds the tiny weight 4e-10; (M, m) is also exactly the reference's arrival cost (M_p, n_p,
// MheSrb.hpp:86-87).  One stage = add the measurement rows (no inverse), eliminate x_k from the joint quadratic in
// (x_k, x_{k+1}) by a dense Cholesky of the 9+3L block.  State <= 21: the blocks live in thread-local memory, one
// instance per thread, plain loops, double arithmetic.
#pragma once
#include "box_solve.cuh"
#include "estimator_core.cuh"

namespace dekf {

// per-stage leg data of the foot-state model, ring [NW][FOOT_REC(L)][ns] (double) beside the common record
// (R_sb, a_s, VO displacement, VO flag live in Buffers::win as for leg_odom_type 0)
DEKF_HD constexpr int foot_rec_size(int L) { return 9 * L + 1; }  // per leg: b_meas 3, Q_meas 6 | contact bit mask

struct FootBuffers {
  double *leg;    // [NW][9L+1][ns]
  double *arr_M;  // [DS(DS+1)/2][ns] arrival cost M_p (packed lower); est_type 1: C_KF_^-1 after the correction
  double *arr_m;  // [DS][ns]         -n_p;                           est_type 1: C_KF_^-1 x_KF_
};

struct FootConst {
  BoxConst bc;                    // dt and the information-form constants of the 9 base states (box_dyn_blocks)
  double q_slide[3], q_swing[3];  // 1 / (dt^2 std^2): weight of the foot random walk, body axes (:438-448)
  double M0[9], M0_foot[3];       // Q_prior diagonal (:239-253, :313-322)
  int N, est_type;
};

// in-place lower Cholesky of an n x n (row-major, lower triangle used)
DEKF_HD bool foot_chol(double *S, int n) {
  for (int j = 0; j < n; ++j) {
    double d = S[j * n + j];
    for (int k = 0; k < j; ++k) d -= S[j * n + k] * S[j * n + k];
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    S[j * n + j] = d;
    const double id = 1.0 / d;
    for (int r = j + 1; r < n; ++r) {
      double v = S[r * n + j];
      for (int k = 0; k < j; ++k) v -= S[r * n + k] * S[j * n + k];
      S[r * n + j] = v * id;
    }
  }
  return true;
}

// ---- smoothed window of the foot-state model (dekf_get_foot_window) ----
// After its leg rows, stage k of the sweep eliminates x_k from the joint quadratic in (x_k, x_{k+1}) with Hxx = L L',
// Y = L^-1 Hxp, y = L^-1 g_x.  Conditioned on x_{k+1}, x_k is Gaussian with information Hxx and mean Hxx^-1 (g_x - Hxp x_{k+1}),
// so the window's optimum and posterior covariance follow backwards from x_T = M_T^-1 m_T, P_T = M_T^-1:
//   x_k = L^-T (y - Y x_{k+1}),      P_k = L^-T (I + Y P_{k+1} Y') L^-1.
// The stage record holds (L, Y, y) in FootWin<L>::W doubles, packed by column so that the lanes of a warp (lane r = row r,
// foot_window.cuh) touch consecutive words for every column:
//   L(r, c), r >= c          at fw_li(r, c) = lcol(c) + r - c, the diagonal as 1 / L_cc                  NL = DS (DS + 1) / 2
//   Y(r, c), r >= fw_rs(c)   at NL + ycol(c) + r - fw_rs(c); Hxp is block diagonal (base 9 x 9, one 3 x 3 block per foot)
//                            and L^-1 lower triangular, so Y(r, c) = 0 above the block of c                    NY
//   y_r                      at NL + NY + r                                                                     DS
// Go1 (DS = 21): 231 + 279 + 21 = 531 doubles per stage.
DEKF_HD constexpr int fw_rs(int c) { return c < 9 ? 0 : 9 + 3 * ((c - 9) / 3); }      // first row of Y's column c that can be nonzero
DEKF_HD constexpr int fw_ce(int r) { return r < 9 ? 9 : 9 + 3 * ((r - 9) / 3 + 1); }  // Y(r, c) = 0 for c >= fw_ce(r)
DEKF_HD constexpr int fw_lcol(int DS, int c) { return c * DS - c * (c - 1) / 2; }
DEKF_HD constexpr int fw_ycol(int DS, int c) {
  int o = 0;
  for (int k = 0; k < c; ++k) o += DS - fw_rs(k);
  return o;
}
template <int L>
struct FootWin {
  static constexpr int DS = 9 + 3 * L;
  static constexpr int NL = DS * (DS + 1) / 2;
  static constexpr int NY = fw_ycol(DS, DS);
  static constexpr int W = NL + NY + DS;  // doubles per stage
  DEKF_HD static constexpr int li(int r, int c) { return fw_lcol(DS, c) + r - c; }
  DEKF_HD static constexpr int yi(int r, int c) { return NL + fw_ycol(DS, c) + r - fw_rs(c); }
  DEKF_HD static constexpr int vi(int r) { return NL + NY + r; }
};

// stage record from the serial factors: Lm row-major lower Cholesky factor (L_rr on the diagonal), Y row-major, y
template <int L>
DEKF_HD void foot_win_record(const double *Lm, const double *Y, const double *y, double *rec) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS;
  for (int c = 0; c < DS; ++c) {
    rec[FW::li(c, c)] = 1.0 / Lm[c * DS + c];
    for (int r = c + 1; r < DS; ++r) rec[FW::li(r, c)] = Lm[r * DS + c];
    for (int r = fw_rs(c); r < DS; ++r) rec[FW::yi(r, c)] = Y[r * DS + c];
  }
  for (int r = 0; r < DS; ++r) rec[FW::vi(r)] = y[r];
}

// z = L^-T z (back substitution with the L of one stage record)
template <typename S, int L>
DEKF_HD void fw_back(const S *rec, S *z) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS;
#pragma unroll
  for (int r = DS - 1; r >= 0; --r) {
    S v = z[r];
#pragma unroll
    for (int k = r + 1; k < DS; ++k) v -= rec[FW::li(k, r)] * z[k];
    z[r] = v * rec[FW::li(r, r)];
  }
}

// backward mean stage: x = L^-T (y - Y xn), xn = x_{k+1}
template <typename S, int L>
DEKF_HD void fw_mean_stage(const S *rec, const S *xn, S *x) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS;
#pragma unroll
  for (int r = 0; r < DS; ++r) {
    S v = rec[FW::vi(r)];
#pragma unroll
    for (int c = 0; c < fw_ce(r); ++c) v -= rec[FW::yi(r, c)] * xn[c];
    x[r] = v;
  }
  fw_back<S, L>(rec, x);
}

// column j of G = L^-T (I + Y P Y'), P = P_{k+1} (full, row stride sp); P null: G = L^-T (for P_T = L^-T L^-1)
template <typename S, int L>
DEKF_HD void fw_cov_col(const S *rec, const S *P, int sp, int j, S *g) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS;
  if (P != nullptr) {
    S v[DS], w[DS];
#pragma unroll
    for (int c = 0; c < DS; ++c) v[c] = j >= fw_rs(c) ? rec[FW::yi(j, c)] : S(0.0);  // row j of Y
#pragma unroll
    for (int a = 0; a < DS; ++a) {  // w = P v
      S t = P[a * sp] * v[0];
#pragma unroll
      for (int c = 1; c < DS; ++c) t += P[a * sp + c] * v[c];
      w[a] = t;
    }
#pragma unroll
    for (int r = 0; r < DS; ++r) {  // e_j + Y w
      S t = r == j ? S(1.0) : S(0.0);
#pragma unroll
      for (int c = 0; c < fw_ce(r); ++c) t += rec[FW::yi(r, c)] * w[c];
      g[r] = t;
    }
  } else {
#pragma unroll
    for (int r = 0; r < DS; ++r) g[r] = r == j ? S(1.0) : S(0.0);
  }
  fw_back<S, L>(rec, g);
}

// column j of the lag-one cross-covariance C_k = Cov(x_k, x_{k+1}) = -L^-T Y P_{k+1} (x_k = L^-T (y - Y x_{k+1})), rows over
// x_k; P = P_{k+1} (full, row stride sp)
template <typename S, int L>
DEKF_HD void fw_cross_col(const S *rec, const S *P, int sp, int j, S *g) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS;
#pragma unroll
  for (int r = 0; r < DS; ++r) {  // Y P e_j
    S t = rec[FW::yi(r, 0)] * P[j];
#pragma unroll
    for (int c = 1; c < fw_ce(r); ++c) t += rec[FW::yi(r, c)] * P[c * sp + j];
    g[r] = t;
  }
  fw_back<S, L>(rec, g);
#pragma unroll
  for (int r = 0; r < DS; ++r) g[r] = -g[r];
}

// serial backward covariance stage: Pk = L^-T (I + Y Pn Y') L^-1 = L^-T G' (Pn null: L^-T L^-1), DS x DS row-major; Pk is
// written from its lower triangle, so every block is exactly symmetric
template <typename S, int L>
DEKF_HD void fw_cov_stage(const S *rec, const S *Pn, S *Pk) {
  constexpr int DS = 9 + 3 * L;
  S G[DS * DS], g[DS];
  for (int j = 0; j < DS; ++j) {
    fw_cov_col<S, L>(rec, Pn, DS, j, g);
    for (int r = 0; r < DS; ++r) G[r * DS + j] = g[r];
  }
  for (int c = 0; c < DS; ++c) {
    for (int r = 0; r < DS; ++r) g[r] = G[c * DS + r];
    fw_back<S, L>(rec, g);  // column c of Pk
    for (int r = c; r < DS; ++r) Pk[r * DS + c] = Pk[c * DS + r] = g[r];
  }
}

template <int L>
struct FootFilter {
  static constexpr int DS = 9 + 3 * L;
  double M[DS * DS];  // information matrix of the current state (full storage, kept symmetric)
  double m[DS];       // information vector: cost 1/2 x' M x - m' x
  bool ok = true;

  DEKF_HD void set_prior(const FootConst &fc, const double *leg_rec, size_t ns) {
    for (int f = 0; f < DS * DS; ++f) M[f] = 0.0;
    for (int f = 0; f < 9; ++f) {
      M[f * DS + f] = fc.M0[f];
      m[f] = 0.0;
    }
    for (int l = 0; l < L; ++l)
      for (int c = 0; c < 3; ++c) {
        M[(9 + 3 * l + c) * DS + 9 + 3 * l + c] = fc.M0_foot[c];
        m[9 + 3 * l + c] = fc.M0_foot[c] * leg_rec[(size_t)(9 * l + c) * ns];  // x_prior feet = b_meas of sample 0 (:321)
      }
  }
  DEKF_HD void load(const FootBuffers &fb, size_t ns, int i) {
    int p = 0;
    for (int r = 0; r < DS; ++r)
      for (int c = 0; c <= r; ++c) {
        const double v = fb.arr_M[(size_t)(p++) * ns + i];
        M[r * DS + c] = v;
        M[c * DS + r] = v;
      }
    for (int f = 0; f < DS; ++f) m[f] = fb.arr_m[(size_t)f * ns + i];
  }
  DEKF_HD void store(const FootBuffers &fb, size_t ns, int i) const {
    int p = 0;
    for (int r = 0; r < DS; ++r)
      for (int c = 0; c <= r; ++c) fb.arr_M[(size_t)(p++) * ns + i] = M[r * DS + c];
    for (int f = 0; f < DS; ++f) fb.arr_m[(size_t)f * ns + i] = m[f];
  }

  // rows  p_foot_l - p - v_l = b_l  with cost 1/2 v_l' Q_l v_l:  M += H' Q H,  m += H' Q b,  H = [-I .. I_l ..]
  DEKF_HD void meas_update(const double *leg_rec, size_t ns) {
    for (int l = 0; l < L; ++l) {
      const double *o = leg_rec + (size_t)(9 * l) * ns;
      const int f0 = 9 + 3 * l;
      const double Q[9] = {o[(size_t)3 * ns], o[(size_t)4 * ns], o[(size_t)5 * ns], o[(size_t)4 * ns], o[(size_t)6 * ns],
                           o[(size_t)7 * ns], o[(size_t)5 * ns], o[(size_t)7 * ns], o[(size_t)8 * ns]};
      const double bl[3] = {o[0], o[ns], o[2 * ns]};
      for (int r = 0; r < 3; ++r) {
        double qb = 0.0;
        for (int c = 0; c < 3; ++c) {
          const double q = Q[r * 3 + c];
          M[r * DS + c] += q;
          M[(f0 + r) * DS + f0 + c] += q;
          M[r * DS + f0 + c] -= q;
          M[(f0 + r) * DS + c] -= q;
          qb += q * bl[c];
        }
        m[r] -= qb;
        m[f0 + r] += qb;
      }
    }
  }

  // x = M^-1 m
  DEKF_HD void solve(double *x) {
    double Lc[DS * DS];
    for (int f = 0; f < DS * DS; ++f) Lc[f] = M[f];
    if (!foot_chol(Lc, DS)) ok = false;
    for (int r = 0; r < DS; ++r) {
      double v = m[r];
      for (int k = 0; k < r; ++k) v -= Lc[r * DS + k] * x[k];
      x[r] = v / Lc[r * DS + r];
    }
    for (int r = DS - 1; r >= 0; --r) {
      double v = x[r];
      for (int k = r + 1; k < DS; ++k) v -= Lc[k * DS + r] * x[k];
      x[r] = v / Lc[r * DS + r];
    }
  }

  // Eliminate x_k from  1/2 x'Mx - m'x + 1/2 |A x - x+ + c|^2_Q (+ 1/2 |p - p+ + Delta|^2_Qc): (M, m) becomes the
  // information of x_{k+1} (DecentralEst.cpp:387-484; marginalizeQP's Schur complement, MheSrb.cpp:475-713).
  // REC: also write the stage's factors L, Y, y into rec (FootWin<L> layout) for the window getter's backward passes.
  template <bool REC = false>
  DEKF_HD void propagate(const FootConst &fc, const double *R, const double *as, int contact_mask, bool vo, const double *dlt,
                         double *rec = nullptr) {
    BoxStage s;
    for (int f = 0; f < 9; ++f) s.R[f] = R[f];
    for (int f = 0; f < 3; ++f) {
      s.as[f] = as[f];
      s.dlt[f] = dlt[f];
      s.eta[f] = 0.0;
    }
    for (int f = 0; f < 6; ++f) s.Lam[f] = 0.0;
    s.vo = vo;
    double AtQA[81], E9[81], Qn9[81], rj[9], rn[9];
    box_dyn_blocks(fc.bc, s, AtQA, E9, Qn9, rj, rn);
    // Hxx = M + blkdiag(A9'Q9A9 (+Qc), Qf);  Hxp = blkdiag(E9, -Qf);  Hpp = blkdiag(Qn9, Qf)
    double Hxp[DS * DS], Hpp[DS * DS], gp[DS];
    for (int f = 0; f < DS * DS; ++f) Hxp[f] = Hpp[f] = 0.0;
    for (int r = 0; r < 9; ++r) {
      for (int c = 0; c < 9; ++c) {
        M[r * DS + c] += AtQA[r * 9 + c];
        Hxp[r * DS + c] = E9[r * 9 + c];
        Hpp[r * DS + c] = Qn9[r * 9 + c];
      }
      m[r] += rj[r];
      gp[r] = rn[r];
    }
    for (int l = 0; l < L; ++l) {
      const double *qf = (contact_mask >> l) & 1 ? fc.q_slide : fc.q_swing;
      const int f0 = 9 + 3 * l;
      for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) {
          const double q = R[r * 3 + 0] * R[c * 3 + 0] * qf[0] + R[r * 3 + 1] * R[c * 3 + 1] * qf[1] + R[r * 3 + 2] * R[c * 3 + 2] * qf[2];
          M[(f0 + r) * DS + f0 + c] += q;
          Hxp[(f0 + r) * DS + f0 + c] = -q;
          Hpp[(f0 + r) * DS + f0 + c] = q;
        }
        gp[f0 + r] = 0.0;
      }
    }
    if (!foot_chol(M, DS)) ok = false;  // M now holds L (lower), Hxx = L L'
    // Y = L^-1 Hxp (overwrites Hxp column by column), y = L^-1 gx (overwrites m)
    for (int c = 0; c < DS; ++c)
      for (int r = 0; r < DS; ++r) {
        double v = Hxp[r * DS + c];
        for (int k = 0; k < r; ++k) v -= M[r * DS + k] * Hxp[k * DS + c];
        Hxp[r * DS + c] = v / M[r * DS + r];
      }
    for (int r = 0; r < DS; ++r) {
      double v = m[r];
      for (int k = 0; k < r; ++k) v -= M[r * DS + k] * m[k];
      m[r] = v / M[r * DS + r];
    }
    if constexpr (REC) foot_win_record<L>(M, Hxp, m, rec);
    // M+ = Hpp - Y'Y,  m+ = gp - Y'y
    for (int r = 0; r < DS; ++r) {
      double v = gp[r];
      for (int k = 0; k < DS; ++k) v -= Hxp[k * DS + r] * m[k];
      gp[r] = v;
    }
    for (int r = 0; r < DS; ++r)
      for (int c = 0; c <= r; ++c) {
        double v = Hpp[r * DS + c];
        for (int k = 0; k < DS; ++k) v -= Hxp[k * DS + r] * Hxp[k * DS + c];
        Hpp[r * DS + c] = v;
      }
    for (int r = 0; r < DS; ++r) {
      m[r] = gp[r];
      for (int c = 0; c <= r; ++c) {
        M[r * DS + c] = Hpp[r * DS + c];
        M[c * DS + r] = Hpp[r * DS + c];
      }
    }
  }
};

template <typename T>
DEKF_HD void foot_common(const Dims &dm, const Buffers<T> &b, int k, int i, double *R, double *as, double *dlt, bool &vo) {
  const T *r = b.win + (size_t)(k % dm.NW) * REC_SIZE * dm.ns + i;
  const size_t ns = (size_t)dm.ns;
  for (int f = 0; f < 9; ++f) R[f] = (double)r[(REC_R + f) * ns];
  for (int f = 0; f < 3; ++f) {
    as[f] = (double)r[(REC_AS + f) * ns];
    dlt[f] = (double)r[(REC_DLT + f) * ns];
  }
  vo = r[REC_FLAG * ns] != T(0);
}

// update(T) (est_type 0: window sweep with marginalisation) or UpdateKF (est_type 1) for the foot-state model;
// writes x (9 + 3L rows) and the body velocity.
template <typename T, int L>
DEKF_HD int foot_solve(const FootConst &fc, const Dims &dm, const Buffers<T> &b, const FootBuffers &fb, const Inputs &in,
                       const Outputs &out, int Tk, int i) {
  constexpr int DS = 9 + 3 * L;
  const size_t ns = (size_t)dm.ns;
  const int n = dm.n, N = dm.N, RS = foot_rec_size(L);
  FootFilter<L> f;
  auto leg = [&](int k) { return fb.leg + (size_t)(k % dm.NW) * RS * ns + i; };
  double R[9], as[3], dlt[3], x[DS];
  bool vo;
  if (fc.est_type == 1) {
    if (Tk == 0) {
      f.set_prior(fc, leg(0), ns);
      f.meas_update(leg(0), ns);
    } else {
      f.load(fb, ns, i);
    }
    const int kp = Tk == 0 ? 0 : Tk - 1;
    foot_common(dm, b, kp, i, R, as, dlt, vo);
    f.propagate(fc, R, as, (int)leg(kp)[(size_t)(9 * L) * ns], false, dlt);
    f.meas_update(leg(Tk), ns);
    f.store(fb, ns, i);
  } else {
    int k0;
    if (Tk <= N) {  // the arrival cost is first written at T == N (marginalizeQP(0)); until then Prior_0 stands
      f.set_prior(fc, leg(0), ns);
      k0 = 0;
    } else {
      f.load(fb, ns, i);
      k0 = Tk - N;
    }
    for (int k = k0;; ++k) {
      f.meas_update(leg(k), ns);
      if (k == Tk) break;
      foot_common(dm, b, k, i, R, as, dlt, vo);
      f.propagate(fc, R, as, (int)leg(k)[(size_t)(9 * L) * ns], vo, dlt);
      if (k == Tk - N) f.store(fb, ns, i);  // marginalizeQP(T-N): (M_p, -n_p)
    }
  }
  f.solve(x);
  foot_common(dm, b, Tk, i, R, as, dlt, vo);
  const double om[3] = {in.gyro[i], in.gyro[(size_t)n + i], in.gyro[(size_t)2 * n + i]};
  const double *lever = fc.bc.lever;
  const double u[3] = {x[3] + (om[1] * lever[2] - om[2] * lever[1]), x[4] + (om[2] * lever[0] - om[0] * lever[2]),
                       x[5] + (om[0] * lever[1] - om[1] * lever[0])};
  int status = 0;
  double chk = 0.0;
  for (int c = 0; c < DS; ++c) chk += x[c];
  if (!f.ok || !(chk == chk) || !(chk - chk == 0.0)) status |= ST_NONFINITE;
  if (out.x != nullptr)
    for (int c = 0; c < DS; ++c) out.x[(size_t)c * n + i] = x[c];
  if (out.v_body != nullptr)
    for (int r = 0; r < 3; ++r) out.v_body[(size_t)r * n + i] = R[r * 3 + 0] * u[0] + R[r * 3 + 1] * u[1] + R[r * 3 + 2] * u[2];
  return status;
}

// Smoothed window of update(Tk) (est_type 0), serial form of dekf_get_foot_window: the K = min(Tk+1, N) states
// Tk-K+1 .. Tk.  The forward sweep of foot_solve from the arrival cost written by that update (the prior of x_{Tk-N+1};
// Prior_0 while Tk < N) records every stage into rec ([K][FootWin<L>::W], the last slot takes L_T); then the backward
// mean and covariance passes.  x: [K][DS] and P: [K][DS * DS] at element stride os (either may be null).  Row K-1 of x is
// foot_solve's x_T bit for bit.  C (may be null): the lag-one cross-covariances [K-1][DS * DS] at stride os (fw_cross_col).
template <typename T, int L>
DEKF_HD void foot_window_smooth(const FootConst &fc, const Dims &dm, const Buffers<T> &b, const FootBuffers &fb, int Tk, int i,
                                double *rec, double *x, double *P, size_t os, double *C = nullptr) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS, W = FW::W;
  const size_t ns = (size_t)dm.ns;
  const int N = dm.N, RS = foot_rec_size(L);
  const int K = Tk + 1 < N ? Tk + 1 : N, k0 = Tk - K + 1;
  FootFilter<L> f;
  auto leg = [&](int k) { return fb.leg + (size_t)(k % dm.NW) * RS * ns + i; };
  double R[9], as[3], dlt[3], xv[DS], xn[DS];
  bool vo;
  if (Tk >= N)
    f.load(fb, ns, i);
  else
    f.set_prior(fc, leg(0), ns);
  for (int k = k0;; ++k) {
    f.meas_update(leg(k), ns);
    if (k == Tk) break;
    foot_common(dm, b, k, i, R, as, dlt, vo);
    f.template propagate<true>(fc, R, as, (int)leg(k)[(size_t)(9 * L) * ns], vo, dlt, rec + (size_t)(k - k0) * W);
  }
  double Lc[DS * DS];  // the factor solve() forms, kept for P_T
  for (int e = 0; e < DS * DS; ++e) Lc[e] = f.M[e];
  foot_chol(Lc, DS);
  f.solve(xv);
  double *rT = rec + (size_t)(K - 1) * W;
  for (int c = 0; c < DS; ++c) {
    rT[FW::li(c, c)] = 1.0 / Lc[c * DS + c];
    for (int r = c + 1; r < DS; ++r) rT[FW::li(r, c)] = Lc[r * DS + c];
  }
  double Pn[DS * DS], Pk[DS * DS];
  if (x != nullptr)
    for (int c = 0; c < DS; ++c) x[((size_t)(K - 1) * DS + c) * os] = xv[c];
  if (P != nullptr || C != nullptr) {
    fw_cov_stage<double, L>(rT, nullptr, Pn);
    if (P != nullptr)
      for (int e = 0; e < DS * DS; ++e) P[((size_t)(K - 1) * DS * DS + e) * os] = Pn[e];
  }
  for (int j = K - 2; j >= 0; --j) {
    const double *rj = rec + (size_t)j * W;
    if (x != nullptr) {
      for (int c = 0; c < DS; ++c) xn[c] = xv[c];
      fw_mean_stage<double, L>(rj, xn, xv);
      for (int c = 0; c < DS; ++c) x[((size_t)j * DS + c) * os] = xv[c];
    }
    if (C != nullptr)
      for (int c = 0; c < DS; ++c) {
        double cg[DS];
        fw_cross_col<double, L>(rj, Pn, DS, c, cg);
        for (int r = 0; r < DS; ++r) C[((size_t)j * DS * DS + r * DS + c) * os] = cg[r];
      }
    if (P != nullptr || C != nullptr) {
      fw_cov_stage<double, L>(rj, Pn, Pk);
      for (int e = 0; e < DS * DS; ++e) {
        if (P != nullptr) P[((size_t)j * DS * DS + e) * os] = Pk[e];
        Pn[e] = Pk[e];
      }
    }
  }
}

}  // namespace dekf
