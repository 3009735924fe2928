// Foot-position-state model (leg_odom_type_ == 1, footstate.cuh), team form: ONE WARP per estimator instance.
//
// Same information-form sweep and the same operand values as FootFilter<L> in footstate.cuh (DecentralEst.cpp:101-111,
// :310-325, :387-484, :550-564; marginalizeQP's Schur complement, MheSrb.cpp:475-713), re-laid out like box_team.cuh: lane r
// of the warp owns ROW r of the DS x DS information matrix (DS = 9 + 3L <= 21) in registers, rows of other lanes arrive
// by warp shuffle.  One stage = add the measurement rows (row-local), then eliminate x_k from the joint quadratic in
// (x_k, x_{k+1}):  M+ = Hpp - Y'Y,  m+ = gp - Y'y  with  Hxx = L L',  Y = L^-1 Hxp,  y = L^-1 m.  Cholesky, both triangular
// solves and both Schur updates run in ONE right-looking loop over the DS columns: at column k lane k broadcasts 1/L_kk,
// its finished row of Y and y_k; every lane updates its rows of the trailing matrix, of Hxp and of M+ at once.
// The thread-per-instance kernel keeps five DS x DS blocks (14.8 KB) in thread-local memory; here nothing leaves registers
// between loading the arrival cost and storing it.
#pragma once
#include "box_team.cuh"
#include "footstate.cuh"

namespace dekf {

#if defined(__CUDACC__)

template <int DS, int K, bool REC = false>
struct FtFactor {
  // column K of the fused elimination (see header).  M: row r of Hxx (becomes L, inverse diagonal), X: row r of Hxp
  // (becomes Y), Mp: row r of M+ (starts as Hpp), m: rhs entry r (becomes y_r), gp: entry r of m+ (starts as gp).
  // REC: *rinv receives this lane's 1 / L_rr (for the window getter's stage record).
  static __device__ __forceinline__ void run(double (&M)[DS], double (&X)[DS], double (&Mp)[DS], double &m, double &gp, bool &ok, int r,
                                             double *rinv = nullptr) {
    const double inv = bt_shfl(rsqrt(M[K]), K);
    if (!(inv > 0.0) || !(inv - inv == 0.0)) ok = false;
    if (REC && r == K) *rinv = inv;
    const double Lrk = M[K] * inv;  // meaningful for r > K
    const double yk = bt_shfl(m * inv, K);
    if (r == K) m = yk;
    if (r > K) m -= Lrk * yk;
    // Hxp is block diagonal (base block 9 x 9, one 3 x 3 block per foot) and L^-1 is lower triangular: row K of Y is zero
    // to the right of the block that contains K
    constexpr int CE = K < 9 ? 9 : 9 + 3 * ((K - 9) / 3 + 1);
    double Yk[CE], ykr = 0.0;
#pragma unroll
    for (int c = 0; c < CE; ++c) {
      Yk[c] = bt_shfl(X[c] * inv, K);  // row K of Y (final: rows < K have been eliminated from it)
      if (c == r) ykr = Yk[c];         // Y[K][r]
    }
#pragma unroll
    for (int c = 0; c < CE; ++c) {
      if (r > K) X[c] -= Lrk * Yk[c];
      Mp[c] -= ykr * Yk[c];
    }
    gp -= ykr * yk;
#pragma unroll
    for (int c = K + 1; c < DS; ++c) {
      const double Lck = bt_shfl(Lrk, c);
      if (r >= c) M[c] -= Lrk * Lck;
    }
    FtFactor<DS, K + 1, REC>::run(M, X, Mp, m, gp, ok, r, rinv);
  }
};
template <int DS, bool REC>
struct FtFactor<DS, DS, REC> {
  static __device__ __forceinline__ void run(double (&)[DS], double (&)[DS], double (&)[DS], double &, double &, bool &, int, double *) {}
};

// x = M^-1 m by Cholesky + forward substitution (column loop) + backward substitution (row K broadcasts L[K][c] x_K)
template <int DS, int K>
struct FtSolveFwd {
  static __device__ __forceinline__ void run(double (&M)[DS], double &m, bool &ok, int r) {
    const double inv = bt_shfl(rsqrt(M[K]), K);
    if (!(inv > 0.0) || !(inv - inv == 0.0)) ok = false;
    double Lrk = M[K] * inv;
    if (r == K) Lrk = inv;  // keep 1 / L_kk on the diagonal
    M[K] = Lrk;
    const double yk = bt_shfl(m * inv, K);
    if (r == K) m = yk;
    if (r > K) m -= Lrk * yk;
#pragma unroll
    for (int c = K + 1; c < DS; ++c) {
      const double Lck = bt_shfl(Lrk, c);
      if (r >= c) M[c] -= Lrk * Lck;
    }
    FtSolveFwd<DS, K + 1>::run(M, m, ok, r);
  }
};
template <int DS>
struct FtSolveFwd<DS, DS> {
  static __device__ __forceinline__ void run(double (&)[DS], double &, bool &, int) {}
};
template <int DS, int K>
struct FtSolveBwd {
  // t: y_r minus the contributions of the x_k already known (k > K); returns x_r in t for r == K .. DS-1
  static __device__ __forceinline__ void run(const double (&M)[DS], double &t, int r) {
    const double xk = bt_shfl(t * M[K], K);  // lane K: t * (1 / L_KK)
    if (r == K) t = xk;
#pragma unroll
    for (int c = 0; c < K; ++c) {
      const double v = bt_shfl(M[c] * xk, K);  // L[K][c] x_K, held by lane K
      if (r == c) t -= v;
    }
    FtSolveBwd<DS, K - 1>::run(M, t, r);
  }
};
template <int DS>
struct FtSolveBwd<DS, -1> {
  static __device__ __forceinline__ void run(const double (&)[DS], double &, int) {}
};

template <int L>
struct FootTeam {
  static constexpr int DS = 9 + 3 * L;
  double M[DS];  // row r of the information matrix
  double m;      // entry r of the information vector
  bool ok = true;
  int r;         // lane = row (lanes >= DS shadow row DS-1 and never store)
  int t, mm;     // base rows: type p/v/b and axis; foot rows: leg and axis
  int leg;       // -1 for the base rows

  __device__ __forceinline__ void init(int lane) {
    r = lane < DS ? lane : DS - 1;
    if (r < 9) {
      t = r / 3;
      mm = r - 3 * t;
      leg = -1;
    } else {
      leg = (r - 9) / 3;
      mm = (r - 9) - 3 * leg;
      t = 3;
    }
  }
  __device__ __forceinline__ void set_prior(const FootConst &fc, const double *leg_rec, size_t ns) {
#pragma unroll
    for (int c = 0; c < DS; ++c) M[c] = 0.0;
    m = 0.0;
#pragma unroll
    for (int c = 0; c < 9; ++c)
      if (r == c) M[c] = fc.M0[c];
#pragma unroll
    for (int l = 0; l < L; ++l)
#pragma unroll
      for (int c = 0; c < 3; ++c)
        if (r == 9 + 3 * l + c) {
          M[9 + 3 * l + c] = fc.M0_foot[c];
          m = fc.M0_foot[c] * leg_rec[(size_t)(9 * l + c) * ns];
        }
  }
  __device__ __forceinline__ void load(const FootBuffers &fb, size_t ns, int i) {
#pragma unroll
    for (int c = 0; c < DS; ++c) {
      const int hi = r > c ? r : c, lo = r > c ? c : r;
      M[c] = fb.arr_M[(size_t)(hi * (hi + 1) / 2 + lo) * ns + i];
    }
    m = fb.arr_m[(size_t)r * ns + i];
  }
  __device__ __forceinline__ void store(const FootBuffers &fb, size_t ns, int i, bool valid, int lane) const {
    if (!valid || lane >= DS) return;
#pragma unroll
    for (int c = 0; c < DS; ++c)
      if (c <= r) fb.arr_M[(size_t)(r * (r + 1) / 2 + c) * ns + i] = M[c];
    fb.arr_m[(size_t)r * ns + i] = m;
  }
  // rows  p_foot_l - p - v_l = b_l  with cost 1/2 v_l' Q_l v_l:  M += H' Q H,  m += H' Q b,  H = [-I .. I_l ..]
  __device__ __forceinline__ void meas_update(const double *leg_rec, size_t ns) {
#pragma unroll
    for (int l = 0; l < L; ++l) {
      const double *o = leg_rec + (size_t)(9 * l) * ns;
      const double q3 = o[(size_t)3 * ns], q4 = o[(size_t)4 * ns], q5 = o[(size_t)5 * ns], q6 = o[(size_t)6 * ns], q7 = o[(size_t)7 * ns],
                   q8 = o[(size_t)8 * ns];
      const double b0 = o[0], b1 = o[ns], b2 = o[2 * ns];
      // row mm of Q_l and (Q_l b_l)[mm]
      const double qr0 = bt_sel3(mm, q3, q4, q5), qr1 = bt_sel3(mm, q4, q6, q7), qr2 = bt_sel3(mm, q5, q7, q8);
      const double qb = qr0 * b0 + qr1 * b1 + qr2 * b2;
      const bool prow = t == 0, frow = leg == l;
      const double sp = prow ? 1.0 : (frow ? -1.0 : 0.0);  // sign on the p columns
      const double sf = prow ? -1.0 : (frow ? 1.0 : 0.0);  // sign on the foot-l columns
      M[0] += sp * qr0;
      M[1] += sp * qr1;
      M[2] += sp * qr2;
      M[9 + 3 * l + 0] += sf * qr0;
      M[9 + 3 * l + 1] += sf * qr1;
      M[9 + 3 * l + 2] += sf * qr2;
      m += sf * qb;  // p rows: -Q b, foot rows: +Q b
    }
  }
  // eliminate x_k (see header); R, as, dlt, vo: the common stage record; contact_mask: bit l = leg l in stance.
  // REC: also write row r of the stage's factors L, Y, y into rec (FootWin<L> layout, footstate.cuh; rec null: this lane
  // takes part in the shuffles only)
  template <bool REC = false>
  __device__ __forceinline__ void propagate(const FootConst &fc, const double *R, const double *as, int contact_mask, bool vo, const double *dlt,
                                            double *rec = nullptr) {
    const BoxConst &bc = fc.bc;
    const double dt = bc.dt, h = 0.5 * bc.dt * bc.dt;
    double X[DS], Mp[DS], gp = 0.0;
#pragma unroll
    for (int c = 0; c < DS; ++c) X[c] = Mp[c] = 0.0;
    {  // base rows (r < 9): rows of A'QA, E, Q and the right-hand sides in closed form (as in box_team.cuh)
      const int tb = t < 3 ? t : 0, mb = mm;
      double Rm[3], Rcm[3], Sa[3], Sb[3], Sc[3], Sv[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        Rm[c] = bt_sel3(mb, R[0 * 3 + c], R[1 * 3 + c], R[2 * 3 + c]);
        Rcm[c] = bt_sel3(mb, R[c * 3 + 0], R[c * 3 + 1], R[c * 3 + 2]);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        Sa[c] = Rm[0] * bc.qa[0] * R[c * 3 + 0] + Rm[1] * bc.qa[1] * R[c * 3 + 1] + Rm[2] * bc.qa[2] * R[c * 3 + 2];
        Sb[c] = Rm[0] * bc.qb[0] * R[c * 3 + 0] + Rm[1] * bc.qb[1] * R[c * 3 + 1] + Rm[2] * bc.qb[2] * R[c * 3 + 2];
        Sc[c] = Rm[0] * bc.qc[0] * R[c * 3 + 0] + Rm[1] * bc.qc[1] * R[c * 3 + 1] + Rm[2] * bc.qc[2] * R[c * 3 + 2];
        Sv[c] = Rm[0] * bc.qvo[0] * R[c * 3 + 0] + Rm[1] * bc.qvo[1] * R[c * 3 + 1] + Rm[2] * bc.qvo[2] * R[c * 3 + 2];
      }
      const double qa_m = bt_sel3(mb, bc.qa[0], bc.qa[1], bc.qa[2]), qb_m = bt_sel3(mb, bc.qb[0], bc.qb[1], bc.qb[2]);
      const double qc_m = bt_sel3(mb, bc.qc[0], bc.qc[1], bc.qc[2]), qab_m = bt_sel3(mb, bc.qab[0], bc.qab[1], bc.qab[2]);
      const double kb_p = -(h * qa_m + dt * qb_m), kb_v = -(h * qb_m + dt * qc_m);
      double Qrow[9], AtQ[9], AtQA[9];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        Qrow[c] = tb == 0 ? Sa[c] : (tb == 1 ? Sb[c] : 0.0);
        Qrow[3 + c] = tb == 0 ? Sb[c] : (tb == 1 ? Sc[c] : 0.0);
        Qrow[6 + c] = (tb == 2 && c == mb) ? qab_m : 0.0;
        AtQ[c] = tb == 0 ? Sa[c] : (tb == 1 ? dt * Sa[c] + Sb[c] : kb_p * Rcm[c]);
        AtQ[3 + c] = tb == 0 ? Sb[c] : (tb == 1 ? dt * Sb[c] + Sc[c] : kb_v * Rcm[c]);
        AtQ[6 + c] = Qrow[6 + c];
      }
      bt_row_times_A(AtQ, R, dt, h, AtQA);
      double rj = 0.0, rn = 0.0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        rj -= AtQ[c] * (h * as[c]) + AtQ[3 + c] * (dt * as[c]);
        rn += Qrow[c] * (h * as[c]) + Qrow[3 + c] * (dt * as[c]);
      }
      double Erow[9], Qn[9];
#pragma unroll
      for (int c = 0; c < 9; ++c) {
        Erow[c] = -AtQ[c];  // row r of E = -A'Q (- Qc on the p block)
        Qn[c] = Qrow[c];
      }
      if (vo && tb == 0) {
        double qd = 0.0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          AtQA[c] += Sv[c];
          Qn[c] += Sv[c];
          Erow[c] -= Sv[c];
          qd += Sv[c] * dlt[c];
        }
        rj -= qd;
        rn += qd;
      }
      if (t < 3) {
#pragma unroll
        for (int c = 0; c < 9; ++c) {
          M[c] += AtQA[c];
          X[c] = Erow[c];
          Mp[c] = Qn[c];
        }
        m += rj;
        gp = rn;
      }
    }
    // foot rows: random walk of the foot position, weight R diag(q) R' (stance: q_slide, swing: q_swing)
#pragma unroll
    for (int l = 0; l < L; ++l) {
      const bool stance = (contact_mask >> l) & 1;
      const double q0 = stance ? fc.q_slide[0] : fc.q_swing[0], q1 = stance ? fc.q_slide[1] : fc.q_swing[1],
                   q2 = stance ? fc.q_slide[2] : fc.q_swing[2];
      if (leg == l) {
        const double r0 = bt_sel3(mm, R[0], R[3], R[6]), r1 = bt_sel3(mm, R[1], R[4], R[7]), r2 = bt_sel3(mm, R[2], R[5], R[8]);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const double q = r0 * R[c * 3 + 0] * q0 + r1 * R[c * 3 + 1] * q1 + r2 * R[c * 3 + 2] * q2;
          M[9 + 3 * l + c] += q;
          X[9 + 3 * l + c] = -q;
          Mp[9 + 3 * l + c] = q;
        }
      }
    }
    if constexpr (REC) {
      double inv = 0.0;
      FtFactor<DS, 0, true>::run(M, X, Mp, m, gp, ok, r, &inv);
      record(X, inv, rec);
    } else {
      FtFactor<DS, 0>::run(M, X, Mp, m, gp, ok, r);
    }
#pragma unroll
    for (int c = 0; c < DS; ++c) M[c] = Mp[c];
    m = gp;
  }
  // after FtFactor: M[c < r] is L(r, c) L_cc, M[r] is L_rr^2, X is row r of Hxp with the rows above eliminated (Y(r, :) L_rr) and
  // m is y_r; inv is 1 / L_rr as FtFactor broadcast it.  The stores of one column cover consecutive words.
  __device__ __forceinline__ void record(const double (&X)[DS], double inv, double *rec) const {
    using FW = FootWin<L>;
#pragma unroll
    for (int c = 0; c < DS; ++c) {
      const double ic = bt_shfl(inv, c);
      if (rec != nullptr && r >= c) rec[FW::li(r, c)] = r == c ? inv : M[c] * ic;
    }
    if (rec == nullptr) return;
#pragma unroll
    for (int c = 0; c < DS; ++c)
      if (r >= fw_rs(c)) rec[FW::yi(r, c)] = X[c] * inv;
    rec[FW::vi(r)] = m;
  }
  // x = M^-1 m; returns x_r (M is destroyed)
  __device__ __forceinline__ double solve() {
    FtSolveFwd<DS, 0>::run(M, m, ok, r);
    double tt = m;
    FtSolveBwd<DS, DS - 1>::run(M, tt, r);
    return tt;
  }
};

// update(T) / UpdateKF for the foot-state model by one warp; mirrors foot_solve() in footstate.cuh
template <typename T, int L>
__device__ int foot_team_solve(const FootConst &fc, const Dims &dm, const Buffers<T> &b, const FootBuffers &fb, const Inputs &in,
                               const Outputs &out, int Tk, int i, bool valid, int lane) {
  constexpr int DS = 9 + 3 * L;
  const size_t ns = (size_t)dm.ns;
  const int n = dm.n, N = dm.N, RS = foot_rec_size(L);
  FootTeam<L> f;
  f.init(lane);
  auto legp = [&](int k) { return fb.leg + (size_t)(k % dm.NW) * RS * ns + i; };
  double R[9], as[3], dlt[3];
  bool vo;
  if (fc.est_type == 1) {
    if (Tk == 0) {
      f.set_prior(fc, legp(0), ns);
      f.meas_update(legp(0), ns);
    } else {
      f.load(fb, ns, i);
    }
    const int kp = Tk == 0 ? 0 : Tk - 1;
    foot_common(dm, b, kp, i, R, as, dlt, vo);
    f.propagate(fc, R, as, (int)legp(kp)[(size_t)(9 * L) * ns], false, dlt);
    f.meas_update(legp(Tk), ns);
    f.store(fb, ns, i, valid, lane);
  } else {
    int k0;
    if (Tk <= N) {
      f.set_prior(fc, legp(0), ns);
      k0 = 0;
    } else {
      f.load(fb, ns, i);
      k0 = Tk - N;
    }
    for (int k = k0;; ++k) {
      f.meas_update(legp(k), ns);
      if (k == Tk) break;
      foot_common(dm, b, k, i, R, as, dlt, vo);
      f.propagate(fc, R, as, (int)legp(k)[(size_t)(9 * L) * ns], vo, dlt);
      if (k == Tk - N) f.store(fb, ns, i, valid, lane);  // marginalizeQP(T-N): (M_p, -n_p)
    }
  }
  const double xr = f.solve();
  foot_common(dm, b, Tk, i, R, as, dlt, vo);
  const unsigned bad = __ballot_sync(0xffffffffu, lane < DS && (!(xr == xr) || !(xr - xr == 0.0) || !f.ok));
  int status = bad ? ST_NONFINITE : 0;
  const double v0 = bt_shfl(xr, 3), v1 = bt_shfl(xr, 4), v2 = bt_shfl(xr, 5);
  if (valid && lane < DS) {
    if (out.x != nullptr) out.x[(size_t)lane * n + i] = xr;
    if (out.v_body != nullptr && lane < 3) {
      const double om0 = in.gyro[i], om1 = in.gyro[(size_t)n + i], om2 = in.gyro[(size_t)2 * n + i];
      const double *lever = fc.bc.lever;
      const double u0 = v0 + (om1 * lever[2] - om2 * lever[1]), u1 = v1 + (om2 * lever[0] - om0 * lever[2]),
                   u2 = v2 + (om0 * lever[1] - om1 * lever[0]);
      out.v_body[(size_t)lane * n + i] = bt_sel3(lane, R[0], R[3], R[6]) * u0 + bt_sel3(lane, R[1], R[4], R[7]) * u1 +
                                         bt_sel3(lane, R[2], R[5], R[8]) * u2;
    }
  }
  return status;
}

#endif  // __CUDACC__

}  // namespace dekf
