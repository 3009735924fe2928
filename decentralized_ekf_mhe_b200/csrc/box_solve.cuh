// State-constrained window solve (builder extension; BASELINE config 4 "active velocity constraints").
//
// The reference's inequality mechanism exists -- MHEproblem::addConstraints(name, lb, ub) with lb < ub,
// decentral_legged_est/src/MheSrb.cpp:58-68 -- but DecentralEst.cpp never exercises it (every shipped row is an
// equality with its own slack, SURVEY.md fact 4).  With cfg.v_box_enable the rows  lo <= v_s of x_k <= hi  are
// added for every state of the window at solve time (after marginalizeQP(T-N)); the arrival cost stays the
// unconstrained marginal, like the reference's marginalizeQP which only knows the rows it was written for.
//
// Method.  Slack elimination leaves a strictly convex QP in the window states only,
//     min 1/2 x' Hh x - r' x   s.t.  lo <= v_k <= hi,
// with Hh block tridiagonal (9x9 blocks).  It is solved EXACTLY by a primal-dual active-set iteration: fix the
// active velocity components at their bound, solve the remaining block-tridiagonal system by a block Cholesky
// (Riccati) recursion, read the multipliers off the gradient of the free problem, update the set, stop when the
// set repeats.  The active set of the previous tick, shifted with the window, is the warm start.  An ADMM
// splitting of the same problem (the reference's OSQP route; oracle/admm.c restates it) needs a median of 3,000
// iterations for eps 1e-9 on this problem class and still misses 1e-6 m/s in 3 % of the steps (DESIGN.md
// section 8); the active-set iteration needs 2-4 factorisations and returns the vertex solution itself.
//
// One estimator instance per thread; the 9x9 blocks live in thread-local arrays, the factor (L_j, F_j, y_j) of
// each window state is streamed through a per-instance scratch in HBM laid out [stage][135][instance].
// All arithmetic is double (also for fp32 handles: the information form needs it).
#pragma once
#include "estimator_core.cuh"

namespace dekf {

enum { BOX_FAC = 144 };  // per stage: L (45, packed lower) + F (81) + y/x (9) + the feasible iterate of the finite method (9)

struct BoxConst {
  int enable;
  int max_iter;
  double lo[3], hi[3];
  // double copies of the model constants (the information form is always carried in double)
  double dt;
  double qa[3], qb[3], qc[3];  // per-axis inverse of [[d1, d2],[d2, d3]]: (a, b; b, c)
  double qab[3];               // 1 / (dt^2 C_accel_bias)
  double qvo[3];               // 1 / vo_p_std^2
  double P0[9];
  double lever[3];             // p_imu_2_opti (cfg), v_body = R_sb (v_s + omega x lever)
  // general per-component bounds (cfg.x_box_* merged with cfg.v_box_*): bit a of mask9 bounds component a of every window
  // state (0..2 p_s, 3..5 v_s, 6..8 accel bias).  general != 0: a component outside v_s is bounded -> box_solve<T, true>.
  int mask9, general;
  double lo9[9], hi9[9];
  // general linear rows (dekf_add_state_rows): the solve runs in y = W x, where rows 0 .. nrows-1 are the components mask9 bounds;
  // BoxBuffers::V holds W^-1.  0: none.
  int nrows;
};

struct BoxBuffers {
  double *fac;       // [N][135][ns]
  uint8_t *act;      // [NW][ns]  bits 0-2: lower bound active on v_x,v_y,v_z; bits 3-5: upper bound
  int32_t *iters;    // [ns] factorisations of the last solve
  int32_t *nactive;  // [ns] active bounds of the last solve
  uint32_t *act32;   // [NW][ns]  general bounds only: bits 0-8 lower bound active on component a, bits 9-17 upper bound
  const double *V;   // [81] W^-1 of the row basis (general linear rows only, else nullptr)
  // [ns] how the last solve ended, for dekf_get_constrained_window: 0 converged, 1 iteration cap (x = the last minimiser),
  // 2 iteration cap inside the finite method (x = its feasible iterate, slot 135).  Null in builds that do not export the window.
  uint8_t *capped = nullptr;
};

// Active-set encodings.  GEN = false: the velocity box (uint8 masks, components 3..5 -- the layout k_box_team shares);
// GEN = true: any of the 9 state components (uint32 masks).
template <bool GEN>
struct BoxSet {
  static constexpr int NC = GEN ? 9 : 3;    // candidate components per state
  static constexpr int OFF = GEN ? 0 : 3;   // state index of candidate 0
  static constexpr int HB = GEN ? 512 : 8;  // bit of the upper bound of candidate 0
  DEKF_HD static bool active(int mask, int c) { return (mask & ((1 << c) | (HB << c))) != 0; }
  DEKF_HD static bool bounded(const BoxConst &bc, int c) { return GEN ? ((bc.mask9 >> c) & 1) != 0 : true; }
  DEKF_HD static double lo(const BoxConst &bc, int c) { return GEN ? bc.lo9[c] : bc.lo[c]; }
  DEKF_HD static double hi(const BoxConst &bc, int c) { return GEN ? bc.hi9[c] : bc.hi[c]; }
  DEKF_HD static double bound(const BoxConst &bc, int mask, int c) { return (mask & (HB << c)) ? hi(bc, c) : lo(bc, c); }
  DEKF_HD static int load(const BoxBuffers &bb, size_t at) { return GEN ? (int)bb.act32[at] : (int)bb.act[at]; }
  DEKF_HD static void store(const BoxBuffers &bb, size_t at, int m) {
    if (GEN)
      bb.act32[at] = (uint32_t)m;
    else
      bb.act[at] = (uint8_t)m;
  }
};

struct BoxStage {
  double R[9], as[3], Lam[6], eta[3], dlt[3];
  bool vo;
};

template <typename T>
DEKF_HD void box_load_stage(const Dims &dm, const Buffers<T> &b, int k, int i, BoxStage &s) {
  const T *r = b.win + (size_t)(k % dm.NW) * REC_SIZE * dm.ns + i;
  const size_t ns = (size_t)dm.ns;
  for (int f = 0; f < 9; ++f) s.R[f] = (double)r[(REC_R + f) * ns];
  for (int f = 0; f < 3; ++f) {
    s.as[f] = (double)r[(REC_AS + f) * ns];
    s.eta[f] = (double)r[(REC_ETA + f) * ns];
    s.dlt[f] = (double)r[(REC_DLT + f) * ns];
  }
  for (int f = 0; f < 6; ++f) s.Lam[f] = (double)r[(REC_LAM + f) * ns];
  s.vo = r[REC_FLAG * ns] != T(0);
}

// R diag(d) R' (3x3, row-major, full)
DEKF_HD void box_rdrt(const double *R, const double *d, double *out) {
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c)
      out[r * 3 + c] = R[r * 3 + 0] * d[0] * R[c * 3 + 0] + R[r * 3 + 1] * d[1] * R[c * 3 + 1] + R[r * 3 + 2] * d[2] * R[c * 3 + 2];
}

// Dynamics + VO rows between window states j and j+1 built from the record of state j:
//   w = A x_j - x_{j+1} + c,  cost 1/2 w' Q w  (DecentralEst.cpp:387-424);  vcam = p_j - p_{j+1} + Delta, cost 1/2 vcam' Qc vcam (:474-484)
// Outputs: AtQA (added to D_j), E = block (j, j+1) = -A'Q - [Qc 0; 0 0], Qn (added to D_{j+1}),
// rj (added to r_j) = -A'Q c - Qc Delta, rn (added to r_{j+1}) = Q c + Qc Delta.
DEKF_HD void box_dyn_blocks(const BoxConst &bc, const BoxStage &s, double *AtQA, double *E, double *Qn, double *rj, double *rn) {
  const double dt = bc.dt, h = 0.5 * bc.dt * bc.dt;
  double A[81], Q[81], AtQ[81];
  for (int f = 0; f < 81; ++f) A[f] = Q[f] = 0.0;
  for (int f = 0; f < 9; ++f) A[f * 9 + f] = 1.0;
  for (int r = 0; r < 3; ++r) {
    A[r * 9 + 3 + r] = dt;
    for (int c = 0; c < 3; ++c) {
      A[r * 9 + 6 + c] = -h * s.R[r * 3 + c];
      A[(3 + r) * 9 + 6 + c] = -dt * s.R[r * 3 + c];
    }
  }
  double Ra[9], Rb[9], Rc[9];
  box_rdrt(s.R, bc.qa, Ra);
  box_rdrt(s.R, bc.qb, Rb);
  box_rdrt(s.R, bc.qc, Rc);
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) {
      Q[r * 9 + c] = Ra[r * 3 + c];
      Q[r * 9 + 3 + c] = Rb[r * 3 + c];
      Q[(3 + r) * 9 + c] = Rb[r * 3 + c];
      Q[(3 + r) * 9 + 3 + c] = Rc[r * 3 + c];
    }
    Q[(6 + r) * 9 + 6 + r] = bc.qab[r];
  }
  for (int r = 0; r < 9; ++r)
    for (int c = 0; c < 9; ++c) {
      double v = 0.0;
      for (int k = 0; k < 9; ++k) v += A[k * 9 + r] * Q[k * 9 + c];
      AtQ[r * 9 + c] = v;
    }
  for (int r = 0; r < 9; ++r)
    for (int c = 0; c < 9; ++c) {
      double v = 0.0;
      for (int k = 0; k < 9; ++k) v += AtQ[r * 9 + k] * A[k * 9 + c];
      AtQA[r * 9 + c] = v;
      E[r * 9 + c] = -AtQ[r * 9 + c];
      Qn[r * 9 + c] = Q[r * 9 + c];
    }
  double cv[9];
  for (int f = 0; f < 3; ++f) {
    cv[f] = h * s.as[f];
    cv[3 + f] = dt * s.as[f];
    cv[6 + f] = 0.0;
  }
  for (int r = 0; r < 9; ++r) {
    double a = 0.0, q = 0.0;
    for (int k = 0; k < 9; ++k) {
      a += AtQ[r * 9 + k] * cv[k];
      q += Q[r * 9 + k] * cv[k];
    }
    rj[r] = -a;
    rn[r] = q;
  }
  if (s.vo) {
    double Qc[9];
    box_rdrt(s.R, bc.qvo, Qc);
    for (int r = 0; r < 3; ++r) {
      double qd = 0.0;
      for (int c = 0; c < 3; ++c) {
        AtQA[r * 9 + c] += Qc[r * 3 + c];
        Qn[r * 9 + c] += Qc[r * 3 + c];
        E[r * 9 + c] -= Qc[r * 3 + c];
        qd += Qc[r * 3 + c] * s.dlt[c];
      }
      rj[r] -= qd;
      rn[r] += qd;
    }
  }
}

// in-place lower Cholesky of a 9x9 (row-major, lower triangle used); returns false if not positive definite
DEKF_HD bool box_chol9(double *S) {
  for (int j = 0; j < 9; ++j) {
    double d = S[j * 9 + j];
    for (int k = 0; k < j; ++k) d -= S[j * 9 + k] * S[j * 9 + k];
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    S[j * 9 + j] = d;
    const double id = 1.0 / d;
    for (int r = j + 1; r < 9; ++r) {
      double v = S[r * 9 + j];
      for (int k = 0; k < j; ++k) v -= S[r * 9 + k] * S[j * 9 + k];
      S[r * 9 + j] = v * id;
    }
  }
  return true;
}

DEKF_HD double box_bound(const BoxConst &bc, int mask, int c) { return (mask & (8 << c)) ? bc.hi[c] : bc.lo[c]; }
DEKF_HD bool box_is_active(int mask, int c) { return (mask & ((1 << c) | (8 << c))) != 0; }

// Gaussian prior (Pa, xa) in information form: M = Pa^-1 (by Cholesky), m = sym(M) xa.  Returns status bits.
DEKF_HD int box_prior_info(const double *Pa /*81*/, const double *xa /*9*/, double *M /*81*/, double *mv /*9*/) {
  int status = 0;
  double L[81];
  for (int f = 0; f < 81; ++f) L[f] = Pa[f];
  if (!box_chol9(L)) status |= ST_NONFINITE;
  for (int c = 0; c < 9; ++c) {
    double y[9];
    for (int r = 0; r < 9; ++r) {
      double v = (r == c) ? 1.0 : 0.0;
      for (int k = 0; k < r; ++k) v -= L[r * 9 + k] * y[k];
      y[r] = v / L[r * 9 + r];
    }
    for (int r = 8; r >= 0; --r) {
      double v = y[r];
      for (int k = r + 1; k < 9; ++k) v -= L[k * 9 + r] * y[k];
      y[r] = v / L[r * 9 + r];
    }
    for (int r = 0; r < 9; ++r) M[r * 9 + c] = y[r];
  }
  for (int r = 0; r < 9; ++r) {
    double v = 0.0;
    for (int k = 0; k < 9; ++k) v += 0.5 * (M[r * 9 + k] + M[k * 9 + r]) * xa[k];
    mv[r] = v;
  }
  return status;
}

// Change of basis x = V y of the block system: A <- V' A V (9x9 row-major, in place), r <- V' r.
DEKF_HD void box_congruence(const double *V, double *A) {
  double t[81];
  for (int a = 0; a < 9; ++a)
    for (int b = 0; b < 9; ++b) {
      double v = 0.0;
      for (int k = 0; k < 9; ++k) v += V[k * 9 + a] * A[k * 9 + b];
      t[a * 9 + b] = v;
    }
  for (int a = 0; a < 9; ++a)
    for (int b = 0; b < 9; ++b) {
      double v = 0.0;
      for (int k = 0; k < 9; ++k) v += t[a * 9 + k] * V[k * 9 + b];
      A[a * 9 + b] = v;
    }
}
DEKF_HD void box_tvec(const double *V, double *r) {
  double t[9];
  for (int a = 0; a < 9; ++a) {
    double v = 0.0;
    for (int k = 0; k < 9; ++k) v += V[k * 9 + a] * r[k];
    t[a] = v;
  }
  for (int a = 0; a < 9; ++a) r[a] = t[a];
}
// One window state's contribution to the block system in the row basis (general linear rows): Ds = V' (Lam on the v block + A'QA) V,
// rs = V' (eta on v + r_j), and E, Dn, rn transformed alike.  `more`: there is a state j+1.
DEKF_HD void box_stage_rows(const BoxConst &bc, const BoxStage &s, const double *V, bool more, double *Ds, double *rs, double *E,
                            double *Dn, double *rn) {
  for (int f = 0; f < 81; ++f) Ds[f] = 0.0;
  for (int f = 0; f < 9; ++f) rs[f] = 0.0;
  if (more) {
    double rj[9];
    box_dyn_blocks(bc, s, Ds, E, Dn, rj, rn);
    for (int f = 0; f < 9; ++f) rs[f] = rj[f];
    box_congruence(V, E);
    box_congruence(V, Dn);
    box_tvec(V, rn);
  }
  for (int a = 0; a < 3; ++a) {
    for (int c = 0; c < 3; ++c) Ds[(3 + a) * 9 + 3 + c] += s.Lam[S3<double>::idx(a, c)];
    rs[3 + a] += s.eta[a];
  }
  box_congruence(V, Ds);
  box_tvec(V, rs);
}

// component a of x = V y (general linear rows: back from the row basis; x_T and the exported window use this one loop)
DEKF_HD double box_row_V(const double *V, const double *y, int a) {
  double v = 0.0;
  for (int k = 0; k < 9; ++k) v += V[a * 9 + k] * y[k];
  return v;
}

// Constrained solve over the window states k0 .. Tk (K = Tk - k0 + 1 <= N) with the Gaussian prior
// (Pa, xa) on x_k0.  Returns status bits; writes x_T to xT.
template <typename T, bool GEN = false>
DEKF_HD int box_solve(const BoxConst &bc, const Dims &dm, const Buffers<T> &b, const BoxBuffers &bb, int k0, int Tk, int i,
                      const double *Pa /*81*/, const double *xa /*9*/, double *xT /*9*/) {
  using BS = BoxSet<GEN>;
  constexpr int NC = BS::NC, OFF = BS::OFF;
  const size_t ns = (size_t)dm.ns;
  const int K = Tk - k0 + 1;
  int status = 0;
  // prior in information form: M = Pa^-1, m = M xa
  double M[81], mv[9];
  status |= box_prior_info(Pa, xa, M, mv);
  const bool rows = GEN && bc.nrows > 0;  // general linear rows: everything below happens in y = W x
  double Vm[81];
  if (rows) {
    for (int f = 0; f < 81; ++f) Vm[f] = bb.V[f];
    double Ms[81];
    for (int f = 0; f < 81; ++f) Ms[f] = 0.5 * (M[f] + M[(f % 9) * 9 + f / 9]);
    box_congruence(Vm, Ms);
    for (int f = 0; f < 81; ++f) M[f] = Ms[f];
    box_tvec(Vm, mv);
  }
  // warm start: masks of the previous tick stay attached to their stage (ring slot), the new state starts free
  BS::store(bb, (size_t)(Tk % dm.NW) * ns + i, 0);
  int iters = 0, nact = 0;
  bool converged = false;
  // general bounds: 0 = plain primal-dual rule; after kSafeIt iterations the finite primal active-set method takes over:
  // 1 = bounds are only added until the iterate is feasible, 2 = at a feasible equality-constrained minimiser: drop the bound with
  // the most negative multiplier (or stop), 3 = move from the feasible iterate xc towards the new minimiser, stopping at (and
  // adding) the first bound the segment crosses.  Monotone in the cost, finite on a strictly convex QP.
  int phase = 0;
  bool have_xc = false;  // the scratch holds a FEASIBLE iterate of the finite method (reported if the iteration cap is hit)
  for (int it = 0; it < bc.max_iter && !converged; ++it) {
    iters = it + 1;
    // ---- forward: assemble, apply the active set, block Cholesky
    double Dc[81], rc[9], Fp[81];  // carry into D_j / r_j from the rows (j-1, j); F_{j-1}
    for (int f = 0; f < 81; ++f) Dc[f] = 0.5 * (M[f] + M[(f % 9) * 9 + f / 9]);
    for (int f = 0; f < 9; ++f) rc[f] = mv[f];
    double yp[9];
    for (int j = 0; j < K; ++j) {
      const int k = k0 + j;
      BoxStage s;
      box_load_stage(dm, b, k, i, s);
      const int mask = BS::load(bb, (size_t)(k % dm.NW) * ns + i);
      const int mask_n = (j + 1 < K) ? BS::load(bb, (size_t)((k + 1) % dm.NW) * ns + i) : 0;
      double D[81], E[81], r[9], Dn[81], rn[9];
      for (int f = 0; f < 81; ++f) D[f] = Dc[f];
      for (int f = 0; f < 9; ++f) r[f] = rc[f];
      if (rows) {
        double Ds[81], rs[9];
        box_stage_rows(bc, s, Vm, j + 1 < K, Ds, rs, E, Dn, rn);
        for (int f = 0; f < 81; ++f) D[f] += Ds[f];
        for (int f = 0; f < 9; ++f) r[f] += rs[f];
      } else {
        // leg odometry rows: 1/2 v' Lam v - eta' v
        for (int a = 0; a < 3; ++a) {
          for (int c = 0; c < 3; ++c) D[(3 + a) * 9 + 3 + c] += s.Lam[S3<double>::idx(a, c)];
          r[3 + a] += s.eta[a];
        }
      }
      if (j + 1 < K) {
        if (!rows) {
          double AtQA[81], rj[9];
          box_dyn_blocks(bc, s, AtQA, E, Dn, rj, rn);
          for (int f = 0; f < 81; ++f) D[f] += AtQA[f];
          for (int f = 0; f < 9; ++f) r[f] += rj[f];
        }
        // fixed components of state j+1: move column to the right-hand side of state j, zero it
        for (int c = 0; c < NC; ++c)
          if (BS::active(mask_n, c)) {
            const double beta = BS::bound(bc, mask_n, c);
            for (int rr = 0; rr < 9; ++rr) {
              r[rr] -= E[rr * 9 + OFF + c] * beta;
              E[rr * 9 + OFF + c] = 0.0;
            }
          }
        // fixed components of state j: their row of E feeds the right-hand side of state j+1
        for (int c = 0; c < NC; ++c)
          if (BS::active(mask, c)) {
            const double beta = BS::bound(bc, mask, c);
            for (int cc = 0; cc < 9; ++cc) {
              rn[cc] -= E[(OFF + c) * 9 + cc] * beta;
              E[(OFF + c) * 9 + cc] = 0.0;
            }
          }
      }
      for (int c = 0; c < NC; ++c)
        if (BS::active(mask, c)) {
          const double beta = BS::bound(bc, mask, c);
          for (int rr = 0; rr < 9; ++rr) r[rr] -= D[rr * 9 + OFF + c] * beta;
        }
      for (int c = 0; c < NC; ++c)
        if (BS::active(mask, c)) {
          for (int rr = 0; rr < 9; ++rr) D[rr * 9 + OFF + c] = D[(OFF + c) * 9 + rr] = 0.0;
          D[(OFF + c) * 9 + OFF + c] = 1.0;
          r[OFF + c] = BS::bound(bc, mask, c);
        }
      // S_j = D_j - F_{j-1} F_{j-1}',  rhs_j = r_j - F_{j-1} y_{j-1}
      if (j > 0) {
        for (int rr = 0; rr < 9; ++rr) {
          for (int cc = 0; cc <= rr; ++cc) {
            double v = 0.0;
            for (int kk = 0; kk < 9; ++kk) v += Fp[rr * 9 + kk] * Fp[cc * 9 + kk];
            D[rr * 9 + cc] -= v;
          }
          double v = 0.0;
          for (int kk = 0; kk < 9; ++kk) v += Fp[rr * 9 + kk] * yp[kk];
          r[rr] -= v;
        }
      }
      if (!box_chol9(D)) status |= ST_NONFINITE;
      // y_j = L^-1 rhs
      for (int rr = 0; rr < 9; ++rr) {
        double v = r[rr];
        for (int kk = 0; kk < rr; ++kk) v -= D[rr * 9 + kk] * yp[kk];
        yp[rr] = v / D[rr * 9 + rr];
      }
      // F_j = E_j' L_j^-T  <=>  F_j L_j' = E_j'   (row rr of F: forward substitution over columns)
      if (j + 1 < K) {
        for (int rr = 0; rr < 9; ++rr)
          for (int cc = 0; cc < 9; ++cc) {
            double v = E[cc * 9 + rr];
            for (int kk = 0; kk < cc; ++kk) v -= Fp[rr * 9 + kk] * D[cc * 9 + kk];
            Fp[rr * 9 + cc] = v / D[cc * 9 + cc];
          }
        for (int f = 0; f < 81; ++f) Dc[f] = Dn[f];
        for (int f = 0; f < 9; ++f) rc[f] = rn[f];
      }
      // spill the factor of this state
      double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
      {
        int p = 0;
        for (int rr = 0; rr < 9; ++rr)
          for (int cc = 0; cc <= rr; ++cc) fj[(size_t)(p++) * ns] = D[rr * 9 + cc];
        if (j + 1 < K)
          for (int f = 0; f < 81; ++f) fj[(size_t)(45 + f) * ns] = Fp[f];
        for (int f = 0; f < 9; ++f) fj[(size_t)(126 + f) * ns] = yp[f];
      }
    }
    // ---- backward: x_j = L_j^-T (y_j - F_j' x_{j+1}); x_j overwrites y_j in the scratch
    double xn[9];
    for (int j = K - 1; j >= 0; --j) {
      const double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
      double L[81], y[9];
      {
        int p = 0;
        for (int rr = 0; rr < 9; ++rr)
          for (int cc = 0; cc <= rr; ++cc) L[rr * 9 + cc] = fj[(size_t)(p++) * ns];
      }
      for (int f = 0; f < 9; ++f) y[f] = fj[(size_t)(126 + f) * ns];
      if (j + 1 < K) {
        for (int cc = 0; cc < 9; ++cc) {
          double v = 0.0;
          for (int rr = 0; rr < 9; ++rr) v += fj[(size_t)(45 + rr * 9 + cc) * ns] * xn[rr];
          y[cc] -= v;
        }
      }
      for (int rr = 8; rr >= 0; --rr) {
        double v = y[rr];
        for (int kk = rr + 1; kk < 9; ++kk) v -= L[kk * 9 + rr] * xn[kk];
        xn[rr] = v / L[rr * 9 + rr];
      }
      double *fw = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
      for (int f = 0; f < 9; ++f) fw[(size_t)(126 + f) * ns] = xn[f];
      if (j == K - 1)
        for (int f = 0; f < 9; ++f) xT[f] = xn[f];
    }
    bool changed = false;
    nact = 0;
    if constexpr (GEN) {
      constexpr int kSafeIt = 8;
      if (phase == 0 && it >= kSafeIt) phase = 1;
      if (phase == 3) {
        // ---- line search of the finite method: xc (feasible) -> the minimiser just computed (x in the scratch)
        double alpha = 1.0;
        int bj = -1, bcmp = -1, bside = 0;
        for (int j = 0; j < K; ++j) {
          const double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
          const int mask = BS::load(bb, (size_t)((k0 + j) % dm.NW) * ns + i);
          for (int c = 0; c < 9; ++c) {
            if (!BS::bounded(bc, c) || BS::active(mask, c)) continue;
            const double xn_ = fj[(size_t)(126 + c) * ns], xc_ = fj[(size_t)(135 + c) * ns], d = xn_ - xc_;
            if (d > 0.0 && xn_ > BS::hi(bc, c)) {
              double t = (BS::hi(bc, c) - xc_) / d;
              t = t < 0.0 ? 0.0 : t;
              if (t < alpha) { alpha = t; bj = j; bcmp = c; bside = 1; }
            } else if (d < 0.0 && xn_ < BS::lo(bc, c)) {
              double t = (BS::lo(bc, c) - xc_) / d;
              t = t < 0.0 ? 0.0 : t;
              if (t < alpha) { alpha = t; bj = j; bcmp = c; bside = -1; }
            }
          }
        }
        for (int j = 0; j < K; ++j) {
          double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
          for (int c = 0; c < 9; ++c) {
            const double xn_ = fj[(size_t)(126 + c) * ns], xc_ = fj[(size_t)(135 + c) * ns];
            fj[(size_t)(135 + c) * ns] = bj < 0 ? xn_ : xc_ + alpha * (xn_ - xc_);
          }
        }
        if (bj >= 0) {  // blocked: the bound joins the set, the equality-constrained problem is solved again
          const size_t at = (size_t)((k0 + bj) % dm.NW) * ns + i;
          BS::store(bb, at, BS::load(bb, at) | (bside > 0 ? (BS::HB << bcmp) : (1 << bcmp)));
          continue;
        }
        phase = 2;
      }
      // ---- multipliers = gradient of the free cost w.r.t. every component of x_j: g_j = D_j x_j + E_{j-1}' x_{j-1} + E_j x_{j+1}
      // - r_j with the UNMODIFIED blocks of the block-tridiagonal system (re-assembled here exactly as in the forward pass).
      // Update rule: the plain primal-dual active set (add every violated bound, drop every bound whose multiplier has the
      // wrong sign) for the first kSafeIt iterations; it can cycle when many bounds of different components interact, so
      // afterwards the finite method above takes over: bounds are only ADDED until the iterate is feasible, then the ONE bound
      // with the most negative multiplier is dropped and the iterate moves by a line search (phase 3).
      const bool safe = phase >= 1;
      int drop_j = -1, drop_c = -1, added = 0;
      double drop_val = 0.0;
      double Dc[81], rc[9], Ep[81], xp[9];
      for (int f = 0; f < 81; ++f) Dc[f] = 0.5 * (M[f] + M[(f % 9) * 9 + f / 9]);
      for (int f = 0; f < 9; ++f) rc[f] = mv[f];
      for (int j = 0; j < K; ++j) {
        const int k = k0 + j;
        BoxStage s;
        box_load_stage(dm, b, k, i, s);
        double D[81], E[81], r[9], Dn[81], rn[9], xj[9], x1[9];
        const double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
        for (int f = 0; f < 9; ++f) xj[f] = fj[(size_t)(126 + f) * ns];
        for (int f = 0; f < 81; ++f) D[f] = Dc[f];
        for (int f = 0; f < 9; ++f) r[f] = rc[f];
        if (rows) {
          double Ds[81], rs[9];
          box_stage_rows(bc, s, Vm, j + 1 < K, Ds, rs, E, Dn, rn);
          for (int f = 0; f < 81; ++f) D[f] += Ds[f];
          for (int f = 0; f < 9; ++f) r[f] += rs[f];
        } else {
          for (int a = 0; a < 3; ++a) {
            for (int c = 0; c < 3; ++c) D[(3 + a) * 9 + 3 + c] += s.Lam[S3<double>::idx(a, c)];
            r[3 + a] += s.eta[a];
          }
        }
        if (j + 1 < K) {
          if (!rows) {
            double AtQA[81], rj[9];
            box_dyn_blocks(bc, s, AtQA, E, Dn, rj, rn);
            for (int f = 0; f < 81; ++f) D[f] += AtQA[f];
            for (int f = 0; f < 9; ++f) r[f] += rj[f];
          }
          const double *f1 = bb.fac + ((size_t)(j + 1) * BOX_FAC) * ns + i;
          for (int f = 0; f < 9; ++f) x1[f] = f1[(size_t)(126 + f) * ns];
        }
        const size_t at = (size_t)(k % dm.NW) * ns + i;
        const int mask = BS::load(bb, at);
        int nm = 0;
        for (int c = 0; c < 9; ++c) {
          if (!BS::bounded(bc, c)) continue;
          // gs: magnitude of the terms that cancel in g.  A multiplier within round-off of zero (degenerate bound) keeps its
          // constraint; the iterate is the same either way to within gtol / curvature.
          double g = -r[c], gs = fabs(r[c]);
          for (int cc = 0; cc < 9; ++cc) {
            const double t = D[c * 9 + cc] * xj[cc];
            g += t;
            gs += fabs(t);
          }
          if (j + 1 < K)
            for (int cc = 0; cc < 9; ++cc) {
              const double t = E[c * 9 + cc] * x1[cc];
              g += t;
              gs += fabs(t);
            }
          if (j > 0)
            for (int rr = 0; rr < 9; ++rr) {
              const double t = Ep[rr * 9 + c] * xp[rr];
              g += t;
              gs += fabs(t);
            }
          const double gtol = 1e-10 * gs;
          const bool up = (mask & (BS::HB << c)) != 0, dn = (mask & (1 << c)) != 0;
          if (up || dn) {
            const double mult = up ? -g : g;  // multiplier of the active bound
            bool keep = mult > -gtol;
            if (!keep && safe) {              // candidate for the single drop, most negative (scaled) multiplier wins
              const double v = mult / (gs > 0.0 ? gs : 1.0);
              if (drop_j < 0 || v < drop_val) {
                drop_val = v;
                drop_j = j;
                drop_c = c;
              }
              keep = true;
            }
            if (keep) nm |= up ? (BS::HB << c) : (1 << c);
          } else if (xj[c] > BS::hi(bc, c)) {
            nm |= (BS::HB << c);
            added++;
          } else if (xj[c] < BS::lo(bc, c)) {
            nm |= (1 << c);
            added++;
          }
          if (BS::active(nm, c)) nact++;
        }
        if (nm != mask) {
          changed = true;
          BS::store(bb, at, nm);
        }
        if (j + 1 < K) {
          for (int f = 0; f < 81; ++f) {
            Ep[f] = E[f];
            Dc[f] = Dn[f];
          }
          for (int f = 0; f < 9; ++f) {
            xp[f] = xj[f];
            rc[f] = rn[f];
          }
        }
      }
      if (safe && added == 0) {
        // feasible equality-constrained minimiser: it becomes the iterate xc of the finite method
        have_xc = true;
        for (int j = 0; j < K; ++j) {
          double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
          for (int c = 0; c < 9; ++c) fj[(size_t)(135 + c) * ns] = fj[(size_t)(126 + c) * ns];
        }
        if (drop_j >= 0) {
          const size_t at = (size_t)((k0 + drop_j) % dm.NW) * ns + i;
          BS::store(bb, at, BS::load(bb, at) & ~((1 << drop_c) | (BS::HB << drop_c)));
          nact--;
          changed = true;
          phase = 3;
        }
      } else if (safe) {
        phase = 1;  // something was violated (added): back to the feasibility phase
      }
    } else {
      // ---- multipliers = gradient of the free cost w.r.t. v_j, active-set update
      //   grad_v(j) = [M (x_0 - xa)]_v (j == 0) + Lam_j v_j - eta_j + [A'Q w_j]_v - [Q w_{j-1}]_v,
      //   w_j = A x_j - x_{j+1} + c_j  (the VO rows only touch p)
      double Qw_prev[3] = {0.0, 0.0, 0.0};
      for (int j = 0; j < K; ++j) {
        const int k = k0 + j;
        BoxStage s;
        box_load_stage(dm, b, k, i, s);
        double xj[9], x1[9];
        const double *fj = bb.fac + ((size_t)j * BOX_FAC) * ns + i;
        for (int f = 0; f < 9; ++f) xj[f] = fj[(size_t)(126 + f) * ns];
        double g[3];
        for (int a = 0; a < 3; ++a) {
          double v = -s.eta[a];
          for (int c = 0; c < 3; ++c) v += s.Lam[S3<double>::idx(a, c)] * xj[3 + c];
          g[a] = v - Qw_prev[a];
        }
        if (j == 0) {
          for (int a = 0; a < 3; ++a) {
            double v = -mv[3 + a];
            for (int c = 0; c < 9; ++c) v += 0.5 * (M[(3 + a) * 9 + c] + M[c * 9 + 3 + a]) * xj[c];
            g[a] += v;
          }
        }
        if (j + 1 < K) {
          const double *f1 = bb.fac + ((size_t)(j + 1) * BOX_FAC) * ns + i;
          for (int f = 0; f < 9; ++f) x1[f] = f1[(size_t)(126 + f) * ns];
          const double dt = bc.dt, h = 0.5 * bc.dt * bc.dt;
          double Rb[3], wp[3], wv[3];
          for (int a = 0; a < 3; ++a) Rb[a] = s.R[a * 3 + 0] * xj[6] + s.R[a * 3 + 1] * xj[7] + s.R[a * 3 + 2] * xj[8];
          for (int a = 0; a < 3; ++a) {
            wp[a] = xj[a] + dt * xj[3 + a] - h * Rb[a] - x1[a] + h * s.as[a];
            wv[a] = xj[3 + a] - dt * Rb[a] - x1[3 + a] + dt * s.as[a];
          }
          double Ra[9], Rbm[9], Rc[9];
          box_rdrt(s.R, bc.qa, Ra);
          box_rdrt(s.R, bc.qb, Rbm);
          box_rdrt(s.R, bc.qc, Rc);
          for (int a = 0; a < 3; ++a) {
            double qp = 0.0, qv = 0.0;
            for (int c = 0; c < 3; ++c) {
              qp += Ra[a * 3 + c] * wp[c] + Rbm[a * 3 + c] * wv[c];
              qv += Rbm[a * 3 + c] * wp[c] + Rc[a * 3 + c] * wv[c];
            }
            g[a] += dt * qp + qv;  // [A'Q w]_v = dt (Qw)_p + (Qw)_v
            Qw_prev[a] = qv;
          }
        }
        uint8_t *mp = bb.act + (size_t)(k % dm.NW) * ns + i;
        const int mask = *mp;
        int nm = 0;
        for (int c = 0; c < 3; ++c) {
          if (mask & (8 << c)) {
            if (-g[c] > 0.0) nm |= (8 << c);  // multiplier of the upper bound stays positive
          } else if (mask & (1 << c)) {
            if (g[c] > 0.0) nm |= (1 << c);
          } else if (xj[3 + c] > bc.hi[c]) {
            nm |= (8 << c);
          } else if (xj[3 + c] < bc.lo[c]) {
            nm |= (1 << c);
          }
          if (nm & ((1 << c) | (8 << c))) nact++;
        }
        if (nm != mask) {
          changed = true;
          *mp = (uint8_t)nm;
        }
      }
    }
    converged = !changed;
  }
  if (!converged) status |= ST_QP_MAXITER;
  if constexpr (GEN) {
    if (!converged && have_xc) {  // cap hit inside the finite method: report its feasible (not yet optimal) iterate, never a violated bound
      const double *fl = bb.fac + ((size_t)(K - 1) * BOX_FAC) * ns + i;
      for (int f = 0; f < 9; ++f) xT[f] = fl[(size_t)(135 + f) * ns];
    }
  }
  if (rows) {  // x_T = V y_T
    double xv[9];
    for (int a = 0; a < 9; ++a) xv[a] = box_row_V(Vm, xT, a);
    for (int a = 0; a < 9; ++a) xT[a] = xv[a];
  }
  bb.iters[i] = iters;
  bb.nactive[i] = nact;
  if (bb.capped != nullptr) bb.capped[i] = (status & ST_QP_MAXITER) ? (GEN && have_xc ? 2 : 1) : 0;
  return status;
}

// marginalizeQP(T-N) as one stage of the unconstrained covariance-form sweep (MheSrb.cpp:475-713; arrival cost updated
// in place), leaving the Gaussian prior (Pa, xa) on the first state k0 that remains in the window.
template <typename T, typename Math = DefaultMath<T>>
DEKF_HD void box_prepare(const MheConst<T> &c, const Dims &dm, const Buffers<T> &b, int Tk, int i, double *Pa /*81*/, double *xa /*9*/,
                         int &k0) {
  const int ns = dm.ns, N = dm.N;
  Cov9<T> P;
  Vec9<T> x;
  GlobalStageSource<T> src(dm, b, i);
  if (Tk < N) {
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
    k0 = 0;
  } else {
    load_cov(b.arr_P, ns, i, P);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      x.p[f] = b.arr_x[(size_t)f * ns + i];
      x.v[f] = b.arr_x[(size_t)(3 + f) * ns + i];
      x.b[f] = b.arr_x[(size_t)(6 + f) * ns + i];
    }
    const int km = Tk - N;
    S3<T> Lam;
    V3<T> eta, as, dlt;
    M3<T> R;
    bool vo;
    src.meas(0, km, Lam, eta);
    Math::meas(P, x, Lam, eta);
    src.rot(0, km, R);
    src.dyn(0, km, as, dlt, vo);
    Math::prop(c, P, x, R, as, vo, dlt);
    store_cov(b.arr_P, ns, i, P);
#pragma unroll
    for (int f = 0; f < 3; ++f) {
      b.arr_x[(size_t)f * ns + i] = x.p[f];
      b.arr_x[(size_t)(3 + f) * ns + i] = x.v[f];
      b.arr_x[(size_t)(6 + f) * ns + i] = x.b[f];
    }
    k0 = km + 1;
  }
  for (int r = 0; r < 3; ++r)
    for (int cc = 0; cc < 3; ++cc) {
      Pa[(0 + r) * 9 + 0 + cc] = (double)P.pp(r, cc);
      Pa[(3 + r) * 9 + 3 + cc] = (double)P.vv(r, cc);
      Pa[(6 + r) * 9 + 6 + cc] = (double)P.bb(r, cc);
      Pa[(0 + r) * 9 + 3 + cc] = Pa[(3 + cc) * 9 + 0 + r] = (double)P.pv(r, cc);
      Pa[(0 + r) * 9 + 6 + cc] = Pa[(6 + cc) * 9 + 0 + r] = (double)P.pb(r, cc);
      Pa[(3 + r) * 9 + 6 + cc] = Pa[(6 + cc) * 9 + 3 + r] = (double)P.vb(r, cc);
    }
  for (int f = 0; f < 3; ++f) {
    xa[f] = (double)x.p[f];
    xa[3 + f] = (double)x.v[f];
    xa[6 + f] = (double)x.b[f];
  }
}

// update(T) with the box rows: marginalizeQP(T-N) as one stage of the unconstrained covariance-form sweep
// (MheSrb.cpp:475-713), then the constrained solve over the states that remain in the window, getsolution(T) and the
// body-velocity read-out (DecentralEst.cpp:179-185).
template <typename T, typename Math = DefaultMath<T>>
DEKF_HD int mhe_solve_box(const MheConst<T> &c, const BoxConst &bc, const Dims &dm, const Buffers<T> &b, const BoxBuffers &bb,
                          const Inputs &in, const Outputs &out, int Tk, int i) {
  const int n = dm.n;
  double Pa[81], xa[9], xT[9];
  int k0;
  box_prepare<T, Math>(c, dm, b, Tk, i, Pa, xa, k0);
  GlobalStageSource<T> src(dm, b, i);
  int status = bc.general ? box_solve<T, true>(bc, dm, b, bb, k0, Tk, i, Pa, xa, xT) : box_solve<T, false>(bc, dm, b, bb, k0, Tk, i, Pa, xa, xT);
  M3<T> RT;
  src.rot(0, Tk, RT);
  double om[3];
  for (int f = 0; f < 3; ++f) om[f] = in.gyro[(size_t)f * n + i];
  const double *lever = bc.lever;
  const double u[3] = {xT[3] + (om[1] * lever[2] - om[2] * lever[1]), xT[4] + (om[2] * lever[0] - om[0] * lever[2]),
                       xT[5] + (om[0] * lever[1] - om[1] * lever[0])};
  double chk = 0.0;
  for (int f = 0; f < 9; ++f) chk += xT[f];
  if (!(chk == chk) || !(chk - chk == 0.0)) status |= ST_NONFINITE;
  if (out.x != nullptr)
    for (int f = 0; f < 9; ++f) out.x[(size_t)f * n + i] = xT[f];
  if (out.v_body != nullptr)
    for (int f = 0; f < 3; ++f)
      out.v_body[(size_t)f * n + i] = (double)RT(f, 0) * u[0] + (double)RT(f, 1) * u[1] + (double)RT(f, 2) * u[2];
  return status;
}

}  // namespace dekf
