// Window of a state-constrained handle (dekf_get_constrained_window): the optimum of every window state, its posterior
// covariance with the active bounds treated as equalities, and the active set, read from what the last active-set solve
// (box_solve in box_solve.cuh, box_team_solve in box_team.cuh) leaves in its per-instance scratch.
//
// The final factorisation of that solve is the block Cholesky factor of the window's reduced system H = L L', with L block
// lower bidiagonal: L_j on the diagonal, F_j below it (F_j L_j' = E_j', E_j the coupling of states j and j+1).  Components
// fixed at a bound have 1 on the diagonal of L_j and no coupling (row and column of E, D and F zeroed by the solve).  The
// x_k blocks of H^-1 follow backwards (selected inversion, the structure of the foot window's P_k of footstate.cuh):
//     S_{K-1} = L^-T L^-1,        S_j = L_j^-T (I + F_j' S_{j+1} F_j) L_j^-1,
// then the fixed components are zeroed: that is the x_k block of the inverse KKT matrix with the active bounds as
// equality rows.  Rows handles (dekf_add_state_rows) solve in y = W x: P = V S_y V' (V = W^-1) with the active y coordinates
// zeroed first, so a_i P = 0 for every active row i.
//
// Per stage the factor is copied into a stage record [126]: L packed lower by rows (L(r, c) at r (r + 1) / 2 + c) with the
// INVERSE diagonal, then F row-major.  Column j of G = L^-T (I + F' S F) is bw_cov_col, S_j = L^-T G' is one bw_back per
// column; S_j is written from its lower triangle, so every block is exactly symmetric.  Every multiply-add is an explicit
// fma (fm, estimator_core.cuh): the host build (-ffp-contract=off) performs the same operations as the device.
//
// Two scratch layouts: the serial solve's [N][BOX_FAC][ns] (SoA over instances, L with its diagonal, x at 126, the finite
// method's feasible iterate at 135) and the team solve's [ns][N][BOX_TFAC] (instance-major, inverse diagonal, x at
// BOX_TFAC_X).  The device reads both in team form: 9 lanes per instance, 3 instances per warp, lane r forms column r of G
// and column r of S_j, the team's record, S_{j+1} and G in shared memory.
#pragma once
#include "box_team.cuh"

namespace dekf {

enum { BW_REC = 126, BW_F = 45 };  // stage record: L (45, inverse diagonal) + F (81)

DEKF_HD constexpr int bw_li(int r, int c) { return r * (r + 1) / 2 + c; }

// z = L^-T z with the L of one stage record
template <typename S>
DEKF_HD void bw_back(const S *rec, S *z) {
#pragma unroll
  for (int r = 8; r >= 0; --r) {
    S v = z[r];
#pragma unroll
    for (int k = r + 1; k < 9; ++k) v = fm<S>(-rec[bw_li(k, r)], z[k], v);
    z[r] = v * rec[bw_li(r, r)];
  }
}

// column j of G = L^-T (I + F' Sn F), Sn = S_{j+1} (row stride sp); Sn null: G = L^-T (the last state of the window)
template <typename S>
DEKF_HD void bw_cov_col(const S *rec, const S *Sn, int sp, int j, S *g) {
  if (Sn != nullptr) {
    S v[9], w[9];
#pragma unroll
    for (int a = 0; a < 9; ++a) v[a] = rec[BW_F + a * 9 + j];  // column j of F
#pragma unroll
    for (int a = 0; a < 9; ++a) {  // w = Sn v
      S t = S(0.0);
#pragma unroll
      for (int c = 0; c < 9; ++c) t = fm<S>(Sn[a * sp + c], v[c], t);
      w[a] = t;
    }
#pragma unroll
    for (int r = 0; r < 9; ++r) {  // e_j + F' w
      S t = r == j ? S(1.0) : S(0.0);
#pragma unroll
      for (int a = 0; a < 9; ++a) t = fm<S>(rec[BW_F + a * 9 + r], w[a], t);
      g[r] = t;
    }
  } else {
#pragma unroll
    for (int r = 0; r < 9; ++r) g[r] = r == j ? S(1.0) : S(0.0);
  }
  bw_back<S>(rec, g);
}

// column j of the lag-one block C_j = Cov(x_j, x_{j+1}) = -L_j^-T F_j' S_{j+1}, the block (j, j+1) of H^-1 = L^-T L^-1 for
// L_{j+1,j} = F_j; Sn = S_{j+1} (row stride sp), rows of C over x_j
template <typename S>
DEKF_HD void bw_cross_col(const S *rec, const S *Sn, int sp, int j, S *g) {
  S w[9];
#pragma unroll
  for (int a = 0; a < 9; ++a) w[a] = Sn[a * sp + j];  // S_{j+1} e_j
#pragma unroll
  for (int r = 0; r < 9; ++r) {  // F' w
    S t = S(0.0);
#pragma unroll
    for (int a = 0; a < 9; ++a) t = fm<S>(rec[BW_F + a * 9 + r], w[a], t);
    g[r] = t;
  }
  bw_back<S>(rec, g);
#pragma unroll
  for (int r = 0; r < 9; ++r) g[r] = -g[r];
}

// row r of V Sz (Sz: S with the rows of the fixed coordinates fx and the columns of those of fxc zeroed: fx of stage j and
// fxc of stage j + 1 for the lag-one block C_j)
template <typename S>
DEKF_HD void bw_vs_row(const double *V, const S *Sm, int sp, int fx, int fxc, int r, S *t) {
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    S v = S(0.0);
#pragma unroll
    for (int b = 0; b < 9; ++b) v = fm<S>(S(V[r * 9 + b]), (((fx >> b) | (fxc >> k)) & 1) ? S(0.0) : Sm[b * sp + k], v);
    t[k] = v;
  }
}
// row r of V Sz for a covariance block (rows and columns of the fixed coordinates fx zeroed); P(r, c) = bw_dot9(t, row c
// of V) for c <= r, written to (r, c) and (c, r) from one value
template <typename S>
DEKF_HD void bw_vs_row(const double *V, const S *Sm, int sp, int fx, int r, S *t) {
  bw_vs_row<S>(V, Sm, sp, fx, fx, r, t);
}
template <typename S>
DEKF_HD S bw_dot9(const S *t, const double *v) {
  S s = S(0.0);
#pragma unroll
  for (int k = 0; k < 9; ++k) s = fm<S>(t[k], S(v[k]), s);
  return s;
}

// serial host form of one backward covariance stage: Sk = L^-T (I + F' Sn F) L^-1 (Sn null: L^-T L^-1), 9 x 9 row-major
template <typename S>
DEKF_HD void bw_cov_stage(const S *rec, const S *Sn, S *Sk) {
  S G[81], g[9];
  for (int j = 0; j < 9; ++j) {
    bw_cov_col<S>(rec, Sn, 9, j, g);
    for (int r = 0; r < 9; ++r) G[r * 9 + j] = g[r];
  }
  for (int c = 0; c < 9; ++c) {
    for (int r = 0; r < 9; ++r) g[r] = G[c * 9 + r];
    bw_back<S>(rec, g);  // column c of Sk
    for (int r = c; r < 9; ++r) Sk[r * 9 + c] = Sk[c * 9 + r] = g[r];
  }
}

// active-set word of the solve -> (public encoding: bit a lower bound of row a active, bit 9 + a upper bound; fixed coordinates)
DEKF_HD uint32_t bw_public_active(int m, bool gen) {
  return gen ? (uint32_t)m : (uint32_t)(((m & 7) << 3) | (((m >> 3) & 7) << 12));
}
DEKF_HD int bw_fixed(uint32_t pub) { return (int)((pub | (pub >> 9)) & 0x1ffu); }

// Where a scratch layout keeps what the getter reads.  SOA: the serial solve, [N][BOX_FAC][ns]; else the team solve,
// [ns][N][BOX_TFAC].  cap: the instance's bb.capped byte.
template <bool SOA>
struct BwLayout {
  const double *fac;
  size_t ns;
  int N;
  DEKF_HD const double *stage(int j, int i) const {
    return SOA ? fac + (size_t)j * BOX_FAC * ns + i : fac + ((size_t)i * N + j) * BOX_TFAC;
  }
  DEKF_HD size_t stride() const { return SOA ? ns : 1; }
  DEKF_HD int xslot(int cap) const { return SOA ? (cap == 2 ? 135 : 126) : BOX_TFAC_X; }
  // record element e of the stage whose factor starts at f (the serial solve keeps L_rr: 1 / L_rr here)
  DEKF_HD double rec(const double *f, int e) const {
    const double v = f[(size_t)e * stride()];
    if (!SOA) return v;
    const bool diag = e == 0 || e == 2 || e == 5 || e == 9 || e == 14 || e == 20 || e == 27 || e == 35 || e == 44;
    return diag ? 1.0 / v : v;
  }
};

DEKF_HD uint32_t bw_load_active(const BoxConst &bc, const BoxBuffers &bb, const Dims &dm, int k, int i) {
  const size_t at = (size_t)(k % dm.NW) * dm.ns + i;
  return bc.general ? bw_public_active((int)bb.act32[at], true) : bw_public_active((int)bb.act[at], false);
}

// Serial form (host build; the device runs box_window_team with the same per-column functions): window of update(Tk) for
// instance i.  x [K][9], P [K][81], act [K], C [K-1][81] (the lag-one blocks, rows of the components fixed at stage j and
// columns of those fixed at j+1 zeroed; rows handles: V C_y V' with the same zeroing in y) at element stride os (any may be
// null).
template <bool SOA>
DEKF_HD void box_window_serial(const BoxConst &bc, const Dims &dm, const BoxBuffers &bb, const BwLayout<SOA> &lay, int Tk, int i,
                               double *x, double *P, uint32_t *act, size_t os, double *C = nullptr) {
  const int N = dm.N, K = Tk + 1 < N ? Tk + 1 : N, k0 = Tk - K + 1;
  const int cap = bb.capped[i];
  const bool rows = bc.general && bc.nrows > 0;
  for (int j = 0; j < K; ++j) {
    const uint32_t pub = bw_load_active(bc, bb, dm, k0 + j, i);
    if (act != nullptr) act[(size_t)j * os] = pub;
    if (x != nullptr) {
      const double *f = lay.stage(j, i);
      double y[9];
      for (int a = 0; a < 9; ++a) y[a] = f[(size_t)(lay.xslot(cap) + a) * lay.stride()];
      for (int a = 0; a < 9; ++a) x[((size_t)j * 9 + a) * os] = rows ? box_row_V(bb.V, y, a) : y[a];
    }
  }
  if (P == nullptr && C == nullptr) return;
  double rec[BW_REC], Sn[81], Sk[81], t[9], Cz[81], g[9];
  int fxn = 0;  // fixed components of stage j + 1
  for (int j = K - 1; j >= 0; --j) {
    const double *f = lay.stage(j, i);
    for (int e = 0; e < BW_REC; ++e) rec[e] = lay.rec(f, e);
    const int fx = bw_fixed(bw_load_active(bc, bb, dm, k0 + j, i));
    if (C != nullptr && j < K - 1) {
      for (int c = 0; c < 9; ++c) {
        bw_cross_col<double>(rec, Sn, 9, c, g);
        for (int r = 0; r < 9; ++r) Cz[r * 9 + c] = g[r];
      }
      double *Cj = C + (size_t)j * 81 * os;
      for (int r = 0; r < 9; ++r) {
        if (rows) bw_vs_row<double>(bb.V, Cz, 9, fx, fxn, r, t);
        for (int c = 0; c < 9; ++c)
          Cj[(size_t)(r * 9 + c) * os] = cap ? NAN
                                        : rows ? bw_dot9<double>(t, bb.V + c * 9)
                                               : ((((fx >> r) | (fxn >> c)) & 1) ? 0.0 : Cz[r * 9 + c]);
      }
    }
    bw_cov_stage<double>(rec, j == K - 1 ? nullptr : Sn, Sk);
    fxn = fx;
    for (int e = 0; e < 81; ++e) Sn[e] = Sk[e];
    if (P == nullptr) continue;
    double *Pj = P + (size_t)j * 81 * os;
    for (int r = 0; r < 9; ++r) {
      if (rows) {
        bw_vs_row<double>(bb.V, Sk, 9, fx, r, t);
        for (int c = 0; c <= r; ++c) Pj[(size_t)(r * 9 + c) * os] = Pj[(size_t)(c * 9 + r) * os] = bw_dot9<double>(t, bb.V + c * 9);
      } else {
        for (int c = 0; c < 9; ++c) Pj[(size_t)(r * 9 + c) * os] = (((fx >> r) | (fx >> c)) & 1) ? 0.0 : Sk[r * 9 + c];
      }
    }
    if (cap)
      for (int e = 0; e < 81; ++e) Pj[(size_t)e * os] = NAN;
  }
}

#if defined(__CUDACC__)

enum { BW_SP = 9, BW_TEAM_WORDS = BW_REC + 2 * 81 };  // shared memory per team: record, S, G

// Team form: lane r (0..8) of the team of instance i; valid: the team owns a real instance (stores are predicated on it).
// sh: the team's BW_TEAM_WORDS doubles of shared memory.  Every lane of the warp runs the same instruction stream.
// CROSS: also the lag-one blocks into C [K-1][81] as in box_window_serial (P may then be null); lane r forms column r of
// C_j from S_{j+1} before the stage overwrites it, and rows handles pass it through the G area to form V C_y V'.
template <bool SOA, bool CROSS = false>
__device__ void box_window_team(const BoxConst &bc, const Dims &dm, const BoxBuffers &bb, const BwLayout<SOA> &lay, int Tk, int i,
                                bool valid, int r, double *sh, double *x, double *P, uint32_t *act, double *C = nullptr) {
  const int N = dm.N, K = Tk + 1 < N ? Tk + 1 : N, k0 = Tk - K + 1;
  const size_t n = (size_t)dm.n;
  const int cap = bb.capped[i];
  const bool rows = bc.general && bc.nrows > 0;
  if (valid && act != nullptr)
    for (int j = r; j < K; j += 9) act[(size_t)j * n + i] = bw_load_active(bc, bb, dm, k0 + j, i);
  if (x != nullptr) {
    for (int j = 0; j < K; ++j) {
      const double *f = lay.stage(j, i) + (size_t)lay.xslot(cap) * lay.stride();
      double xr;
      if (rows) {
        double y[9];
#pragma unroll
        for (int a = 0; a < 9; ++a) y[a] = f[(size_t)a * lay.stride()];
        xr = box_row_V(bb.V, y, r);
      } else {
        xr = f[(size_t)r * lay.stride()];
      }
      if (valid) x[((size_t)j * 9 + r) * n + i] = xr;
    }
  }
  if (!CROSS && P == nullptr) return;
  const bool wp = !CROSS || P != nullptr;
  double *srec = sh, *sS = sh + BW_REC, *sG = sS + 81;
  int fxn = 0;  // fixed components of stage j + 1
  for (int j = K - 1; j >= 0; --j) {
    const double *f = lay.stage(j, i);
    __syncwarp();  // every lane is done with the previous record and with G
    for (int e = r; e < BW_REC; e += 9) srec[e] = lay.rec(f, e);
    __syncwarp();
    double g[9], cg[9];
    if (CROSS && j < K - 1) bw_cross_col<double>(srec, sS, BW_SP, r, cg);  // column r of C_j
    bw_cov_col<double>(srec, j == K - 1 ? nullptr : sS, BW_SP, r, g);     // column r of G
#pragma unroll
    for (int a = 0; a < 9; ++a) sG[a * BW_SP + r] = g[a];
    __syncwarp();  // every lane has read S_{j+1} and written its column of G
#pragma unroll
    for (int a = 0; a < 9; ++a) g[a] = sG[r * BW_SP + a];  // row r of G
    bw_back<double>(srec, g);                              // column r of S_j
#pragma unroll
    for (int a = 0; a < 9; ++a)
      if (a >= r) sS[a * BW_SP + r] = sS[r * BW_SP + a] = g[a];
    __syncwarp();
    const int fx = bw_fixed(bw_load_active(bc, bb, dm, k0 + j, i));
    double *Pj = P + (size_t)j * 81 * n + i;
    if (wp && rows) {
      double t[9];
      bw_vs_row<double>(bb.V, sS, BW_SP, fx, r, t);
      for (int c = 0; c <= r; ++c) {
        const double v = bw_dot9<double>(t, bb.V + c * 9);
        if (valid) Pj[(size_t)(r * 9 + c) * n] = Pj[(size_t)(c * 9 + r) * n] = cap ? NAN : v;
      }
    } else if (wp && valid) {
#pragma unroll
      for (int c = 0; c < 9; ++c)
        Pj[(size_t)(r * 9 + c) * n] = cap ? NAN : ((((fx >> r) | (fx >> c)) & 1) ? 0.0 : sS[r * BW_SP + c]);
    }
    if constexpr (CROSS) {
      if (j < K - 1) {
        double *Cj = C + (size_t)j * 81 * n + i;
        if (rows) {  // G is consumed: its area takes C_y
#pragma unroll
          for (int a = 0; a < 9; ++a) sG[a * BW_SP + r] = cg[a];
          __syncwarp();
          double t[9];
          bw_vs_row<double>(bb.V, sG, BW_SP, fx, fxn, r, t);
#pragma unroll
          for (int c = 0; c < 9; ++c) {
            const double v = bw_dot9<double>(t, bb.V + c * 9);
            if (valid) Cj[(size_t)(r * 9 + c) * n] = cap ? NAN : v;
          }
        } else if (valid) {
#pragma unroll
          for (int a = 0; a < 9; ++a) Cj[(size_t)(a * 9 + r) * n] = cap ? NAN : ((((fx >> a) | (fxn >> r)) & 1) ? 0.0 : cg[a]);
        }
      }
      fxn = fx;
    }
  }
}

#endif  // __CUDACC__

}  // namespace dekf
