// Smoothed window of the foot-position-state model (leg_odom_type 1, dekf_get_foot_window), team form: ONE WARP per
// instance, lane r owns row r as in foot_team.cuh.  Three phases in one launch:
//   1. forward sweep from the arrival cost (Prior_0 while T < N) through the same FootTeam meas_update / propagate as the
//      step, each stage writing its factors L, Y, y (FootWin<L> layout, footstate.cuh) into a device ring
//      [N-1][ns][W] -- instance-major within a stage, so that the warp's stores and loads of one stage are coalesced;
//   2. backward mean pass  x_k = L^-T (y - Y x_{k+1});
//   3. backward covariance pass  P_k = L^-T (I + Y P_{k+1} Y') L^-1  (only when P or C is requested), starting from
//      P_T = L_T^-T L_T^-1 with the factor of M_T that solve() leaves in registers; with WC, lane j first forms column j of
//      the lag-one block C_k = -L^-T Y P_{k+1} (fw_cross_col) from P_{k+1} before the stage overwrites it.
// Per stage the warp copies the record into shared memory; the backward passes then read it with warp-uniform addresses
// (broadcasts) or, for row j of Y, consecutive ones.  The mean pass runs redundantly in every lane (no shuffles); in the
// covariance pass lane j forms column j of G = L^-T (I + Y P Y'), G goes through shared memory to transpose, and lane c
// forms column c of P_k = L^-T G' and writes it as (r, c) and (c, r) from one value.  The arithmetic of the backward
// passes is fw_mean_stage / fw_cov_col / fw_back of footstate.cuh, the functions of the serial form.
#pragma once
#include "foot_team.cuh"

namespace dekf {

#if defined(__CUDACC__)

// shared memory per warp: the stage record, P_{k+1}, the transpose buffer (row stride DS | 1: odd, conflict-free) and x_{k+1}
template <int L>
__host__ __device__ constexpr int foot_win_smem_words() {
  return FootWin<L>::W + 2 * FootWin<L>::DS * (FootWin<L>::DS | 1) + FootWin<L>::DS;
}

// P_k from the record in srec and P_{k+1} in sP (null: P_T = L^-T L^-1); overwrites sP with P_k
template <int L>
__device__ __forceinline__ void foot_win_cov_team(const double *srec, double *sP, bool first, double *sG, int lane) {
  constexpr int DS = FootWin<L>::DS, SP = DS | 1;
  const int j = lane < DS ? lane : DS - 1;
  double g[DS];
  fw_cov_col<double, L>(srec, first ? nullptr : sP, SP, j, g);
  __syncwarp();  // every lane has read P_{k+1}
  if (lane < DS) {
#pragma unroll
    for (int r = 0; r < DS; ++r) sG[r * SP + j] = g[r];
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < DS; ++r) g[r] = sG[j * SP + r];  // row j of G
  fw_back<double, L>(srec, g);                          // column j of P_k
  if (lane < DS) {
#pragma unroll
    for (int r = 0; r < DS; ++r)
      if (r >= j) sP[r * SP + j] = sP[j * SP + r] = g[r];
  }
  __syncwarp();
}

// WX / WP: store the window / its covariances; WC: store the lag-one cross-covariances [K-1][DS * DS] at Cout (the covariance
// pass then runs whether or not WP is set)
template <int L, bool WX, bool WP, bool WC = false>
__device__ void foot_window_team(const FootConst &fc, const Dims &dm, const Buffers<double> &b, const FootBuffers &fb, double *ring,
                                 int Tk, int i, int lane, double *sh, double *xout, double *Pout, double *Cout = nullptr) {
  using FW = FootWin<L>;
  constexpr int DS = FW::DS, W = FW::W, SP = DS | 1;
  double *srec = sh, *sP = sh + W, *sG = sP + DS * SP, *sX = sG + DS * SP;
  const size_t ns = (size_t)dm.ns, n = (size_t)dm.n;
  const int N = dm.N, RS = foot_rec_size(L);
  const int K = Tk + 1 < N ? Tk + 1 : N, k0 = Tk - K + 1;
  const bool st = lane < DS;
  FootTeam<L> f;
  f.init(lane);
  auto legp = [&](int k) { return fb.leg + (size_t)(k % dm.NW) * RS * ns + i; };
  double R[9], as[3], dlt[3];
  bool vo;
  // phase 1: the step's sweep over the window (update(Tk) wrote the arrival cost of x_{Tk-N+1} at its stage Tk-N)
  if (Tk >= N)
    f.load(fb, ns, i);
  else
    f.set_prior(fc, legp(0), ns);
  for (int k = k0;; ++k) {
    f.meas_update(legp(k), ns);
    if (k == Tk) break;
    foot_common(dm, b, k, i, R, as, dlt, vo);
    f.template propagate<true>(fc, R, as, (int)legp(k)[(size_t)(9 * L) * ns], vo, dlt,
                               st ? ring + ((size_t)(k - k0) * ns + i) * W : nullptr);
  }
  const double xr = f.solve();  // x_T exactly as the step computed it; f.M: row r of L_T, 1 / L_rr on the diagonal
  if constexpr (WX) {  // x_{k+1} lives in shared memory between stages, not in registers across the covariance pass
    if (st) {
      sX[lane] = xr;
      xout[((size_t)(K - 1) * DS + lane) * n + i] = xr;
    }
  }
  if constexpr (WP || WC) {
    if (st) {
#pragma unroll
      for (int c = 0; c < DS; ++c)
        if (c <= lane) srec[FW::li(lane, c)] = f.M[c];
    }
    __syncwarp();
    foot_win_cov_team<L>(srec, sP, true, sG, lane);
    if (WP && st) {
#pragma unroll
      for (int c = 0; c < DS; ++c) Pout[(((size_t)(K - 1) * DS + lane) * DS + c) * n + i] = sP[lane * SP + c];
    }
  }
  // phases 2 and 3: stages Tk-1 .. Tk-K+1
  for (int j = K - 2; j >= 0; --j) {
    __syncwarp();  // every lane is done with the previous record
    const double *g = ring + ((size_t)j * ns + i) * W;
    for (int w = lane; w < W; w += 32) srec[w] = g[w];
    __syncwarp();
    if constexpr (WX) {
      double xv[DS];
      fw_mean_stage<double, L>(srec, sX, xv);
      double mine = xv[0];
#pragma unroll
      for (int c = 1; c < DS; ++c)
        if (c == lane) mine = xv[c];
      __syncwarp();  // every lane has read x_{k+1}
      if (st) {
        sX[lane] = mine;
        xout[((size_t)j * DS + lane) * n + i] = mine;
      }
    }
    if constexpr (WC) {
      double cg[DS];
      fw_cross_col<double, L>(srec, sP, SP, st ? lane : DS - 1, cg);  // column `lane` of C_j, from P_{j+1}
      if (st) {
#pragma unroll
        for (int r = 0; r < DS; ++r) Cout[(((size_t)j * DS + r) * DS + lane) * n + i] = cg[r];
      }
    }
    if constexpr (WP || WC) {
      foot_win_cov_team<L>(srec, sP, false, sG, lane);
      if (WP && st) {
#pragma unroll
        for (int c = 0; c < DS; ++c) Pout[(((size_t)j * DS + lane) * DS + c) * n + i] = sP[lane * SP + c];
      }
    }
  }
}

#endif  // __CUDACC__

}  // namespace dekf
