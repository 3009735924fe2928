// Exact operation tally of the lag-one cross block of dekf_get_window_cross_cov, per stage and handle kind, obtained by
// instantiating the header functions with a counting scalar (add + mul + div + sqrt; the device's fused multiply-add counts
// 2): phase 5 of window_cov_stage (9-state; the stage with CROSS minus the stage without), ds columns of fw_cross_col (foot
// states, L = 1, 2, 4 legs), 9 columns of bw_cross_col and the full V C V' of rows handles (state-constrained).  Dev tool:
// tests/test_window_cross_cov.py checks the constants of tools/window_probe.py against it.  Not a product path.
#include <cmath>
#include <cstdio>
#include <vector>

struct Cnt {
  static long add, mul, div, sq;
  static void reset() { add = mul = div = sq = 0; }
  static long flops() { return add + mul + div + sq; }
};
long Cnt::add = 0, Cnt::mul = 0, Cnt::div = 0, Cnt::sq = 0;

struct CT {
  double v;
  CT() : v(0) {}
  CT(double x) : v(x) {}
  CT(int x) : v(x) {}
  explicit operator double() const { return v; }
  explicit operator float() const { return (float)v; }
};
inline CT operator+(CT a, CT b) { Cnt::add++; return CT(a.v + b.v); }
inline CT operator-(CT a, CT b) { Cnt::add++; return CT(a.v - b.v); }
inline CT operator*(CT a, CT b) { Cnt::mul++; return CT(a.v * b.v); }
inline CT operator/(CT a, CT b) { Cnt::div++; return CT(a.v / b.v); }
inline CT operator-(CT a) { return CT(-a.v); }
inline CT &operator+=(CT &a, CT b) { Cnt::add++; a.v += b.v; return a; }
inline CT &operator-=(CT &a, CT b) { Cnt::add++; a.v -= b.v; return a; }
inline CT &operator*=(CT &a, CT b) { Cnt::mul++; a.v *= b.v; return a; }
inline bool operator!=(CT a, CT b) { return a.v != b.v; }
inline bool operator==(CT a, CT b) { return a.v == b.v; }
inline CT sqrt(CT a) { Cnt::sq++; return CT(std::sqrt(a.v)); }

#include "../../decentralized_ekf_mhe_b200/csrc/host_setup.hpp"
#include "../../decentralized_ekf_mhe_b200/csrc/box_window.cuh"
namespace dekf {
template <>
inline void sincos_t<CT>(CT x, CT *s, CT *c) {
  *s = CT(std::sin(x.v));
  *c = CT(std::cos(x.v));
}
}  // namespace dekf
using namespace dekf;

template <int L>
long foot_cross() {
  constexpr int DS = FootWin<L>::DS, W = FootWin<L>::W;
  std::vector<CT> rec(W), g(DS), Pn(DS * DS);
  for (int w = 0; w < W; ++w) rec[w] = CT(1.0 + 1e-3 * w);
  for (int e = 0; e < DS * DS; ++e) Pn[e] = CT(e / DS == e % DS ? 1.0 : 0.0);
  Cnt::reset();
  for (int c = 0; c < DS; ++c) fw_cross_col<CT, L>(rec.data(), Pn.data(), DS, c, g.data());
  return Cnt::flops();
}

int main() {
  dekf_config cfg;
  fill_go1_defaults(&cfg);
  cfg.ekf_rate = 200;
  cfg.n_instances = 1;
  MheConst<CT> mc = make_mhe_const<CT>(cfg);
  Cov9<CT> P;
  for (int f = 0; f < 6; ++f) P.pp.a[f] = P.vv.a[f] = P.bb.a[f] = CT(f == 0 || f == 3 || f == 5 ? 1e-3 : 1e-5);
  for (int f = 0; f < 9; ++f) P.pv.a[f] = P.pb.a[f] = P.vb.a[f] = CT(1e-6 * (f + 1));
  M3<CT> R = quat_to_rot<CT>(CT(0.9), CT(0.1), CT(0.2), CT(0.3));
  V3<CT> as = v3<CT>(CT(0.1), CT(0.0), CT(0.2)), dlt = v3<CT>(CT(0.002), CT(0.0), CT(0.0));
  // the 9-state cross block: the same with and without a VO row
  std::vector<CT> ck(54), rec(REC_SIZE);
  store_cov(ck.data(), 1, 0, P);
  for (int f = 0; f < 9; ++f) ck[45 + f] = CT(0.1 * (f + 1));
  for (int f = 0; f < 9; ++f) rec[REC_R + f] = R.a[f];
  for (int f = 0; f < 3; ++f) {
    rec[REC_AS + f] = as[f];
    rec[REC_DLT + f] = dlt[f];
  }
  rec[REC_FLAG] = CT(0);
  double pn[81], po[81], co[81], sh[126];
  for (int e = 0; e < 81; ++e) pn[e] = (e / 9 == e % 9) ? 1e-4 : 0.0;
  Cnt::reset();
  window_cov_stage<CT, CT>(mc, ck.data(), rec.data(), 1, pn, po, 1, sh, 1);
  const long cov = Cnt::flops();
  Cnt::reset();
  window_cov_stage<CT, CT, true>(mc, ck.data(), rec.data(), 1, pn, po, 1, sh, 1, co);
  const long nine = Cnt::flops() - cov;
  // the constrained cross block and V C V'
  std::vector<CT> brec(BW_REC), Sn(81), t(9);
  std::vector<double> V(81);
  for (int e = 0; e < BW_REC; ++e) brec[e] = CT(1.0 + 1e-3 * e);
  for (int e = 0; e < 81; ++e) {
    Sn[e] = CT(e / 9 == e % 9 ? 1.0 : 0.0);
    V[e] = e / 9 == e % 9 ? 1.0 : 0.01;
  }
  Cnt::reset();
  for (int c = 0; c < 9; ++c) bw_cross_col<CT>(brec.data(), Sn.data(), 9, c, t.data());
  const long box = Cnt::flops();
  Cnt::reset();
  for (int r = 0; r < 9; ++r) {
    bw_vs_row<CT>(V.data(), Sn.data(), 9, 0, 0, r, t.data());
    for (int c = 0; c < 9; ++c) bw_dot9<CT>(t.data(), V.data() + c * 9);
  }
  const long vcvt = Cnt::flops();
  std::printf("{\"window_cross\": %ld, \"foot\": {\"1\": %ld, \"2\": %ld, \"4\": %ld}, \"box_cross\": %ld, "
              "\"box_rows_vcvt\": %ld}\n", nine, foot_cross<1>(), foot_cross<2>(), foot_cross<4>(), box, vcvt);
  return 0;
}
