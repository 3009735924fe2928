// Exact operation tally of one backward stage of the smoothed-covariance getter (dekf_get_window_cov, window_cov_stage in
// csrc/estimator_core.cuh) without and with a VO row, obtained by instantiating it with the counting scalar of
// window_flopcount.cpp.  Dev tool: prints the constants tools/window_probe.py uses (tests/test_window_covariance.py keeps them
// in sync).  Not a product path.
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
namespace dekf {
template <>
inline void sincos_t<CT>(CT x, CT *s, CT *c) {
  *s = CT(std::sin(x.v));
  *c = CT(std::cos(x.v));
}
}  // namespace dekf
using namespace dekf;

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
  // one backward covariance stage without / with a VO row; the count does not depend on the values
  long f_cov[2];
  for (int v = 0; v < 2; ++v) {
    std::vector<CT> ck(54), rec(REC_SIZE);
    store_cov(ck.data(), 1, 0, P);
    for (int f = 0; f < 9; ++f) ck[45 + f] = CT(0.1 * (f + 1));
    for (int f = 0; f < 9; ++f) rec[REC_R + f] = R.a[f];
    for (int f = 0; f < 3; ++f) {
      rec[REC_AS + f] = as[f];
      rec[REC_DLT + f] = dlt[f];
    }
    rec[REC_FLAG] = CT(v);
    double pn[81], po[81], sh[126];
    for (int e = 0; e < 81; ++e) pn[e] = (e / 9 == e % 9) ? 1e-4 : 0.0;
    Cnt::reset();
    window_cov_stage<CT, CT>(mc, ck.data(), rec.data(), 1, pn, po, 1, sh, 1);
    f_cov[v] = Cnt::flops();
  }
  std::printf("{\"window_cov\": %ld, \"window_cov_vo\": %ld}\n", f_cov[0], f_cov[1]);
  return 0;
}
