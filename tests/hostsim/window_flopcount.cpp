// Exact operation tally of the smoothed-window getter (dekf_get_window, csrc/estimator_core.cuh), obtained by instantiating
// its stage bodies with a counting scalar, like flopcount.cpp does for the tick.  Dev tool: prints the constants
// tools/window_probe.py uses (tests/test_window_smoother.py keeps them in sync).  Not a product path.
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
  Vec9<CT> x;
  for (int f = 0; f < 6; ++f) P.pp.a[f] = P.vv.a[f] = P.bb.a[f] = CT(f == 0 || f == 3 || f == 5 ? 1e-3 : 1e-5);
  for (int f = 0; f < 9; ++f) P.pv.a[f] = P.pb.a[f] = P.vb.a[f] = CT(1e-6 * (f + 1));
  x.p = x.v = x.b = v3<CT>(CT(0.1), CT(0.2), CT(0.3));
  S3<CT> Lam;
  for (int f = 0; f < 6; ++f) Lam.a[f] = CT(f == 0 || f == 3 || f == 5 ? 200.0 : 3.0);
  V3<CT> eta = v3<CT>(CT(1.0), CT(2.0), CT(3.0));
  M3<CT> R = quat_to_rot<CT>(CT(0.9), CT(0.1), CT(0.2), CT(0.3));
  V3<CT> as = v3<CT>(CT(0.1), CT(0.0), CT(0.2)), dlt = v3<CT>(CT(0.002), CT(0.0), CT(0.0));
  using Mth = DefaultMath<CT>;
  // one backward stage without / with a VO row, and one stage of the FULL-mode forward sweep into the getter's scratch ring
  // (P_pp carried: meas<1> + prop<1>); the count does not depend on the values
  long f_back[2], f_fwd[2];
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
    double xn[9], xo[9];
    for (int f = 0; f < 9; ++f) xn[f] = 0.1 * f;
    Cnt::reset();
    window_back_stage<CT, CT>(mc, ck.data(), rec.data(), 1, xn, xo, 1);
    f_back[v] = Cnt::flops();
    Cov9<CT> Pw = P;
    Vec9<CT> xw = x;
    Cnt::reset();
    Mth::meas<1>(Pw, xw, Lam, eta);
    Mth::prop<1>(mc, Pw, xw, R, as, v == 1, dlt);
    f_fwd[v] = Cnt::flops();
  }
  std::printf("{\"window_back\": %ld, \"window_back_vo\": %ld, \"window_fwd\": %ld, \"window_fwd_vo\": %ld}\n", f_back[0], f_back[1],
              f_fwd[0], f_fwd[1]);
  return 0;
}
