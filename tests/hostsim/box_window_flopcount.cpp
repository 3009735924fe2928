// Exact operation tally of the covariance pass of the constrained-window getter (dekf_get_constrained_window; bw_cov_stage,
// bw_vs_row and bw_dot9 in csrc/box_window.cuh), obtained by instantiating them with a counting scalar (add + mul + div; the
// device's fused multiply-add counts 2).  Dev tool: tests/test_constrained_window.py checks the constants of
// tools/window_probe.py against it.  Not a product path.
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
};
inline CT operator+(CT a, CT b) { Cnt::add++; return CT(a.v + b.v); }
inline CT operator-(CT a, CT b) { Cnt::add++; return CT(a.v - b.v); }
inline CT operator*(CT a, CT b) { Cnt::mul++; return CT(a.v * b.v); }
inline CT operator/(CT a, CT b) { Cnt::div++; return CT(a.v / b.v); }
inline CT operator-(CT a) { return CT(-a.v); }
inline CT &operator+=(CT &a, CT b) { Cnt::add++; a.v += b.v; return a; }
inline CT &operator-=(CT &a, CT b) { Cnt::add++; a.v -= b.v; return a; }

#include "../../decentralized_ekf_mhe_b200/csrc/host_setup.hpp"
#include "../../decentralized_ekf_mhe_b200/csrc/box_window.cuh"
using namespace dekf;

int main() {
  std::vector<CT> rec(BW_REC), Sn(81), Sk(81), t(9);
  std::vector<double> V(81);
  for (int e = 0; e < BW_REC; ++e) rec[e] = CT(1.0 + 1e-3 * e);
  for (int e = 0; e < 81; ++e) {
    Sn[e] = CT(e / 9 == e % 9 ? 1.0 : 0.0);
    V[e] = e / 9 == e % 9 ? 1.0 : 0.01;
  }
  Cnt::reset();
  bw_cov_stage<CT>(rec.data(), Sn.data(), Sk.data());
  const long cov = Cnt::flops();
  Cnt::reset();
  bw_cov_stage<CT>(rec.data(), nullptr, Sk.data());
  const long covT = Cnt::flops();
  Cnt::reset();
  for (int r = 0; r < 9; ++r) {  // P = V S V' from the lower triangle, as the getter forms it on rows handles
    bw_vs_row<CT>(V.data(), Sk.data(), 9, 0, r, t.data());
    for (int c = 0; c <= r; ++c) bw_dot9<CT>(t.data(), V.data() + c * 9);
  }
  const long vsvt = Cnt::flops();
  std::printf("{\"cov\": %ld, \"cov_T\": %ld, \"rows_vsvt\": %ld}\n", cov, covT, vsvt);
  return 0;
}
