// Exact operation tally of the backward passes of the foot-state window getter (dekf_get_foot_window; fw_mean_stage and
// fw_cov_stage in csrc/footstate.cuh) for L = 1, 2, 4 legs, obtained by instantiating them with a counting scalar (add + mul
// + div + sqrt; the device's fused multiply-add counts 2).  Dev tool: tests/test_foot_window.py checks the closed forms of
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
inline CT &operator+=(CT &a, CT b) { Cnt::add++; a.v += b.v; return a; }
inline CT &operator-=(CT &a, CT b) { Cnt::add++; a.v -= b.v; return a; }

#include "../../decentralized_ekf_mhe_b200/csrc/host_setup.hpp"
using namespace dekf;

template <int L>
void tally(bool last) {
  constexpr int DS = FootWin<L>::DS, W = FootWin<L>::W;
  std::vector<CT> rec(W), xn(DS), x(DS), Pn(DS * DS), Pk(DS * DS);
  for (int w = 0; w < W; ++w) rec[w] = CT(1.0 + 1e-3 * w);
  for (int e = 0; e < DS * DS; ++e) Pn[e] = CT(e / DS == e % DS ? 1.0 : 0.0);
  Cnt::reset();
  fw_mean_stage<CT, L>(rec.data(), xn.data(), x.data());
  const long mean = Cnt::flops();
  Cnt::reset();
  fw_cov_stage<CT, L>(rec.data(), Pn.data(), Pk.data());
  const long cov = Cnt::flops();
  Cnt::reset();
  fw_cov_stage<CT, L>(rec.data(), nullptr, Pk.data());
  const long covT = Cnt::flops();
  std::printf("\"%d\": {\"mean\": %ld, \"cov\": %ld, \"cov_T\": %ld}%s", L, mean, cov, covT, last ? "" : ", ");
}

int main() {
  std::printf("{");
  tally<1>(false);
  tally<2>(false);
  tally<4>(true);
  std::printf("}\n");
  return 0;
}
