// MinSR through the C++ host wrapper (include/peps_b200.hpp): Evaluate with collect_sr_buffers, then
// CalculateNaturalGradientMinSR on the device-resident samples.
// Reads: rows cols phys D walkers chi nsamples seed diag_shift, then the packed TPS and the initial configuration from stdin;
// prints |x|^2, the energy mean and the stored sample count.
#include <cstdio>
#include <iostream>
#include "../../include/peps_b200.hpp"

int main() {
  int rows, cols, phys, D, walkers, chi, nsamples;
  unsigned seed;
  double shift;
  std::cin >> rows >> cols >> phys >> D >> walkers >> chi >> nsamples >> seed >> shift;
  size_t n;
  std::cin >> n;
  std::vector<double> tps(n);
  for (auto &x : tps) std::cin >> x;
  peps_b200::MonteCarloParams mc;
  mc.num_samples = (size_t)nsamples; mc.sweeps_between_samples = 1;
  mc.initial_config.resize((size_t)rows * cols);
  for (auto &c : mc.initial_config) std::cin >> c;
  try {
    peps_b200::MCEnergyGradEvaluator ev(mc, peps_b200::BMPSTruncateParams::SVD(chi, chi, 0.0), rows, cols, phys, D, walkers,
                                        peps_b200::XXZModel{1.0, 1.0, 0.0}, seed);
    auto r = ev.Evaluate(tps, true);
    auto ng = ev.CalculateNaturalGradientMinSR(r, shift);
    double x2 = 0.0;
    for (double x : std::get<0>(ng)) x2 += x * x;
    std::printf("%.17g %.17g %zu\n", x2, std::get<1>(ng), ev.batch().SrCount());
  } catch (const std::exception &e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 1;
  }
  return 0;
}
