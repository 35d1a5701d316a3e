// CPU check of csrc/phase_round.cuh: phase_fixed_rn(d) and both lanes of the two-wide phase_fixed_rn2 against
// round-to-nearest-even of d * 2^22 for EVERY float d with |d| < 512, i.e. every input whose rounded fixed-point value
// fits an int32 (what __float2int_rn returns there).  Prints the number of inputs with any mismatch and the number of
// inputs checked.  Built and run by tests/test_phase_round.py.
#include <cmath>
#include <cstdio>
#include "../../adaptive_optics_gym_b200/csrc/phase_round.cuh"
int main() {
  const uint32_t lim = 0x44000000u;                  // bits of 512.0f: every non-negative float below it
  unsigned long long bad = 0, n = 0;
  for (uint32_t sign = 0; sign < 2; ++sign) {
#pragma omp parallel for reduction(+ : bad, n) schedule(static)
    for (int64_t b = 0; b < (int64_t)lim; ++b) {
      const uint32_t bits = (uint32_t)b | (sign << 31);
      float d;
      std::memcpy(&d, &bits, sizeof d);
      const double ref = std::nearbyint((double)d * 4194304.0);   // exact product, ties to even
      // the two-wide form with d in one lane and -d in the other: over both signs, every input in both lanes
      int32_t p0, p1;
      phase_fixed_rn2(d, -d, &p0, &p1);
      bad += (double)phase_fixed_rn(d) != ref || (double)p0 != ref || (double)p1 != -ref;
      ++n;
    }
  }
  std::printf("%llu %llu\n", bad, n);
  return bad ? 1 : 0;
}
