// Host-side twiddle tables of the k_spectra row-transform plans (spectra_plan.cuh).
#pragma once
#include <math.h>

#include <vector>

#include "spectra_plan.cuh"

namespace ppb {

inline double2 unit_root(long num, long den) {   // e^{-2 pi i num/den} with exact quadrant values
  num %= den;
  if (num == 0) return make_double2(1.0, 0.0);
  if (4 * num == den) return make_double2(0.0, -1.0);
  if (2 * num == den) return make_double2(-1.0, 0.0);
  if (4 * num == 3 * den) return make_double2(0.0, 1.0);
  const double a = -2.0 * M_PI * (double)num / (double)den;
  return make_double2(cos(a), sin(a));
}

template <class PL> struct TwBuilder;
template <> struct TwBuilder<SpecPlan16> {
  static void build(std::vector<double2>& out) {
    using PL = SpecPlan16;
    out.assign(PL::kTwTotal, make_double2(0.0, 0.0));
    for (int k = 0; k < 16; ++k) out[k] = unit_root(k, 256);
    for (int p2 = 0; p2 <= 128; ++p2) out[PL::kSplitOff + p2] = unit_root(p2, 2048);
  }
};
// per-pass twiddle tables in the layout of TwLayout<N> (fft8.cuh)
template <int N> struct TwBuilder<SpecPlan8<N>> {
  static void build(std::vector<double2>& out) {
    using P = Plan8<N>;
    using L = TwLayout<N>;
    out.assign(L::kTotal, make_double2(0.0, 0.0));
    for (int i = 1; i < P::n; ++i) {
      const int Ns = L::ns(i), R = P::radix(i);
      for (int k = 0; k < Ns; ++k) out[L::off(i) + k] = unit_root((long)k, (long)Ns * R);
    }
    for (int p2 = 0; p2 <= N / 2; ++p2) out[L::kSplitOff + p2] = unit_root(p2, 2L * N);
  }
};

template <int N, class PL = SpecPlan<N>> constexpr size_t spectra_smem_bytes_of() {
  return (size_t)(((PL::kTwTotal + 1) & ~1) + PL::kSlots * N) * sizeof(cx<double>) +
         (size_t)PL::kSlots * PL::kStages * (2 * N) * sizeof(float);
}

}  // namespace ppb
