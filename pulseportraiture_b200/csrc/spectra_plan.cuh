// Row plans of k_spectra.  A plan fixes how many threads own a row, how the N-point
// transform is split into register butterflies, and how the fused last pass + real-FFT
// split hands harmonics to threads ("units" of kOut outputs):
//
//   SpecPlan8<N>   N/8 threads per row, radix-8/4 passes + (radix-2 fused with the
//                  split), units = quads: slots p, N-p, N/2-p, N/2+p
//   SpecPlan16     N = 1024 only: 64 threads per row, units = octs: slots p+256j, N-p-256j.
//                  The layout of k_spectra16 (spectra16.cuh: two radix-16 passes + radix-4
//                  fused with the split) and of its twiddle table.  k_spectra runs it only on
//                  rows that arrive transformed (FROMSPEC, nbin 1026..2046): there it fixes
//                  which thread sums which harmonic powers, and SpecPlan8<1024> would sum the
//                  noise estimate in another order.
//
// In both, unit 0 of thread 0 is the special unit that holds the self-paired and
// the Nyquist harmonic; its outputs are ordered so that the per-output rules
// (slot formula, "is in the top quarter", "may carry a lo part") stay uniform.
#pragma once
#include "fft16.cuh"

namespace ppb {

template <int N> struct SpecPlan8 {
  using S8 = Slot8<N>;
  static constexpr int kT = S8::kT, kSlots = S8::kSlots, kThreads = S8::kThreads;
  static constexpr int kUnits = S8::kQuads, kOut = 4;
  static constexpr int kTwTotal = TwLayout<N>::kTotal;
  static constexpr int kMinBlocks = N >= 2048 ? 2 : 4;   // CTAs per SM, chosen by measurement (DESIGN.md §4)
  static constexpr int kStages = 2;
  __device__ static __forceinline__ void sync(int slot) { slot_sync<N>(slot); }
  template <typename F, typename Src, typename Fn, typename Fn2>
  __device__ static __forceinline__ void transform(cx<F>* buf, const cx<F>* tw, int t, int slot, const Src g, bool used,
                                                   Fn after_first_reads, Fn2 in_last_pass) {
    fft8_rows<N, F>(buf, tw, t, slot, g, used, after_first_reads, in_last_pass);
  }
  template <typename F>
  __device__ static __forceinline__ F split(const cx<F>* buf, const cx<F>* tw, int t, int i, bool first, cx<F> (&d)[kOut]) {
    if (i > 0 || !first) { split_quad8<N, F>(buf, tw, t + i * kT, d); return F(0); }
    return split_quad0<N, F>(buf, tw, d);     // the row's DC term
  }
  // slot (index into a row of X / conj(model); slot 0 = Nyquist) of output q of unit i
  __device__ static __forceinline__ int slot_of(int t, int i, int q, bool first) {
    const int p = t + i * kT;
    if (q == 0) return p;
    if (q == 2) return N / 2 - p;
    if (q == 1) return (i == 0 && first) ? 3 * (N / 4) : N - p;
    return (i == 0 && first) ? N / 4 : N / 2 + p;
  }
  // harmonic >= 3N/4 (the noise estimate of pplib.py:2243-2245 sums these)
  __device__ static __forceinline__ bool top(int i, int q, bool first) { return q == 1 || (q == 0 && i == 0 && first); }
};

struct SpecPlan16 {
  static constexpr int N = 1024;
  static constexpr int kT = 64, kSlots = 1, kThreads = 64;
  static constexpr int kUnits = 2, kOut = 8;
  static constexpr int kSplitOff = 16;                    // tw[0..15] = e^{-2 pi i k/256}; then e^{-2 pi i p/2048}, p <= 128
  static constexpr int kTwTotal = kSplitOff + 129;
  static constexpr int kMinBlocks = 6;                    // CTAs per SM (register budget 65536 / (64 kMinBlocks))
  static constexpr int kStages = 2;                       // staging space of two raw rows (k_spectra16: raw + model row)
  __device__ static __forceinline__ void sync(int) { __syncthreads(); }
  // q = 2j: slot p + 256 j; q = 2j + 1: slot N - p - 256 j; the special unit uses p = 0 for
  // the even and p = 128 for the odd outputs
  __device__ static __forceinline__ int slot_of(int t, int i, int q, bool first) {
    const int p = t + i * kT;
    if ((q & 1) == 0) return p + 256 * (q >> 1);
    return N - 256 * (q >> 1) - ((i == 0 && first) ? 128 : p);
  }
  __device__ static __forceinline__ bool top(int i, int q, bool first) { return q == 1 || q == 6 || (q == 0 && i == 0 && first); }
};

template <int N> struct SpecPlanSel { using type = SpecPlan8<N>; };
template <> struct SpecPlanSel<1024> { using type = SpecPlan16; };
template <int N> using SpecPlan = typename SpecPlanSel<N>::type;

}  // namespace ppb
