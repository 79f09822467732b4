// Register-radix (8/4/2) Stockham FFT rows for the K1 hot kernel (k_spectra).
//
// A row of N complex points is owned by T = N/8 threads (a "row slot"); several
// slots share one CTA and synchronise independently with named barriers, so a
// slot that waits on its global loads does not stall the others.  Each pass
// pulls R points per butterfly into registers, applies the twiddles, runs an
// in-register DFT_R and writes the autosort permutation back IN PLACE (all
// reads of a pass complete before its writes: one barrier in between), which
// keeps the footprint at one padded buffer per slot.
//
// The radix plan covers N/2; the last radix-2 pass of the N-point transform is
// fused into the real-FFT split (unpack), which saves one shared-memory round
// trip: Z[k] = a[k] + w^k b[k], Z[k+N/2] = a[k] - w^k b[k].
#pragma once
#include "fft.cuh"

namespace ppb {

// 16-byte elements, 8 per 128-byte bank row: XOR-swizzle the position inside a
// group of 8 with the group index, so that a stride-8 (radix-8 output) pattern
// hits 8 different bank groups while contiguous runs stay inside whole rows
// (no padding gaps: a warp reading 32 consecutive elements costs 4 wavefronts).
__device__ __forceinline__ int phys(int i) { return i ^ ((i >> 3) & 7); }
template <int N> struct Padded { static constexpr int value = N; };

__device__ __forceinline__ void bar_slot(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- 1-D bulk async copy (TMA) + mbarrier helpers ---------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy of `bytes` (multiple of 16, both 16-byte aligned),
// completion is signalled on `bar` as transaction bytes.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <typename F> __device__ __forceinline__ void dft4(cx<F>& v0, cx<F>& v1, cx<F>& v2, cx<F>& v3) {
  const cx<F> a0 = cadd(v0, v2), a1 = csub(v0, v2), a2 = cadd(v1, v3), a3 = csub(v1, v3);
  const cx<F> b3 = mk<F>(a3.y, -a3.x);  // -i a3
  v0 = cadd(a0, a2); v1 = cadd(a1, b3); v2 = csub(a0, a2); v3 = csub(a1, b3);
}

// in-register forward DFT of R points, natural-order output
template <int R, typename F> __device__ __forceinline__ void dftR(cx<F> (&v)[R]) {
  if constexpr (R == 2) {
    const cx<F> t = v[0];
    v[0] = cadd(t, v[1]); v[1] = csub(t, v[1]);
  } else if constexpr (R == 4) {
    dft4(v[0], v[1], v[2], v[3]);
  } else {
    static_assert(R == 8, "radix");
    dft4(v[0], v[2], v[4], v[6]);   // E_q -> v[2q]
    dft4(v[1], v[3], v[5], v[7]);   // O_q -> v[2q+1]
    const F h = F(0.70710678118654752440);
    const cx<F> o0 = v[1];
    const cx<F> o1 = mk<F>(h * (v[3].x + v[3].y), h * (v[3].y - v[3].x));    // * W8
    const cx<F> o2 = mk<F>(v[5].y, -v[5].x);                                  // * W8^2 = -i
    const cx<F> o3 = mk<F>(h * (v[7].y - v[7].x), -h * (v[7].x + v[7].y));   // * W8^3
    const cx<F> e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6];
    v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
    v[1] = cadd(e1, o1); v[5] = csub(e1, o1);
    v[2] = cadd(e2, o2); v[6] = csub(e2, o2);
    v[3] = cadd(e3, o3); v[7] = csub(e3, o3);
  }
}

// Radix plan for the first N/2 of the transform (the trailing radix-2 is fused
// into the split).  kPlan[i] = radix of pass i, 0-terminated.
template <int N> struct Plan8 {
  // packed radices, 4 bits each, pass 0 in the low nibble
  static constexpr unsigned code = N == 32 ? 0x44u : N == 64 ? 0x48u : N == 128 ? 0x88u : N == 256 ? 0x448u
                                 : N == 512 ? 0x488u : N == 1024 ? 0x888u : 0x4488u;
  static constexpr int n = N <= 128 ? 2 : (N <= 1024 ? 3 : 4);
  __host__ __device__ static constexpr int radix(int i) { return (int)((code >> (4 * i)) & 0xFu); }
};

template <int N> struct Slot8 {
  static constexpr int kT = N / 8;                     // threads per row slot
  static constexpr int kCtaThreads = 128;              // CTA size asked for; a row of more threads takes a CTA alone
  static constexpr int kSlots = (kCtaThreads / kT) > 0 ? (kCtaThreads / kT) : 1;  // row slots per CTA
  static constexpr int kThreads = kSlots * kT;         // CTA size
  static constexpr int kQuads = (N / 4) / kT;          // = 2 split quads (4 harmonics each) per thread
  static constexpr int kBufElems = Padded<N>::value;   // padded complex elements per slot
  static_assert(kT >= 4 && kT <= 256, "slot size");
};

template <int N> __device__ __forceinline__ void slot_sync(int slot) {
  if constexpr (Slot8<N>::kT >= 32) bar_slot(1 + slot, Slot8<N>::kT);
  else __syncwarp();
}

// Twiddle tables: per pass one base factor w1[k] = e^{-2 pi i k/(Ns R)}, k < Ns
// (its powers w^2..w^{R-1} are formed in registers: shared-memory bandwidth, not
// the FP64 pipe, bounds this kernel), then the N/2+1 split factors
// e^{-2 pi i p/(2N)}; the factors of the fused last radix-2 pass are their
// squares.
template <int N> struct TwLayout {
  using P = Plan8<N>;
  __host__ __device__ static constexpr int ns(int i) { int v = 1; for (int q = 0; q < i; ++q) v *= P::radix(q); return v; }
  __host__ __device__ static constexpr int off(int i) { int o = 0; for (int q = 1; q < i; ++q) o += ns(q); return o; }
  static constexpr int kPassTotal = off(P::n);
  static constexpr int kSplitOff = kPassTotal;              // e^{-2 pi i p/(2N)}, p <= N/2
  static constexpr int kTotal = kSplitOff + N / 2 + 1;
};

template <typename F> __device__ __forceinline__ cx<F> csqr(cx<F> a) {
  return mk<F>(fma(a.x, a.x, -a.y * a.y), F(2) * a.x * a.y);
}

// The staged raw row of a channel as N packed complex samples (x[2j], x[2j+1]):
// float32 as stored, or 16-bit integers with the PSRFITS scale and offset of the row
// (value = raw * DAT_SCL + DAT_OFFS, formed in float32 with the two roundings PSRCHIVE
// makes when it decodes the DATA column, so that both sources give identical samples).
struct RowSrcF32 {
  const float2* g;
  __device__ __forceinline__ bool has() const { return g != nullptr; }
  __device__ __forceinline__ float2 operator()(int j) const { return g[j]; }
};
struct RowSrcI16 {
  const short2* g;
  float scl, offs;
  __device__ __forceinline__ bool has() const { return g != nullptr; }
  __device__ __forceinline__ float2 operator()(int j) const {
    const short2 v = g[j];
    return make_float2(__fadd_rn(__fmul_rn((float)v.x, scl), offs), __fadd_rn(__fmul_rn((float)v.y, scl), offs));
  }
};

// One in-place pass of radix R.  First pass: inputs come from `g` (the staged
// packed real row, shared memory) and carry no twiddles.
template <int N, int R, typename F, typename Hook, typename Src>
__device__ __forceinline__ void pass8(cx<F>* __restrict__ buf, const cx<F>* __restrict__ twp, int t, int slot, int Ns,
                                      const Src g, bool gvalid, Hook hook) {
  constexpr int T = Slot8<N>::kT;
  constexpr int NB = N / R;       // butterflies per pass
  constexpr int PER = NB / T;     // butterflies per thread (R=8:1, 4:2, 2:4)
  static_assert(PER >= 1, "plan");
  cx<F> v[PER][R];
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int j = t + i * T;
    if (g.has()) {
      if (gvalid) {      // uniform over the row
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float2 x = g(j + r * NB);
          v[i][r] = mk<F>((F)x.x, (F)x.y);
        }
      } else {
#pragma unroll
        for (int r = 0; r < R; ++r) v[i][r] = mk<F>(F(0), F(0));
      }
    } else {
      const int k = j & (Ns - 1);
      cx<F> w[R];
      w[1] = twp[k];
      if constexpr (R >= 4) { w[2] = csqr(w[1]); w[3] = cmul(w[2], w[1]); }
      if constexpr (R >= 8) { w[4] = csqr(w[2]); w[5] = cmul(w[4], w[1]); w[6] = csqr(w[3]); w[7] = cmul(w[4], w[3]); }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        cx<F> x = buf[phys(j + r * NB)];
        if (r > 0) x = cmul(x, w[r]);
        v[i][r] = x;
      }
    }
  }
  slot_sync<N>(slot);   // every read of this pass (and of the previous row's split) is done
  hook();               // issue independent global loads here: they overlap the butterflies
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int j = t + i * T;
    const int k = j & (Ns - 1);
    dftR<R, F>(v[i]);
    const int j0 = (j - k) * R + k;
#pragma unroll
    for (int r = 0; r < R; ++r) buf[phys(j0 + r * Ns)] = v[i][r];
  }
  slot_sync<N>(slot);
}

// All passes of Plan8<N>: afterwards buf holds the input of the fused last
// radix-2 pass (a = buf[0:N/2], b = buf[N/2:N], both through phys()).
// `after_first_reads` runs right after the first pass has pulled the staged row
// into registers (the staging buffer may then be refilled); `in_last_pass` runs
// inside the last pass, after its reads and before its butterflies.
template <int N, typename F, typename Src, typename Fn, typename Fn2>
__device__ __forceinline__ void fft8_rows(cx<F>* __restrict__ buf, const cx<F>* __restrict__ tw, int t, int slot,
                                          const Src g, bool gvalid, Fn after_first_reads,
                                          Fn2 in_last_pass) {
  using P = Plan8<N>;
  using L = TwLayout<N>;
  auto nop = []() {};
  const RowSrcF32 none{nullptr};
  pass8<N, P::radix(0), F>(buf, tw, t, slot, 1, g, gvalid, nop);
  after_first_reads();
  if constexpr (P::n == 2) {
    constexpr int o = L::off(1), ns = L::ns(1);
    pass8<N, P::radix(1), F>(buf, tw + o, t, slot, ns, none, false, in_last_pass);
  } else {
    constexpr int o = L::off(1), ns = L::ns(1);
    pass8<N, P::radix(1), F>(buf, tw + o, t, slot, ns, none, false, nop);
  }
  if constexpr (P::n == 3) {
    constexpr int o = L::off(2), ns = L::ns(2);
    pass8<N, P::radix(2), F>(buf, tw + o, t, slot, ns, none, false, in_last_pass);
  } else if constexpr (P::n > 3) {
    constexpr int o = L::off(2), ns = L::ns(2);
    pass8<N, P::radix(2), F>(buf, tw + o, t, slot, ns, none, false, nop);
  }
  if constexpr (P::n == 4) {
    constexpr int o = L::off(3), ns = L::ns(3);
    pass8<N, P::radix(3), F>(buf, tw + o, t, slot, ns, none, false, in_last_pass);
  }
}

// Real-FFT split of one conjugate pair: from Z[k], Z[N-k] of the packed complex
// transform to the real-series harmonics d[k] and d[N-k].  wh = 0.5 e^{-2 pi i k/(2N)}:
// with the halved factor the 1/2 of E = (Z[k] + conj Z[N-k])/2 rides on the final
// FMAs (12 instead of 16 operations, same roundings as the textbook form).
template <typename F>
__device__ __forceinline__ void real_pair_h(cx<F> zp, cx<F> zq, cx<F> wh, cx<F>& dp, cx<F>& dq) {
  const cx<F> E2 = mk<F>(zp.x + zq.x, zp.y - zq.y);      // 2 E   = Z[k] + conj(Z[N-k])
  const cx<F> O2 = mk<F>(zp.y + zq.y, zq.x - zp.x);      // 2 O   = -i (Z[k] - conj(Z[N-k]))
  const cx<F> tt = cmul(wh, O2);                          // w O
  dp = mk<F>(fma(F(0.5), E2.x, tt.x), fma(F(0.5), E2.y, tt.y));
  dq = mk<F>(fma(F(0.5), E2.x, -tt.x), fma(F(-0.5), E2.y, tt.y));
}
template <typename F> __device__ __forceinline__ cx<F> chalf(cx<F> a) { return mk<F>(F(0.5) * a.x, F(0.5) * a.y); }

// Fused last radix-2 pass + real-FFT split, four harmonics per call so that every
// element of the buffer is read exactly once per row.  With H = N/2, a = buf[0:H],
// b = buf[H:N] and 1 <= p < N/4 the inputs a[p], b[p], a[H-p], b[H-p] give
// Z[p], Z[p+H], Z[H-p], Z[N-p], i.e. the two conjugate pairs (p, N-p) and
// (H-p, H+p):  d[0..3] = harmonics p, N-p, H-p, H+p.
template <int N, typename F>
__device__ __forceinline__ void split_quad8(const cx<F>* __restrict__ buf, const cx<F>* __restrict__ tw, int p,
                                            cx<F> (&d)[4]) {
  constexpr int H = N / 2;
  const cx<F> w2 = tw[TwLayout<N>::kSplitOff + p];    // e^{-2 pi i p/(2N)}
  const cx<F> A1 = buf[phys(p)], B1 = buf[phys(p + H)], A2 = buf[phys(H - p)], B2 = buf[phys(N - p)];
  const cx<F> wn = csqr(w2);                          // e^{-2 pi i p/N}; e^{-2 pi i (H-p)/N} = -conj(wn)
  const cx<F> wb1 = cmul(wn, B1), wb2 = cmul(cconj(wn), B2);
  const cx<F> Zp = cadd(A1, wb1), ZpH = csub(A1, wb1);   // Z[p], Z[p+H]
  const cx<F> Zq = csub(A2, wb2), ZqH = cadd(A2, wb2);   // Z[H-p], Z[N-p]
  const cx<F> wh = chalf(w2);
  real_pair_h(Zp, ZqH, wh, d[0], d[1]);
  real_pair_h(Zq, ZpH, mk<F>(-wh.y, -wh.x), d[2], d[3]);   // e^{-2 pi i (H-p)/(2N)} = -i conj(w2)
}

// The p = 0 quad: a[0], b[0] give Z[0] (DC and Nyquist of the real series) and the
// self-paired Z[H]; a[N/4], b[N/4] give the pair (N/4, 3N/4).  The outputs are ordered
// so that they resemble the general quad (slot p = 0 first, a top-quarter harmonic
// second): d[0..3] = harmonics N (Nyquist, real; stored in slot 0), 3N/4, H, N/4.
// Returns the DC term.
template <int N, typename F>
__device__ __forceinline__ F split_quad0(const cx<F>* __restrict__ buf, const cx<F>* __restrict__ tw, cx<F> (&d)[4]) {
  constexpr int H = N / 2, Q = N / 4;
  const cx<F> A1 = buf[phys(0)], B1 = buf[phys(H)], A2 = buf[phys(Q)], B2 = buf[phys(H + Q)];
  const cx<F> z0 = cadd(A1, B1), zh = csub(A1, B1);
  cx<F> unused;
  real_pair_h(zh, zh, chalf(tw[TwLayout<N>::kSplitOff + H]), d[2], unused);
  d[0] = mk<F>(z0.x - z0.y, F(0));
  const cx<F> wb = mk<F>(B2.y, -B2.x);                // e^{-2 pi i Q/N} = -i
  real_pair_h(cadd(A2, wb), csub(A2, wb), chalf(tw[TwLayout<N>::kSplitOff + Q]), d[3], d[1]);
  return z0.x + z0.y;
}

}  // namespace ppb
