// Radix-16 register butterflies of k_spectra16 (spectra16.cuh), the N = 1024 row
// transform: 1024 = 16 * 16 * 4, two shared-memory passes of 64 threads (16 points
// per thread) and a last radix-4 pass fused into the real-FFT split.  Compared with
// the radix-8 plan (8 * 8 * 8 * 2) one full shared-memory round trip per row
// disappears; shared-memory bandwidth is what bounds the radix-8 passes.
#pragma once
#include "fft8.cuh"

namespace ppb {

// 16 B elements: the radix-16 passes read stride-64 / write stride-16 (pass 1) and
// stride-16 within 256 (pass 2); XOR the column with bits 4..6 of the position.
__device__ __forceinline__ int phys16(int i) { return i ^ ((i >> 4) & 7); }

// In-register forward DFT of 16 points.  Input natural order; output X[k] is left
// in v[(k >> 2) + 4 (k & 3)] (read it through dft16_at()).
// 4 x 4 decomposition.  The inner twiddles W16^(r q) are not applied as separate complex multiplications:
// W16^2 and W16^6 are h (1 -/+ i)-type factors, W16^1, W16^3, W16^9 are c1 (1 - i t), c1 (t - i), -c1 (1 - i t)
// with t = tan(pi/8); the unscaled rotations cost two operations each and the common factors h, c1 ride on the
// FMAs of the second stage's butterflies (constant multiplier: two register operands, full FP64 rate).
// 144 operations instead of 160.
template <typename F> __device__ __forceinline__ void dft16_group13(cx<F>& x0, cx<F>& v1, cx<F>& v2, cx<F>& v3, bool third) {
  const F h = F(0.70710678118654752440), c1 = F(0.92387953251128675613), t = F(0.41421356237309504880);
  cx<F> p2, q1, q3;
  if (!third) {   // W16^1, W16^2, W16^3
    p2 = mk<F>(v2.x + v2.y, v2.y - v2.x);
    q1 = mk<F>(fma(t, v1.y, v1.x), fma(-t, v1.x, v1.y));
    q3 = mk<F>(fma(t, v3.x, v3.y), fma(t, v3.y, -v3.x));
  } else {        // W16^3, W16^6, W16^9
    p2 = mk<F>(v2.y - v2.x, -(v2.x + v2.y));
    q1 = mk<F>(fma(t, v1.x, v1.y), fma(t, v1.y, -v1.x));
    q3 = mk<F>(-fma(t, v3.y, v3.x), fma(t, v3.x, -v3.y));
  }
  const cx<F> a0 = mk<F>(fma(h, p2.x, x0.x), fma(h, p2.y, x0.y)), a1 = mk<F>(fma(-h, p2.x, x0.x), fma(-h, p2.y, x0.y));
  const cx<F> b2 = cadd(q1, q3), b3 = csub(q1, q3);
  x0 = mk<F>(fma(c1, b2.x, a0.x), fma(c1, b2.y, a0.y));
  v2 = mk<F>(fma(-c1, b2.x, a0.x), fma(-c1, b2.y, a0.y));
  v1 = mk<F>(fma(c1, b3.y, a1.x), fma(-c1, b3.x, a1.y));
  v3 = mk<F>(fma(-c1, b3.y, a1.x), fma(c1, b3.x, a1.y));
}
template <typename F> __device__ __forceinline__ void dft16(cx<F> (&v)[16]) {
#pragma unroll
  for (int r = 0; r < 4; ++r) dft4(v[r], v[r + 4], v[r + 8], v[r + 12]);   // A_r[q] -> v[r + 4q]
  const F h = F(0.70710678118654752440);
  dft4(v[0], v[1], v[2], v[3]);                                            // q = 0: X[4s] -> v[s]
  dft16_group13(v[4], v[5], v[6], v[7], false);                            // q = 1: X[1 + 4s] -> v[4 + s]
  {                                                                        // q = 2: W16^2, W16^4 = -i, W16^6
    const cx<F> p1 = mk<F>(v[9].x + v[9].y, v[9].y - v[9].x), p3 = mk<F>(v[11].y - v[11].x, -(v[11].x + v[11].y));
    const cx<F> x2 = mk<F>(v[10].y, -v[10].x);
    const cx<F> a0 = cadd(v[8], x2), a1 = csub(v[8], x2), b2 = cadd(p1, p3), b3 = csub(p1, p3);
    v[8] = mk<F>(fma(h, b2.x, a0.x), fma(h, b2.y, a0.y));
    v[10] = mk<F>(fma(-h, b2.x, a0.x), fma(-h, b2.y, a0.y));
    v[9] = mk<F>(fma(h, b3.y, a1.x), fma(-h, b3.x, a1.y));
    v[11] = mk<F>(fma(-h, b3.y, a1.x), fma(h, b3.x, a1.y));
  }
  dft16_group13(v[12], v[13], v[14], v[15], true);                         // q = 3: X[3 + 4s] -> v[12 + s]
}
__host__ __device__ constexpr int dft16_at(int k) { return (k >> 2) + 4 * (k & 3); }

// v[r] *= w^r, r = 1..15
template <typename F> __device__ __forceinline__ void twiddle16(cx<F> (&v)[16], cx<F> w1) {
  const cx<F> w2 = csqr(w1), w3 = cmul(w2, w1), w4 = csqr(w2);
  v[1] = cmul(v[1], w1); v[2] = cmul(v[2], w2); v[3] = cmul(v[3], w3); v[4] = cmul(v[4], w4);
  v[5] = cmul(v[5], cmul(w4, w1)); v[6] = cmul(v[6], cmul(w4, w2)); v[7] = cmul(v[7], cmul(w4, w3));
  const cx<F> w8 = csqr(w4);
  v[8] = cmul(v[8], w8);
  v[9] = cmul(v[9], cmul(w8, w1)); v[10] = cmul(v[10], cmul(w8, w2)); v[11] = cmul(v[11], cmul(w8, w3));
  const cx<F> w12 = cmul(w8, w4);
  v[12] = cmul(v[12], w12);
  v[13] = cmul(v[13], cmul(w12, w1)); v[14] = cmul(v[14], cmul(w12, w2)); v[15] = cmul(v[15], cmul(w12, w3));
}

// Last radix-4 pass fused with the real-FFT split (N = 1024).  The butterflies p and
// 256 - p (1 <= p <= 127) give Z[p + 256 j] and Z[256 - p + 256 j], i.e. the four
// conjugate pairs (p + 256 j, N - p - 256 j): d[2j] = harmonic p + 256 j,
// d[2j + 1] = harmonic N - p - 256 j.  pa = &buf[phys16(p)], pb = &buf[phys16(256 - p)]
// (phys16 moves an element within its 16-element block, so the other three inputs of
// each butterfly sit 256, 512 and 768 elements further on); w2 = e^{-2 pi i p/2048}.
template <typename F>
__device__ __forceinline__ void split16_general(const cx<F>* __restrict__ pa, const cx<F>* __restrict__ pb, cx<F> w2, cx<F> (&d)[8]) {
  const F h = F(0.70710678118654752440);
  cx<F> a0 = pa[0], a1 = pa[256], a2 = pa[512], a3 = pa[768];
  cx<F> b0 = pb[0], b1 = pb[256], b2 = pb[512], b3 = pb[768];
  const cx<F> wn1 = csqr(w2), wn2 = csqr(wn1), wn3 = cmul(wn1, wn2);     // e^{-2 pi i c p/N}
  a1 = cmul(a1, wn1); a2 = cmul(a2, wn2); a3 = cmul(a3, wn3);
  dft4(a0, a1, a2, a3);                                                  // Z[p + 256 j]
  // e^{-2 pi i c (256 - p)/N} = (-i)^c conj(wn_c)
  b1 = cmul(b1, mk<F>(-wn1.y, -wn1.x)); b2 = cmul(b2, mk<F>(-wn2.x, wn2.y)); b3 = cmul(b3, mk<F>(wn3.y, wn3.x));
  dft4(b0, b1, b2, b3);                                                  // Z[256 - p + 256 j]
  // split factors e^{-2 pi i (p + 256 j)/2048} = w2 W8^j
  const F hh = F(0.5) * h;
  const cx<F> wh = chalf(w2);
  real_pair_h(a0, b3, wh, d[0], d[1]);
  real_pair_h(a1, b2, mk<F>(hh * (w2.x + w2.y), hh * (w2.y - w2.x)), d[2], d[3]);
  real_pair_h(a2, b1, mk<F>(wh.y, -wh.x), d[4], d[5]);
  real_pair_h(a3, b0, mk<F>(hh * (w2.y - w2.x), -hh * (w2.x + w2.y)), d[6], d[7]);
}

// The special unit: butterflies p = 0 and p = 128.  d[0] = Nyquist (real, slot 0),
// d[2], d[4], d[6] = harmonics 256, 512, 768; d[1], d[3], d[5], d[7] = 896, 640, 384, 128.
// Returns the DC term.
template <typename F>
__device__ __forceinline__ F split_oct0(const cx<F>* __restrict__ buf, const cx<F>* __restrict__ w2s, cx<F> (&d)[8]) {
  const F h = F(0.70710678118654752440);
  cx<F> a0 = buf[phys16(0)], a1 = buf[phys16(256)], a2 = buf[phys16(512)], a3 = buf[phys16(768)];
  cx<F> b0 = buf[phys16(128)], b1 = buf[phys16(384)], b2 = buf[phys16(640)], b3 = buf[phys16(896)];
  dft4(a0, a1, a2, a3);                                                  // Z[0], Z[256], Z[512], Z[768]
  b1 = mk<F>(h * (b1.x + b1.y), h * (b1.y - b1.x));                      // W8^1
  b2 = mk<F>(b2.y, -b2.x);                                               // W8^2
  b3 = mk<F>(h * (b3.y - b3.x), -h * (b3.x + b3.y));                     // W8^3
  dft4(b0, b1, b2, b3);                                                  // Z[128], Z[384], Z[640], Z[896]
  cx<F> unused;
  d[0] = mk<F>(a0.x - a0.y, F(0));
  const F hh = F(0.5) * h;
  real_pair_h(a1, a3, mk<F>(hh, -hh), d[2], d[6]);                       // e^{-2 pi i 256/2048} / 2
  real_pair_h(a2, a2, mk<F>(F(0), F(-0.5)), d[4], unused);
  const cx<F> w = w2s[128];                                              // e^{-2 pi i 128/2048}
  real_pair_h(b0, b3, chalf(w), d[7], d[1]);
  real_pair_h(b1, b2, mk<F>(hh * (w.x + w.y), hh * (w.y - w.x)), d[5], d[3]);
  return a0.x + a0.y;                                                    // DC of the real series
}

}  // namespace ppb
