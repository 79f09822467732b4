// PCA / B-spline model building (pplib.make_spline_model, after ppspline.py make_spline_model): the weighted
// moments of a portrait, back-projection of Gram eigenvectors, projections onto a basis, and the per-row low-pass
// of the mean profile and eigenvectors.  FP64 throughout; no floating-point atomics and a fixed summation order in
// every kernel, so that a call's outputs are bit-identical run to run.
//
// Rows d_n = sqrt(w_n) (x_n - mu) of a float64 portrait X [nchan, nbin] with channel weights w >= 0:
//   mu = sum_n w_n x_n / W,  W = sum_n w_n            (k_pca_mean)
//   C = D^T D / W  [nbin, nbin]  or  G = D D^T / W  [nchan, nchan]       (k_pca_tile, symmetric)
//   e_j = D^T u_j / ||D^T u_j||  [nbin]                (k_pca_tile, then k_pca_unit)
//   P = (X - mu~) E  [nchan, m]                        (k_pca_tile)
// The eigen decomposition between them runs on the host (pplib.make_spline_model).
#pragma once
#include "kernels.cuh"

namespace ppb {

// mu[b] and W over the channels in order (skipped when mu is null); rw[n] = sqrt(w_n).  One thread per bin (and per
// channel for rw).
__global__ void __launch_bounds__(256) k_pca_mean(const double* __restrict__ x, const double* __restrict__ w, double* mu,
                                                   double* rw, double* wsum, int nchan, int nbin) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (mu && i < nbin) {
    double s = 0.0, sw = 0.0;
    for (int n = 0; n < nchan; ++n) {
      const double wn = w[n];
      sw += wn;
      s = fma(wn, x[(size_t)n * nbin + i], s);
    }
    mu[i] = s / sw;
    if (i == 0) wsum[0] = sw;
  }
  if (i < nchan) rw[i] = sqrt(w[i]);
}

// Element (r, c) of a row-major matrix p [*, ld], centred by mean[c] and scaled by rw[r] when those are given.
struct PcaOp {
  const double* p;
  const double* mean;
  const double* rw;
  int ld;
  int trans;   // A: a(i, k) = trans ? at(k, i) : at(i, k);  B: b(k, j) = trans ? at(j, k) : at(k, j)
  __device__ __forceinline__ double at(int r, int c) const {
    double v = p[(size_t)r * ld + c];
    if (mean) v -= mean[c];
    if (rw) v *= rw[r];
    return v;
  }
};

struct PcaTileArgs {
  PcaOp a, b;
  double* out;         // [I, J] row-major: sum_k a(i, k) b(k, j) / div
  const double* div;   // device scalar or null (1)
  int I, J, K;
  int sym;             // a(i, k) = b(k, i): only tiles on or above the diagonal run; those above it write the mirror
};

constexpr int kPcaTile = 64, kPcaK = 16;

// One 64 x 64 output tile per CTA, 256 threads of 4 x 4 outputs, operands staged 16 k at a time in shared memory.
// Every output adds its K products in order k = 0 .. K - 1 with one fma each, so a symmetric product is symmetric
// bit for bit (fma(a, b, c) = fma(b, a, c)) and the result does not depend on the grid.
__global__ void __launch_bounds__(256) k_pca_tile(PcaTileArgs t) {
  __shared__ double As[kPcaK][kPcaTile + 1];
  __shared__ double Bs[kPcaK][kPcaTile + 1];
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (t.sym && bj < bi) return;
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  const int i0 = bi * kPcaTile, j0 = bj * kPcaTile;
  double acc[4][4];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) acc[u][v] = 0.0;
  for (int k0 = 0; k0 < t.K; k0 += kPcaK) {
    for (int e = tid; e < kPcaTile * kPcaK; e += 256) {
      // consecutive threads walk the operand's stored rows
      int ii, kk;
      if (t.a.trans) { ii = e % kPcaTile; kk = e / kPcaTile; } else { kk = e % kPcaK; ii = e / kPcaK; }
      const int i = i0 + ii, k = k0 + kk;
      As[kk][ii] = (i < t.I && k < t.K) ? (t.a.trans ? t.a.at(k, i) : t.a.at(i, k)) : 0.0;
      int jj;
      if (t.b.trans) { kk = e % kPcaK; jj = e / kPcaK; } else { jj = e % kPcaTile; kk = e / kPcaTile; }
      const int j = j0 + jj, k2 = k0 + kk;
      Bs[kk][jj] = (j < t.J && k2 < t.K) ? (t.b.trans ? t.b.at(j, k2) : t.b.at(k2, j)) : 0.0;
    }
    __syncthreads();
    const int kn = min(kPcaK, t.K - k0);
    for (int kk = 0; kk < kn; ++kk) {
      double av[4], bv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { av[u] = As[kk][ty + 16 * u]; bv[u] = Bs[kk][tx + 16 * u]; }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fma(av[u], bv[v], acc[u][v]);
    }
    __syncthreads();
  }
  const double dv = t.div ? *t.div : 1.0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + ty + 16 * u;
    if (i >= t.I) continue;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int j = j0 + tx + 16 * v;
      if (j >= t.J) continue;
      const double r = acc[u][v] / dv;
      t.out[(size_t)i * t.J + j] = r;
      if (t.sym && bj > bi) t.out[(size_t)j * t.J + i] = r;
    }
  }
}

// Column j of E [nbin, m] to unit norm, with the sign that makes its entry of largest |value| (the first such) positive.
// One CTA per column.
__global__ void __launch_bounds__(256) k_pca_unit(double* E, int nbin, int m) {
  __shared__ double sh[8];
  __shared__ double shv[8];
  __shared__ int shi[8];
  __shared__ double scale;
  const int j = blockIdx.x, tid = threadIdx.x;
  double v[1] = {0.0};
  double best = -1.0;
  int bi = 0x7fffffff;
  for (int b = tid; b < nbin; b += 256) {
    const double e = E[(size_t)b * m + j];
    v[0] = fma(e, e, v[0]);
    if (fabs(e) > best) { best = fabs(e); bi = b; }
  }
  auto before = [](double av, int ai, double bv, int bidx) { return av > bv || (av == bv && ai < bidx); };
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (before(ov, oi, best, bi)) { best = ov; bi = oi; }
  }
  if ((tid & 31) == 0) { shv[tid >> 5] = best; shi[tid >> 5] = bi; }
  block_sum<1, 256>(v, sh);   // (synchronises: shv / shi are complete after it)
  if (tid == 0) {
    for (int w = 1; w < 8; ++w) if (before(shv[w], shi[w], best, bi)) { best = shv[w]; bi = shi[w]; }
    const double nrm = sqrt(v[0]);
    scale = (E[(size_t)bi * m + j] < 0.0 ? -1.0 : 1.0) / nrm;
  }
  __syncthreads();
  const double s = scale;
  for (int b = tid; b < nbin; b += 256) E[(size_t)b * m + j] *= s;
}

// ---- low-pass of rows: rfft, k_c = find_kc (get_noise_fit's cut-off, fact = 1), harmonics above k_c set to zero
// (the DC term kept; the Nyquist term kept only when k_c reaches it), irfft ------------------------------------------
struct LowpassArgs {
  const double* in;    // [nrows, nbin]
  double* out;         // [nrows, nbin]
  int* kc;             // [nrows]
  const void* twN;     // FP64 tables of the power-of-two row transform (fft.cuh)
  const void* tw2N;
};

template <int N> constexpr size_t lowpass_smem_bytes() {
  return (size_t)(N + N / 2 + 2 + 2 * N + N + 1) * sizeof(cx<double>) + (size_t)2 * (N + 1) * sizeof(double);
}

// Power-of-two nbin = 2N: one CTA per row, the whole transform pair in shared memory.
template <int N>
__global__ void __launch_bounds__(256) k_lowpass(LowpassArgs a) {
  using T = double;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufA = tw2N + (N / 2 + 2);
  cx<T>* bufB = bufA + N;
  cx<T>* d = bufB + N;                                // [N + 1] half-spectrum
  double* y = reinterpret_cast<double*>(d + N + 1);   // [N + 1] log10 pows
  double* ek = y + (N + 1);                           // [N + 1] find_kc scratch
  const int tid = threadIdx.x;
  const long row = blockIdx.x;
  {
    const cx<T>* g1 = reinterpret_cast<const cx<T>*>(a.twN);
    const cx<T>* g2 = reinterpret_cast<const cx<T>*>(a.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  const double2* src = reinterpret_cast<const double2*>(a.in + (size_t)row * 2 * N);
  for (int j = tid; j < N; j += 256) { const double2 v = src[j]; bufA[j] = mk<T>(v.x, v.y); }
  __syncthreads();
  const cx<T>* Z = fft_forward<N, 256, T>(bufA, bufB, twN, tid);
  for (int p = tid + 1; p <= N / 2; p += 256) {
    cx<T> dp, dq;
    unpack_pair<T>(Z, tw2N, N, p, dp, dq);
    d[p] = dp;
    if (p < N / 2) d[N - p] = dq;
  }
  if (tid == 0) { d[0] = mk<T>(Z[0].x + Z[0].y, 0.0); d[N] = mk<T>(Z[0].x - Z[0].y, 0.0); }
  __syncthreads();
  const double inv_n = 1.0 / (double)(2 * N);
  for (int k = tid; k <= N; k += 256) y[k] = log10((d[k].x * d[k].x + d[k].y * d[k].y) * inv_n);
  __syncthreads();
  const int kc = find_kc(y, ek, N + 1);   // (synchronises: Z is no longer read)
  const cx<T> zero = mk<T>(0.0, 0.0);
  for (int p = tid + 1; p <= N / 2; p += 256) {
    const cx<T> dp = p <= kc ? d[p] : zero;
    const cx<T> dq = p < N / 2 ? (N - p <= kc ? d[N - p] : zero) : dp;
    cx<T> zp, zq;
    pack_pair<T>(dp, dq, tw2N[p], zp, zq);
    bufA[p] = cconj(zp);   // conj for the inverse transform
    if (p < N / 2) bufA[N - p] = cconj(zq);
  }
  if (tid == 0) {
    const T d0 = d[0].x, dN = kc >= N ? d[N].x : 0.0;
    bufA[0] = mk<T>(T(0.5) * (d0 + dN), -T(0.5) * (d0 - dN));
    a.kc[row] = kc;
  }
  __syncthreads();
  const cx<T>* Y = fft_forward<N, 256, T>(bufA, bufB, twN, tid);
  const T sc = T(1) / T(N);
  double2* dst = reinterpret_cast<double2*>(a.out + (size_t)row * 2 * N);
  for (int j = tid; j < N; j += 256) dst[j] = make_double2(Y[j].x * sc, -Y[j].y * sc);
}

// Other even nbin: the cut-off and the zeroing on the k_fwd_any spectrum rows (slot k = harmonic k, 1..L; dc =
// harmonic 0), in place, before k_inv_any.  One CTA per row; y, ek: 2 (L + 1) doubles of dynamic shared memory.
__global__ void __launch_bounds__(256) k_lowpass_spec(cx<double>* spec, const double* __restrict__ dc, int* kc_out, int Npad,
                                                       int L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* y = reinterpret_cast<double*>(smem_raw);
  double* ek = y + (L + 1);
  const long row = blockIdx.x;
  const int tid = threadIdx.x;
  cx<double>* s = spec + (size_t)row * Npad;
  const double inv_n = 1.0 / (double)(2 * L);
  for (int k = tid; k <= L; k += 256) {
    double p;
    if (k == 0) p = dc[row] * dc[row];
    else p = s[k].x * s[k].x + s[k].y * s[k].y;
    y[k] = log10(p * inv_n);
  }
  __syncthreads();
  const int kc = find_kc(y, ek, L + 1);
  for (int k = tid + 1; k <= L; k += 256) {
    if (k > kc) s[k] = mk<double>(0.0, 0.0);
    else if (k == L) s[k].y = 0.0;   // irfft keeps the real part of the Nyquist term
  }
  if (tid == 0) kc_out[row] = kc;
}

}  // namespace ppb
