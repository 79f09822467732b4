// Arbitrary (even) nbin: the reference transforms rows of any length with numpy's rfft
// (pplib.py:2127-2130, pptoaslib.py:976-979).  The tuned kernels need nbin = 2^m; every other even nbin
// runs through the chirp-z (Bluestein) form of the same DFT on top of the power-of-two row FFT:
//   packed row z_j = x_2j + i x_2j+1, j < L = nbin/2;  Z_k = sum_j z_j e^{-2 pi i jk/L}
//   j k = (j^2 + k^2 - (k - j)^2)/2  ->  Z_k = c_k sum_j (z_j c_j) conj(c_{k-j}),  c_j = e^{-pi i j^2/L}
// i.e. one circular convolution of length M = 2^m >= 2L - 1: two M-point FFTs per row (the transform of the
// chirp filter is a table), then the usual real-FFT split with e^{-2 pi i k/nbin}.  Everything in FP64.
// The spectra land in rows of Npad = 2^m > L slots (slot k = harmonic k, 1 <= k <= L; slot 0 and the slots
// above L are zero), so the solver kernels (k_guess, k_pass2, k_pass5, k_update*, k_align_spec) run
// unchanged on Npad; only the normalisations that contain nbin take the true value (kc, ntop, nbin/2, dof).
// Lengths L = 2^a 3^b 5^c (nbin = 1000, 1200, 1536, 2000, 3000, ...) skip the convolution: one Stockham transform
// of length L with radix-2/3/4/5 passes (fft_mixed), a fifth of the work.
// Not tuned: one CTA of 256 threads per row and an FP64 spectrum scratch in HBM between the transform
// and the kernels that consume it.
#pragma once
#include "fft.cuh"

namespace ppb {

struct AnyPlan {
  const cx<double>* chirp;  // [L]       c_j = e^{-pi i j^2 / L}
  const cx<double>* Bspec;  // [M]       FFT_M of the wrapped chirp filter conj(c_|m|), divided by M
  const cx<double>* twM;    // [M]       e^{-2 pi i j / M}
  const cx<double>* tw2n;   // [L/2 + 1] e^{-2 pi i k / (2 L)}
  const cx<double>* twL;    // [L]       e^{-2 pi i j / L} (mixed-radix path)
  int L, Npad;
  int nrad;                 // > 0: L = product of rad[0..nrad) with radices 2, 3, 4, 5: direct Stockham transform of
  int rad[12];              //      length L instead of the Bluestein convolution
};

// ---- L = 2^a 3^b 5^c: Stockham autosort passes of mixed radix in shared memory ---------------------------------
template <int R> __device__ __forceinline__ void dft_small(cx<double> (&v)[R]) {
  if constexpr (R == 2) {
    const cx<double> t = v[0];
    v[0] = cadd(t, v[1]); v[1] = csub(t, v[1]);
  } else if constexpr (R == 3) {
    const double s = 0.86602540378443864676;
    const cx<double> t1 = cadd(v[1], v[2]), d = csub(v[1], v[2]);
    const cx<double> t2 = mk<double>(v[0].x - 0.5 * t1.x, v[0].y - 0.5 * t1.y);
    const cx<double> r = mk<double>(s * d.y, -s * d.x);                       // -i s d
    v[0] = cadd(v[0], t1); v[1] = cadd(t2, r); v[2] = csub(t2, r);
  } else if constexpr (R == 4) {
    const cx<double> a0 = cadd(v[0], v[2]), a1 = csub(v[0], v[2]);
    const cx<double> a2 = cadd(v[1], v[3]), a3 = csub(v[1], v[3]);
    const cx<double> b3 = mk<double>(a3.y, -a3.x);                            // -i a3
    v[0] = cadd(a0, a2); v[1] = cadd(a1, b3); v[2] = csub(a0, a2); v[3] = csub(a1, b3);
  } else {
    static_assert(R == 5, "radix");
    const double c1 = 0.30901699437494742410, c2 = -0.80901699437494742410;   // cos(2 pi/5), cos(4 pi/5)
    const double s1 = 0.95105651629515357212, s2 = 0.58778525229247312917;    // sin(2 pi/5), sin(4 pi/5)
    const cx<double> a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]), b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
    const cx<double> m1 = mk<double>(v[0].x + c1 * a1.x + c2 * a2.x, v[0].y + c1 * a1.y + c2 * a2.y);
    const cx<double> m2 = mk<double>(v[0].x + c2 * a1.x + c1 * a2.x, v[0].y + c2 * a1.y + c1 * a2.y);
    const cx<double> n1 = mk<double>(s1 * b1.x + s2 * b2.x, s1 * b1.y + s2 * b2.y);
    const cx<double> n2 = mk<double>(s2 * b1.x - s1 * b2.x, s2 * b1.y - s1 * b2.y);
    v[0] = mk<double>(v[0].x + a1.x + a2.x, v[0].y + a1.y + a2.y);
    v[1] = mk<double>(m1.x + n1.y, m1.y - n1.x);                              // m1 - i n1
    v[4] = mk<double>(m1.x - n1.y, m1.y + n1.x);
    v[2] = mk<double>(m2.x + n2.y, m2.y - n2.x);
    v[3] = mk<double>(m2.x - n2.y, m2.y + n2.x);
  }
}

template <int R, int NT>
__device__ __forceinline__ void pass_mixed(const cx<double>* __restrict__ src, cx<double>* __restrict__ dst,
                                           const cx<double>* __restrict__ twL, int L, int Ns, int tid) {
  const int Q = L / R;             // butterflies of this pass
  const int tstep = Q / Ns;        // index step of e^{-2 pi i k/(Ns R)} in twL
  for (int j = tid; j < Q; j += NT) {
    const int k = j % Ns;
    cx<double> v[R];
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = src[j + r * Q];
    if (Ns > 1) {
#pragma unroll
      for (int r = 1; r < R; ++r) v[r] = cmul(v[r], twL[k * tstep * r]);
    }
    dft_small<R>(v);
    const int j0 = (j - k) * R + k;
#pragma unroll
    for (int r = 0; r < R; ++r) dst[j0 + r * Ns] = v[r];
  }
}

// Forward DFT of length L = prod rad[] of bufA[0..L); returns the buffer that holds the result.
template <int NT>
__device__ __forceinline__ cx<double>* fft_mixed(cx<double>* bufA, cx<double>* bufB, const AnyPlan& p, int tid) {
  cx<double>* src = bufA;
  cx<double>* dst = bufB;
  int Ns = 1;
  for (int q = 0; q < p.nrad; ++q) {
    const int R = p.rad[q];
    if (R == 4) pass_mixed<4, NT>(src, dst, p.twL, p.L, Ns, tid);
    else if (R == 5) pass_mixed<5, NT>(src, dst, p.twL, p.L, Ns, tid);
    else if (R == 3) pass_mixed<3, NT>(src, dst, p.twL, p.L, Ns, tid);
    else pass_mixed<2, NT>(src, dst, p.twL, p.L, Ns, tid);
    __syncthreads();
    cx<double>* t = src; src = dst; dst = t;
    Ns *= R;
  }
  return src;
}

// Forward DFT of length L of bufA[0..L) by Bluestein.  All NT threads of the CTA call; returns the buffer
// (bufA or bufB) that holds Z[0..L).
template <int M, int NT>
__device__ __forceinline__ cx<double>* bluestein(cx<double>* bufA, cx<double>* bufB, const AnyPlan& p, int tid) {
  if (p.nrad > 0) return fft_mixed<NT>(bufA, bufB, p, tid);   // (uniform over the grid)
  for (int j = tid; j < M; j += NT) bufA[j] = j < p.L ? cmul(bufA[j], p.chirp[j]) : mk<double>(0.0, 0.0);
  __syncthreads();
  cx<double>* A = fft_forward<M, NT, double>(bufA, bufB, p.twM, tid);
  cx<double>* other = (A == bufA) ? bufB : bufA;
  for (int j = tid; j < M; j += NT) {          // times the filter; conjugate: the next forward FFT is the inverse
    const cx<double> v = cmul(A[j], p.Bspec[j]);
    A[j] = mk<double>(v.x, -v.y);
  }
  __syncthreads();
  cx<double>* C = fft_forward<M, NT, double>(A, other, p.twM, tid);
  for (int k = tid; k < p.L; k += NT) {
    const cx<double> c = C[k];
    C[k] = cmul(p.chirp[k], mk<double>(c.x, -c.y));
  }
  __syncthreads();
  return C;
}

// complex FFT of one row of length M in place (table set-up: the chirp filter's transform)
template <int M>
__global__ void __launch_bounds__(256) k_cfft_row(cx<double>* row, const cx<double>* twM, double scale) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<double>* bufA = reinterpret_cast<cx<double>*>(smem_raw);
  cx<double>* bufB = bufA + M;
  const int tid = threadIdx.x;
  for (int j = tid; j < M; j += 256) bufA[j] = row[j];
  __syncthreads();
  cx<double>* Z = fft_forward<M, 256, double>(bufA, bufB, twM, tid);
  for (int j = tid; j < M; j += 256) row[j] = mk<double>(Z[j].x * scale, Z[j].y * scale);
}

struct FwdAnyArgs {
  const void* in;          // [nrows, 2L] float32 (or int16: I16) real rows
  const float* dat_scl;    // [nrows] int16 only
  const float* dat_offs;
  const double* in64;      // [nrows, 2L] float64 rows read instead of `in` when non-null (not with I16)
  cx<double>* spec;        // [nrows, Npad] out: slot k = harmonic k (1 <= k <= L), the rest zero
  double* dc;              // [nrows] out: harmonic 0, or null
  AnyPlan p;
  long nrows;
};

// rfft of real rows of length 2L: one CTA of 256 threads per row
template <int M, bool I16>
__global__ void __launch_bounds__(256) k_fwd_any(FwdAnyArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<double>* bufA = reinterpret_cast<cx<double>*>(smem_raw);
  cx<double>* bufB = bufA + (a.p.nrad > 0 ? a.p.L : M);   // (the launch sizes the shared memory accordingly)
  const int tid = threadIdx.x, L = a.p.L;
  for (long row = blockIdx.x; row < a.nrows; row += gridDim.x) {
    if constexpr (I16) {
      const short2* src = static_cast<const short2*>(a.in) + (size_t)row * L;
      const float scl = a.dat_scl[row], offs = a.dat_offs[row];
      for (int j = tid; j < L; j += 256) {
        const short2 v = src[j];
        bufA[j] = mk<double>((double)__fadd_rn(__fmul_rn((float)v.x, scl), offs), (double)__fadd_rn(__fmul_rn((float)v.y, scl), offs));
      }
    } else if (a.in64) {
      const double2* src = reinterpret_cast<const double2*>(a.in64) + (size_t)row * L;
      for (int j = tid; j < L; j += 256) { const double2 v = src[j]; bufA[j] = mk<double>(v.x, v.y); }
    } else {
      const float2* src = static_cast<const float2*>(a.in) + (size_t)row * L;
      for (int j = tid; j < L; j += 256) { const float2 v = src[j]; bufA[j] = mk<double>((double)v.x, (double)v.y); }
    }
    __syncthreads();
    const cx<double>* Z = bluestein<M, 256>(bufA, bufB, a.p, tid);
    cx<double>* out = a.spec + (size_t)row * a.p.Npad;
    for (int k = tid; k < a.p.Npad; k += 256) if (k == 0 || k > L) out[k] = mk<double>(0.0, 0.0);
    for (int p = tid + 1; 2 * p <= L; p += 256) {
      cx<double> dp, dq;
      unpack_pair<double>(Z, a.p.tw2n, L, p, dp, dq);
      out[p] = dp;
      if (2 * p < L) out[L - p] = dq;
    }
    if (tid == 0) {
      out[L] = mk<double>(Z[0].x - Z[0].y, 0.0);      // the Nyquist harmonic is real
      if (a.dc) a.dc[row] = Z[0].x + Z[0].y;
    }
    __syncthreads();   // Z (shared) is overwritten by the next row
  }
}

struct InvAnyArgs {
  const cx<double>* spec;  // [nrows, Npad] slot layout
  const double* dc;        // [nrows] harmonic 0 or null (= 0)
  void* out;               // [nrows, 2L] float32 or float64 real rows
  AnyPlan p;
  long nrows;
};

// irfft: the real rows of length 2L whose half spectra are given
template <int M, typename OutT>
__global__ void __launch_bounds__(256) k_inv_any(InvAnyArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<double>* bufA = reinterpret_cast<cx<double>*>(smem_raw);
  cx<double>* bufB = bufA + (a.p.nrad > 0 ? a.p.L : M);   // (the launch sizes the shared memory accordingly)
  const int tid = threadIdx.x, L = a.p.L;
  for (long row = blockIdx.x; row < a.nrows; row += gridDim.x) {
    const cx<double>* d = a.spec + (size_t)row * a.p.Npad;
    // packed spectrum Z (conjugated: the forward transform below then is the inverse one)
    for (int p = tid + 1; 2 * p <= L; p += 256) {
      const cx<double> dp = d[p], dq = (2 * p < L) ? d[L - p] : d[p];
      cx<double> zp, zq;
      pack_pair<double>(dp, dq, a.p.tw2n[p], zp, zq);
      bufA[p] = cconj(zp);
      if (2 * p < L) bufA[L - p] = cconj(zq);
    }
    if (tid == 0) {
      const double d0 = a.dc ? a.dc[row] : 0.0, dN = d[L].x;
      bufA[0] = mk<double>(0.5 * (d0 + dN), -0.5 * (d0 - dN));
    }
    __syncthreads();
    const cx<double>* Y = bluestein<M, 256>(bufA, bufB, a.p, tid);
    OutT* out = static_cast<OutT*>(a.out) + (size_t)row * 2 * L;
    const double sc = 1.0 / (double)L;
    for (int j = tid; j < L; j += 256) { out[2 * j] = (OutT)(Y[j].x * sc); out[2 * j + 1] = (OutT)(-Y[j].y * sc); }
    __syncthreads();
  }
}

}  // namespace ppb
