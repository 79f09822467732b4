// Hand-written sm_100a kernels of the wideband-TOA hot path.
//
//   k_model    conj(rfft(model)), |m|^2, p_n               (pplib.py:2129-2138)
//   k_prep     per-subint reference frequencies, counts    (pptoas.py:400-402)
//   k_spectra  K1+K2: per-channel rfft of the data, noise (get_noise_PS),
//              Sd, cross-spectrum X = d conj(m), partial frequency-averaged
//              profile spectra for the FFTFIT guess        (pplib.py:2127-2138,
//                                                           2227-2253; pptoas.py:422-424)
//   k_guess    K4: brute-force grid argmin + exact polish  (pplib.py:2054-2100)
//   k_pass2    K3: fused rotate-reduce C, C', C'' per channel (pplib.py:1315-1381)
//   k_update2  K3': per-subint reduction, safeguarded Newton step, epilogue
//              (nu_zero, covariance, scales, chi2)          (pplib.py:2146-2204,
//                                                           pptoaslib.py:1040-1096)
//
// Storage: X is float2 [subint][channel][N], N = nbin/2, slot j holds harmonic
// j for 1 <= j < N and slot 0 holds the Nyquist harmonic k = N (harmonic 0 is
// dropped: F0_fact = 0, pplib.py:66).  Rotation phasors and all accumulators
// are double precision.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <type_traits>

#include "fft.cuh"
#include "spectra_plan.cuh"
#include "bluestein.cuh"

namespace ppb {

constexpr double kDconst = 1.0 / 0.000241;  // pplib.py:48-51
constexpr double kTwoPi = 6.283185307179586476925286766559;
constexpr int kNCsum = 9;                   // per-channel sums kept per subint
// The first kLoK slots of every X row also keep the float32 rounding residual
// ("lo" part): the low harmonics carry almost all of |X|^2, so their float
// quantisation dominates the error of C_n (5.7e-9 rms of chi^2 on a 32x256
// portrait); with 64 lo slots it drops to ~2e-11 for +64/N traffic.
template <int N> struct LoK { static constexpr int value = N < 64 ? N : 64; };

// ----------------------------------------------------------------------------
// small device helpers
// ----------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deterministic CTA-wide sum of NV doubles per thread (result valid in all threads).
template <int NV, int NT>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* sh /* >= NV * NT/32 */) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  constexpr int NW = NT / 32;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) sh[i * NW + w] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < NW; ++j) s += sh[i * NW + j];
    v[i] = s;
  }
}

// e^{2 pi i x} in double precision for any finite x (range-reduced first).
__device__ __forceinline__ void cis2pi(double x, double& c, double& s) {
  x -= rint(x);
  sincospi(2.0 * x, &s, &c);
}

// (vx + i vy) e^{2 pi i x}, out of line: the rarely used DM_guess rotation of k_spectra
// would otherwise put one double sincospi per harmonic into its hot loop's code.
__device__ __noinline__ float2 rot2pi(float vx, float vy, double x) {
  double c, sn;
  cis2pi(x, c, sn);
  const float cf = (float)c, sf = (float)sn;
  return make_float2(vx * cf - vy * sf, vx * sf + vy * cf);
}

__device__ __forceinline__ double wrap_phase(double phi) {
  // pplib.py:2611-2613 / pptoaslib.py:1056-1057: onto [-0.5, 0.5)
  if (fabs(phi) >= 0.5) phi = phi - floor(phi);
  if (phi >= 0.5) phi -= 1.0;
  return phi;
}

// Model-side arrays (conj(m), |m|^2, p_n, cut-offs, frequency tables) hold nmodel models one after the other:
// [nmodel * nchan, ...] rows.  Subint s is fit against model index[s]; index null: model 0, the one model of
// pp_set_model.  A kernel reads channel ch of subint s's model at row row0(s) + ch (row0 is taken once per subint;
// the base pointers stay kernel parameters).
struct ModelRows {
  const int* index;   // [nsub] model of each subint (global subint index), or null
  int nchan;
  __device__ __forceinline__ int of(int s) const { return index ? __ldg(index + s) : 0; }
  __device__ __forceinline__ int row0(int s) const { return of(s) * nchan; }
};

// ----------------------------------------------------------------------------
// k_model: one CTA of 256 threads, RowGeom<N>::kRows channels at a time.
// Always runs in double (once per model); stores conj(m) both as double and
// rounded to float, |m|^2 as float, p_n as double.
// ----------------------------------------------------------------------------
struct ModelArgs {
  const float* model;   // [nchan, 2N]
  const double* model64;  // the same rows in double (then `model` is unused): no float32 rounding floor in the spectrum
  cx<float>* mconj32;   // [nchan, N] conj(m), slot layout
  cx<double>* mconj64;  // [nchan, N]
  double* mpow;         // [nchan, N] |m|^2, slot layout
  double* pn;           // [nchan]
  const cx<double>* twN;
  const cx<double>* tw2N;
  cx<double>* spec;     // [nchan, N + 1] or null: harmonic k at slot k, 0..N, and nothing else is written
                        // (the model spectra of pp_simulate_batch; the fit's model set is left alone)
  int nchan;
};

template <int N>
__global__ void __launch_bounds__(256) k_model(ModelArgs a) {
  using G = RowGeom<N>;
  using T = double;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufs = tw2N + (N / 2 + 2);
  __shared__ double red[8];
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  for (int i = tid; i < N; i += 256) twN[i] = a.twN[i];
  for (int i = tid; i <= N / 2; i += 256) tw2N[i] = a.tw2N[i];
  cx<T>* bufA = bufs + (size_t)r * 2 * N;
  cx<T>* bufB = bufA + N;
  const int ch = blockIdx.x * G::kRows + r;
  const bool valid = ch < a.nchan;
  if (a.model64) {
    const double2* src = reinterpret_cast<const double2*>(a.model64 + (size_t)(valid ? ch : 0) * 2 * N);
    for (int j = t_row; j < N; j += G::kTRow) {
      const double2 v = valid ? src[j] : make_double2(0.0, 0.0);
      bufA[j] = mk<T>(v.x, v.y);
    }
  } else {
    const float4* src = reinterpret_cast<const float4*>(a.model + (size_t)(valid ? ch : 0) * 2 * N);
#pragma unroll
    for (int m = 0; m < G::kLoads; ++m) {
      const int i4 = t_row + m * G::kTRow;
      const float4 v = valid ? src[i4] : make_float4(0, 0, 0, 0);
      bufA[2 * i4] = mk<T>(v.x, v.y);
      bufA[2 * i4 + 1] = mk<T>(v.z, v.w);
    }
  }
  __syncthreads();
  cx<T>* Z = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
  double psum = 0.0;
  const size_t ro = (size_t)(valid ? ch : 0) * N;
  auto put = [&](int slot, cx<T> d) {
    if (a.spec) {
      if (valid) a.spec[(size_t)ch * (N + 1) + (slot == 0 ? N : slot)] = d;
      return;
    }
    const double pw = d.x * d.x + d.y * d.y;
    psum += pw;
    if (valid) {
      a.mconj64[ro + slot] = cconj(d);
      a.mconj32[ro + slot] = mk<float>((float)d.x, (float)(-d.y));
      a.mpow[ro + slot] = pw;
    }
  };
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) {
    const int p = t_row + 1 + i * G::kTRow;
    if (p <= N / 2) {
      cx<T> dp, dq;
      unpack_pair<T>(Z, tw2N, N, p, dp, dq);
      put(p, dp);
      if (p < N / 2) put(N - p, dq);
    }
  }
  if (t_row == 0) put(0, mk<T>(Z[0].x - Z[0].y, 0.0));  // harmonic N (real)
  if (a.spec) {   // (uniform over the grid) harmonic 0: the row sum
    if (t_row == 0 && valid) a.spec[(size_t)ch * (N + 1)] = mk<T>(Z[0].x + Z[0].y, 0.0);
    return;
  }
  // reduce psum over the row-slot
#pragma unroll
  for (int o = (G::kTRow < 32 ? G::kTRow : 32) / 2; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
  if (G::kTRow > 32) {
    if ((tid & 31) == 0) red[tid >> 5] = psum;
    __syncthreads();
    if (t_row == 0) {
      double s = 0.0;
      for (int w = 0; w < G::kTRow / 32; ++w) s += red[r * (G::kTRow / 32) + w];
      psum = s;
    }
  }
  if (t_row == 0 && valid) a.pn[ch] = psum;
}

// mean over (all) channels of conj(m): one thread per slot, fixed order; grid.y = model.
__global__ void k_model_mean(const cx<double>* __restrict__ mconj, float2* __restrict__ mmean, int nchan, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  mconj += (size_t)blockIdx.y * nchan * N;
  mmean += (size_t)blockIdx.y * N;
  double sx = 0.0, sy = 0.0;
  for (int n = 0; n < nchan; ++n) {
    const cx<double> v = mconj[(size_t)n * N + i];
    sx += v.x; sy += v.y;
  }
  mmean[i] = make_float2((float)(sx / nchan), (float)(sy / nchan));
}

// mean of conj(m) over the USED channels of each subint (modelx.mean(axis=0) with
// modelx = model[ok_ichans], pptoas.py:446, 454) of the subint's model: grid (ceil(N/128), subints in chunk).
__global__ void k_model_mean_masked(const cx<double>* __restrict__ mconj, const uint8_t* __restrict__ mask,
                                    const float2* __restrict__ mmean_all, float2* __restrict__ out, int s0, int nchan,
                                    int N, ModelRows mr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int sl = blockIdx.y;
  if (i >= N) return;
  const int mi = mr.of(s0 + sl);
  mconj += (size_t)mi * nchan * N;
  mmean_all += (size_t)mi * N;
  const uint8_t* m = mask + (size_t)(s0 + sl) * nchan;
  double sx = 0.0, sy = 0.0;
  int cnt = 0;
  for (int n = 0; n < nchan; ++n) {
    if (m[n]) {
      const cx<double> v = mconj[(size_t)n * N + i];
      sx += v.x; sy += v.y; ++cnt;
    }
  }
  // nothing masked: bit-identical to the all-channel mean; nothing used: keep it finite
  out[(size_t)sl * N + i] = (cnt == nchan || cnt == 0) ? mmean_all[i] : make_float2((float)(sx / cnt), (float)(sy / cnt));
}

// FP64 pipe yardstick for the roofline record: independent DFMA chains, 8 per thread
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double a, double b) {
  double v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = threadIdx.x * 1e-3 + i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = fma(v[i], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += v[i];
  out[blockIdx.x * (size_t)blockDim.x + threadIdx.x] = s;
}

// float64 portraits (the reference's array type) -> the float32 the row kernels stage
__global__ void __launch_bounds__(256) k_cvt_f64_f32(const double2* __restrict__ in, float2* __restrict__ out, size_t n2) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x) {
    const double2 v = in[i];
    out[i] = make_float2((float)v.x, (float)v.y);
  }
}

// ----------------------------------------------------------------------------
// k_prep: one warp per subint.
// ----------------------------------------------------------------------------
struct PrepArgs {
  const double* freqs;      // [nchan]
  const uint8_t* mask;      // [nsub,nchan] or null
  const double* weights;    // [nsub,nchan] or null
  const double* snrs;       // [nsub,nchan] or null
  const double* nu_fits_in; // [nsub,3] or null
  double* nu_fit;           // [nsub,3] out
  double* nu_mean;          // [nsub] out
  double* wsum;             // [nsub] out
  int* nok;                 // [nsub] out
  int nsub, nchan, nu_fit_mode;
  ModelRows mr;             // freqs of the subint's model
};

__global__ void k_prep(PrepArgs a) {
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (s >= a.nsub) return;
  const int mb = a.mr.row0(s);
  double cnt = 0, ws = 0, fs = 0, fmin = 1e300, fmax = -1e300, num = 0, den = 0;
  for (int n = lane; n < a.nchan; n += 32) {
    const bool ok = a.mask ? (a.mask[(size_t)s * a.nchan + n] != 0) : true;
    if (!ok) continue;
    const double f = a.freqs[mb + n];
    cnt += 1.0;
    ws += a.weights ? a.weights[(size_t)s * a.nchan + n] : 1.0;
    fs += f;
    fmin = fmin < f ? fmin : f;
    fmax = fmax > f ? fmax : f;
  }
  cnt = warp_sum(cnt); ws = warp_sum(ws); fs = warp_sum(fs);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    fmin = fmin < __shfl_xor_sync(0xffffffffu, fmin, o) ? fmin : __shfl_xor_sync(0xffffffffu, fmin, o);
    fmax = fmax > __shfl_xor_sync(0xffffffffu, fmax, o) ? fmax : __shfl_xor_sync(0xffffffffu, fmax, o);
  }
  const double nu0 = 0.5 * (fmin + fmax);
  for (int n = lane; n < a.nchan; n += 32) {
    const bool ok = a.mask ? (a.mask[(size_t)s * a.nchan + n] != 0) : true;
    if (!ok) continue;
    const double f = a.freqs[mb + n];
    const double w = (a.snrs ? a.snrs[(size_t)s * a.nchan + n] : 1.0) / (f * f);
    num += (f - nu0) * w;
    den += w;
  }
  num = warp_sum(num); den = warp_sum(den);
  if (lane == 0) {
    const double mean = cnt > 0 ? fs / cnt : 0.0;
    a.nok[s] = (int)cnt;
    a.wsum[s] = ws;
    a.nu_mean[s] = mean;
    const double dflt = (a.nu_fit_mode == 1) ? (nu0 + num / den) : mean;  // pplib.py:2618-2632
    for (int i = 0; i < 3; ++i) {
      double v = a.nu_fits_in ? a.nu_fits_in[(size_t)s * 3 + i] : CUDART_NAN;
      if (!(v == v)) v = dflt;
      a.nu_fit[(size_t)s * 3 + i] = v;
    }
  }
}

// ----------------------------------------------------------------------------
// k_spectra: K1 + K2.  grid = (ceil(nchan/G), subints in chunk); a CTA holds
// PL::kSlots row slots of PL::kT threads and walks G channel rows (row plan PL:
// spectra_plan.cuh).  Rows arrive by TMA bulk copies into a double-buffered
// staging area; the FFT runs in double (DESIGN.md "precision"); X is stored as
// float2 plus the float32 residual of the first LoK slots.  Rows of nbin = 2048
// are transformed by k_spectra16 (spectra16.cuh) instead.
// ----------------------------------------------------------------------------
struct SpectraArgs {
  const void* data;          // [nsub,nchan,2N] float32 (or int16: k_spectra<N, PL, true>), global subint index
  const float* dat_scl;      // [nsub,nchan] int16 only: value = raw * dat_scl + dat_offs (PSRFITS DAT_SCL / DAT_OFFS)
  const float* dat_offs;     // [nsub,nchan]
  const cx<double>* mconj64; // [nchan,N]
  const cx<float>* mconj32;  // [nchan,N]
  const double* pn;          // [nchan]
  const double* nu2;         // [nchan] nu^-2
  const double* errs;        // [nsub,nchan] or null
  const uint8_t* mask;       // or null
  const double* weights;     // or null
  const double* P;           // [nsub]
  const double* DMg;         // [nsub] or null
  const double* nu_mean;     // [nsub]
  float2* X;                 // [chunk,nchan,N]  (null: do not store)
  float2* Xlo;               // [chunk,nchan,LoK<N>] float32 residuals of the first slots
  float2* partial;           // [chunk,nparts,N] (null: no guess)
  float2* D;                 // [chunk,nchan,N] data spectra d (slot layout) or null; kept for the
  double* Ddc;               // [chunk,nchan] ... and their DC terms: the fused ppalign accumulation
  double* sigma;             // [nsub,nchan] out
  double* Ssn;               // [nsub,nchan] out: p_n / sigma_F^2 (0 = channel unused)
  double* Sdn;               // [nsub,nchan] out
  const cx<double>* tw8;     // [TwLayout<N>::kTotal] per-pass twiddle tables
  int s0;                    // first global subint of the chunk
  int nchan, G, nparts;
  // arbitrary nbin (bluestein.cuh; k_spectra<N, PL, false, true>): the rows' FP64 spectra, already
  // transformed, in rows of N = Npad slots; the normalisations take the true nbin = 2 nhalf
  const cx<double>* dspec;   // [chunk,nchan,N] or null
  const double* ddc;         // [chunk,nchan] harmonic 0 of those rows
  int nhalf, kc_true;        // true nbin/2; first harmonic of the noise estimate, int(0.75 (nhalf + 1))
  const int* njn;            // [nchan] groups of 16 harmonics where the model has power (k_model_cutoff): X is stored
                             // for those only, the pass kernels read no others (null: all)
  ModelRows mr;              // mconj64, mconj32, pn, nu2, njn of the subint's model
};

template <int N, class PL = SpecPlan<N>, bool I16 = false, bool FROMSPEC = false>
__global__ void __launch_bounds__(PL::kThreads, PL::kMinBlocks) k_spectra(SpectraArgs a) {
  using F = double;
  constexpr int T = PL::kT, NS = PL::kSlots, NUNIT = PL::kUnits, NOUT = PL::kOut, NACC = NUNIT * NOUT;
  static_assert(NACC * T == N, "every harmonic slot has one owner");
  static_assert(FROMSPEC || !std::is_same<PL, SpecPlan16>::value, "nbin 2048 rows are transformed by k_spectra16");
  constexpr unsigned kRowBytes = 2 * N * (I16 ? sizeof(short) : sizeof(float));   // raw row as stored
  constexpr int NSTG = PL::kStages;   // staged raw rows per slot (TMA prefetch depth)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<F>* tw = reinterpret_cast<cx<F>*>(smem_raw);                       // [PL::kTwTotal] (+pad)
  cx<F>* bufs = tw + ((PL::kTwTotal + 1) & ~1);                         // [NS][N]
  float* stage_all = reinterpret_cast<float*>(bufs + (size_t)NS * N);   // [NS][NSTG][2N]
  __shared__ double red[2][NS][(T >= 32 ? T / 32 : 1)][2];   // per-warp power sums, by row parity
  __shared__ __align__(8) unsigned long long mbar[NS][2];
  const int tid = threadIdx.x, slot = tid / T, t = tid % T;
  if constexpr (!FROMSPEC) { for (int i = tid; i < PL::kTwTotal; i += PL::kThreads) tw[i] = a.tw8[i]; }
  if (t == 0) { mbar_init(&mbar[slot][0], 1); mbar_init(&mbar[slot][1], 1); }
  mbar_fence_init();
  __syncthreads();
  cx<F>* buf = bufs + (size_t)slot * N;
  float* stage = stage_all + (size_t)slot * NSTG * (2 * N);

  const int sl = blockIdx.y, s = a.s0 + sl;
  const int mb = a.mr.row0(s);   // the subint's model
  const int ch_begin = blockIdx.x * a.G;
  const int ch_end = min(ch_begin + a.G, a.nchan);
  const int nsteps = (a.G + NS - 1) / NS;
  constexpr int kc = (3 * (N + 1)) / 4;           // int(0.75*nharm), pplib.py:2244
  constexpr int ntop = N + 1 - kc;
  const bool want_guess = a.partial != nullptr;
  const double dmg = (want_guess && a.DMg) ? a.DMg[s] : 0.0;
  const double Dfac = dmg != 0.0 ? kDconst * dmg / a.P[s] : 0.0;  // pplib.py:2381
  const double numean = a.nu_mean[s];
  const double numean2 = 1.0 / (numean * numean);

  float2 acc[NACC];
  float2* const part_row = want_guess ? a.partial + ((size_t)sl * a.nparts + blockIdx.x * NS + slot) * N : nullptr;
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = make_float2(0.f, 0.f);
  double keep_all = 0.0, keep_top = 0.0;
  // thread r of a slot collects the power sums of row r (T > 32: from the per-warp totals)
  auto latch = [&](int r) {
    if constexpr (T > 32) {
      if (r == t) {
        double sa = 0.0, st = 0.0;
#pragma unroll
        for (int w = 0; w < T / 32; ++w) { sa += red[r & 1][slot][w][0]; st += red[r & 1][slot][w][1]; }
        keep_all = sa; keep_top = st;
      }
    }
  };

  auto row_used = [&](int step) -> bool {
    const int ch = ch_begin + step * NS + slot;
    if (step >= nsteps || ch >= ch_end) return false;
    return a.mask ? (a.mask[(size_t)s * a.nchan + ch] != 0) : true;
  };
  // TMA producer (one thread per slot): bulk-copy the raw row into the staging buffer
  auto fetch = [&](int step) {
    if constexpr (FROMSPEC) return;
    if (t == 0 && row_used(step)) {
      const int ch = ch_begin + step * NS + slot;
      unsigned long long* bar = &mbar[slot][step % NSTG];
      mbar_expect_tx(bar, kRowBytes);
      bulk_g2s(stage + (size_t)(step % NSTG) * 2 * N,
               static_cast<const char*>(a.data) + ((size_t)s * a.nchan + ch) * kRowBytes, kRowBytes, bar);
    }
  };
  fetch(0);
  if (NSTG > 1) fetch(1);
  unsigned ph0 = 0u, ph1 = 0u;

  for (int step = 0; step < nsteps; ++step) {
    const int ch = ch_begin + step * NS + slot;
    const bool inrange = ch < ch_end;
    const bool used = row_used(step);
    if (used && !FROMSPEC) {
      if (NSTG > 1 && (step & 1)) { mbar_wait(&mbar[slot][1], ph1); ph1 ^= 1u; }
      else { mbar_wait(&mbar[slot][0], ph0); ph0 ^= 1u; }
    }
    const float* graw = stage + (size_t)(step % NSTG) * 2 * N;
    auto make_src = [&]() {
      if constexpr (I16) {
        const size_t o = (size_t)s * a.nchan + (inrange ? ch : 0);
        return RowSrcI16{reinterpret_cast<const short2*>(graw), a.dat_scl[o], a.dat_offs[o]};
      } else {
        return RowSrcF32{reinterpret_cast<const float2*>(graw)};
      }
    };
    const auto g = make_src();
    // conj(model spectrum) of this thread's harmonics: L2 loads issued inside the last
    // FFT pass so that their latency hides behind its butterflies.  Output q of unit i
    // lives in slot PL::slot_of(t, i, q, first) (spectra_plan.cuh).
    // Slots >= LoK carry no lo part: float product and float conj(model) suffice there (kMix:
    // for N >= 512 the only lo slot a thread can own is slot t, output 0 of unit 0).
    constexpr bool kMix = (T >= 64);
    constexpr int kLo = LoK<N>::value;
    static_assert(kc == 3 * (N / 4), "PL::top() assumes the top quarter starts at 3N/4");
    const bool first = (t == 0);
    auto slot_of = [&](int i, int q) -> int { return PL::slot_of(t, i, q, first); };
    const bool doX = a.X != nullptr && inrange;
    const int kcut = (a.njn && inrange) ? 16 * a.njn[mb + ch] : N;
    const cx<F>* mc = a.mconj64 + (size_t)(mb + (inrange ? ch : 0)) * N;
    const cx<float>* mcf = a.mconj32 + (size_t)(mb + (inrange ? ch : 0)) * N;
    cx<F> mc64[kMix ? 1 : NACC];
    cx<float> mc32[kMix ? NACC : 1];
    auto load_mc = [&]() {
      if (doX && used) {
        if constexpr (kMix) mc64[0] = mc[t];
#pragma unroll
        for (int i = 0; i < NUNIT; ++i) {
#pragma unroll
          for (int q = 0; q < NOUT; ++q) {
            if constexpr (kMix) mc32[NOUT * i + q] = mcf[slot_of(i, q)];
            else mc64[NOUT * i + q] = mc[slot_of(i, q)];
          }
        }
      } else {   // unused rows store zeros
        if constexpr (kMix) mc64[0] = mk<F>(0.0, 0.0);
#pragma unroll
        for (int i = 0; i < NACC; ++i) {
          if constexpr (kMix) mc32[i] = mk<float>(0.f, 0.f);
          else mc64[i] = mk<F>(0.0, 0.0);
        }
      }
    };
    // per-row scalars: loaded before the transform so that their latency is hidden
    float2* const Xrow = a.X + ((size_t)sl * a.nchan + (inrange ? ch : 0)) * N;
    float2* const Xlorow = a.Xlo + ((size_t)sl * a.nchan + (inrange ? ch : 0)) * kLo;
    float2* const Drow = a.D + ((size_t)sl * a.nchan + (inrange ? ch : 0)) * N;
    const float wgt = (used && want_guess) ? (float)(a.weights ? a.weights[(size_t)s * a.nchan + ch] : 1.0) : 0.f;
    const double shift = (Dfac != 0.0 && inrange) ? Dfac * (a.nu2[mb + ch] - numean2) : 0.0;
    if constexpr (FROMSPEC) {     // the rows arrive transformed: only the barrier discipline of the power-sum hand-off
      PL::sync(slot);
      latch(step - 1);
      load_mc();
      (void)g;
    } else {
      PL::template transform<F>(buf, tw, t, slot, g, used, [&]() { fetch(step + NSTG); latch(step - 1); }, load_mc);
    }
    const cx<F>* const dsrow = FROMSPEC ? a.dspec + ((size_t)sl * a.nchan + (inrange ? ch : 0)) * N : nullptr;

    // ---- split + power sums; X and the guess accumulators need no sigma ------------
    double s_all = 0.0, s_top = 0.0;
    float wrow = wgt;
    // rows that arrive transformed: thread 0's first output is slot 0, which holds no harmonic of the row, so
    // the test below cannot see a non-finite row there; the row's DC term can
    if (FROMSPEC && used && !isfinite(a.ddc[(size_t)sl * a.nchan + ch])) wrow = 0.f;
#pragma unroll
    for (int i = 0; i < NUNIT; ++i) {
      cx<F> d[NOUT];
      F dc_term = F(0);
      if constexpr (FROMSPEC) {
#pragma unroll
        for (int q = 0; q < NOUT; ++q) d[q] = used ? dsrow[slot_of(i, q)] : mk<F>(F(0), F(0));
        if (i == 0 && first && used) dc_term = a.ddc[(size_t)sl * a.nchan + ch];
      } else {
        dc_term = PL::template split<F>(buf, tw, t, i, first, d);   // DC of the row (special unit only)
      }
      // a NaN / Inf sample makes every harmonic of the row non-finite: such a row must not enter
      // the profile for the FFTFIT guess (its sigma comes out non-finite, so the fit skips it too)
      if (i == 0 && !(isfinite(d[0].x) && isfinite(d[0].y))) wrow = 0.f;
      float vx[NOUT], vy[NOUT];
      double sa0 = 0.0, sa1 = 0.0;      // two chains: the power sum is latency, not throughput, bound
#pragma unroll
      for (int q = 0; q < NOUT; ++q) {
        double& sa = (q & 1) ? sa1 : sa0;
        if (FROMSPEC) {                             // any nbin: the cut is a run-time harmonic (slot = harmonic)
          const double pw = fma(d[q].x, d[q].x, d[q].y * d[q].y);
          sa += pw;
          if (slot_of(i, q) >= a.kc_true) s_top += pw;
        } else if (q == 1 || q == 6 || q == 0) {    // outputs that can be in the top quarter (PL::top)
          const double pw = fma(d[q].x, d[q].x, d[q].y * d[q].y);
          sa += pw;
          if (PL::top(i, q, first)) s_top += pw;    // harmonics >= kc = 3N/4
        } else {
          sa = fma(d[q].x, d[q].x, sa);
          sa = fma(d[q].y, d[q].y, sa);
        }
        vx[q] = (float)d[q].x; vy[q] = (float)d[q].y;
      }
      s_all += sa0 + sa1;
      if (doX) {        // uniform over the row
#pragma unroll
        for (int q = 0; q < NOUT; ++q) {
          const int idx = NOUT * i + q;
          const int sk = slot_of(i, q);
          if (sk >= kcut) continue;      // the model has no power there: never read
          bool lo;
          if constexpr (kMix) lo = (i == 0 && q == 0) && (t < kLo);
          else lo = true;
          if (!lo) {
            const cx<float> m = mc32[kMix ? idx : 0];
            Xrow[sk] = make_float2(fmaf(vx[q], m.x, -vy[q] * m.y), fmaf(vx[q], m.y, vy[q] * m.x));
          } else {
            const cx<F> pr = cmul(d[q], mc64[kMix ? 0 : idx]);
            const float2 xv = make_float2((float)pr.x, (float)pr.y);
            Xrow[sk] = xv;
            if (kMix || sk < kLo) Xlorow[sk] = make_float2((float)(pr.x - (double)xv.x), (float)(pr.y - (double)xv.y));
          }
        }
      }
      if (a.D != nullptr && inrange) {     // uniform: raw spectra for k_align_spec (unused rows are skipped there)
#pragma unroll
        for (int q = 0; q < NOUT; ++q) Drow[slot_of(i, q)] = make_float2(vx[q], vy[q]);
        if (i == 0 && first) a.Ddc[(size_t)sl * a.nchan + ch] = dc_term;
      }
      if (shift != 0.0) {           // rotate_data with DM_guess (pptoas.py:422); uniform, rare
#pragma unroll
        for (int q = 0; q < NOUT; ++q) {
          const int sk = slot_of(i, q);
          const float2 r = rot2pi(vx[q], vy[q], (double)(sk == 0 ? N : sk) * shift);
          // the Nyquist term (slot 0; harmonic nbin/2 in slot nhalf of rows that arrive transformed) keeps its
          // real part only, as the irfft of rotate_data does
          const bool nyquist = FROMSPEC ? (sk == a.nhalf) : (sk == 0);
          vx[q] = r.x; vy[q] = nyquist ? 0.f : r.y;
        }
      }
      if (wrow != 0.f) {   // uniform: 0 when no guess is wanted, the row is unused or not finite
#pragma unroll
        for (int q = 0; q < NOUT; ++q) {
          acc[NOUT * i + q].x = fmaf(wrow, vx[q], acc[NOUT * i + q].x);
          acc[NOUT * i + q].y = fmaf(wrow, vy[q], acc[NOUT * i + q].y);
        }
      }
    }
    // ---- power sums of the row: warp totals go to shared memory (by row parity); thread
    // `step` of the slot picks them up after the next barrier (inside the next transform)
    if constexpr (T > 32) {
      s_all = warp_sum(s_all); s_top = warp_sum(s_top);
      if ((tid & 31) == 0) { red[step & 1][slot][t >> 5][0] = s_all; red[step & 1][slot][t >> 5][1] = s_top; }
    } else {
#pragma unroll
      for (int o = T / 2; o > 0; o >>= 1) {
        s_all += __shfl_xor_sync(0xffffffffu, s_all, o);
        s_top += __shfl_xor_sync(0xffffffffu, s_top, o);
      }
      if (step == t) { keep_all = s_all; keep_top = s_top; }
    }
  }
  // ---- noise, Sd, S: one row per thread (the host keeps nsteps <= T), so that the sqrt and
  // the two divisions are off the per-row critical path ------------------------------------
  if constexpr (T > 32) { PL::sync(slot); latch(nsteps - 1); }
  {
    const int fch = ch_begin + t * NS + slot;
    if (t < nsteps && fch < ch_end) {
      const bool fused = row_used(t);
      double sig;
      const double nh = FROMSPEC ? (double)a.nhalf : (double)N;             // true nbin / 2
      const double nt = FROMSPEC ? (double)(a.nhalf + 1 - a.kc_true) : (double)ntop;
      if (a.errs) sig = fused ? a.errs[(size_t)s * a.nchan + fch] : 0.0;
      else sig = sqrt(keep_top / (2.0 * nh * nt));                         // pplib.py:2243-2245
      const double sF2 = sig * sig * nh;                                  // sigma^2 * nbin/2
      const bool ok = fused && (sF2 > 0.0) && (sF2 < 1e300);
      const size_t o = (size_t)s * a.nchan + fch;
      a.sigma[o] = ok ? sig : 0.0;
      a.Ssn[o] = ok ? a.pn[mb + fch] / sF2 : 0.0;
      a.Sdn[o] = ok ? keep_all / sF2 : 0.0;
    }
  }
  if (want_guess) {
    const bool first = (t == 0);
#pragma unroll
    for (int i = 0; i < NUNIT; ++i) {
#pragma unroll
      for (int q = 0; q < NOUT; ++q) part_row[PL::slot_of(t, i, q, first)] = acc[NOUT * i + q];
    }
  }
}

}  // namespace ppb
#include "spectra16.cuh"
namespace ppb {

// ----------------------------------------------------------------------------
// k_guess: K4, one CTA (256 threads) per profile / subint.
// ----------------------------------------------------------------------------
struct GuessArgs {
  const float2* partial;   // [n, nparts, N] spectra to be summed (slot layout)
  const float2* mconj;     // [nmodel, N] conj(model spectrum)
  int nparts, nmodel, N, Ns;
  int nhalf;               // true nbin/2 when the spectra sit in N = Npad > nbin/2 slots (arbitrary nbin), else 0
  int nused;               // the grid and the polish sum over slots 1..nused only (the model's harmonic cut-off: the
                           // products d_k conj(m_k) beyond it are nothing); 0 or N: all of them, Nyquist included
  double polish_tol;       // stop the exact polish when |dx| < polish_tol [rot]
  const double* wsum;      // [n] divisor of the partial sum, or null (=1)
  const double* noise;     // [n] time-domain sigma or null (measure from spectrum)
  const double2* table;    // [Ns-1] e^{2 pi i m/(Ns-1)}; general grid: [Ns] e^{2 pi i phi_j}
  int grid_general;        // 0: np.mgrid[-0.5:0.5:Ns j]; 1: phi_j = phi_lo + j phi_step (other bounds)
  double phi_lo, phi_step;
  int s0;                  // global index offset for per-subint arrays below
  // outputs of the 1-D fit (global index), any may be null
  double* phase; double* phase_err; double* scale; double* scale_err; double* snr; double* red_chi2;
  int* lag;
  // solver start state (fit batch only; null for the stand-alone 1-D fit)
  double* x;               // [nsub,5]
  const double* DMg;       // [nsub] or null
  const double* P;         // [nsub]
  const double* nu_mean;   // [nsub]
  const double* nu_fit;    // [nsub,3]
  const double* init;      // [nsub,5] or null: template for GM,tau,alpha start values
  const double* scat;      // [nsub,2] tau_guess [rot, linear] and alpha_guess, or null
  int log10_tau, fit_scat;
  // fit batch with several models: subint s uses template model[s] when tmpl_by_model (else the i mod nmodel rule,
  // which picks the per-subint masked templates) and the cut-off nused_of[model[s]]; model null: one model
  const int* model;        // [nsub] or null
  const int* nused_of;     // [nmodel]
  int tmpl_by_model;
};

__global__ void __launch_bounds__(256) k_guess(GuessArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* Y = reinterpret_cast<double2*>(smem_raw);  // [N]
  __shared__ double sh[8 * 4];
  __shared__ double bestv[8];
  __shared__ int besti[8];
  __shared__ double bc[4];
  const int N = a.N, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int il = blockIdx.x, ig = a.s0 + il;
  const int NH = a.nhalf > 0 ? a.nhalf : N;          // true nbin/2: noise cut, normalisations, degrees of freedom
  const int kc = (3 * (NH + 1)) / 4;
  const double inv_w = a.wsum ? 1.0 / a.wsum[ig] : 1.0;
  const int mi = a.model ? __ldg(a.model + ig) : 0;
  // profile i uses model i mod nmodel, a subint of a batch with several models its own model's template
  const float2* mc = a.mconj + (size_t)(a.tmpl_by_model ? mi : (a.nmodel > 1 ? il % a.nmodel : 0)) * N;
  const int nused = a.model ? __ldg(a.nused_of + mi) : a.nused;
  double v[3] = {0.0, 0.0, 0.0};  // sum |d|^2, sum |m|^2, top-quarter power
  const double tau_g = (a.scat && a.fit_scat) ? a.scat[(size_t)ig * 2] : 0.0;
  for (int i = tid; i < N; i += 256) {
    float sx = 0.f, sy = 0.f;
    for (int q = 0; q < a.nparts; ++q) {
      const float2 t = a.partial[((size_t)il * a.nparts + q) * N + i];
      sx += t.x; sy += t.y;
    }
    const double dx = (double)sx * inv_w, dy = (double)sy * inv_w;
    const int k = (i == 0) ? N : i;   // (arbitrary nbin: slot 0 and the slots above nbin/2 are zero)
    double mx = mc[i].x, my = mc[i].y;
    if (tau_g != 0.0) {   // scattered mean model (pptoas.py:444-447): conj(m B) = conj(m) conj(B)
      const double b = kTwoPi * (double)k * tau_g, q = 1.0 / (1.0 + b * b);
      const double tx = mx * q - my * (b * q);
      // the irfft there keeps the real part of the Nyquist term: Re(B m) at k = nbin/2
      my = (k == NH) ? 0.0 : mx * (b * q) + my * q; mx = tx;
    }
    Y[i] = make_double2(dx * mx - dy * my, dx * my + dy * mx);
    const double pw = dx * dx + dy * dy;
    v[0] += pw;
    v[1] += mx * mx + my * my;
    if (k >= kc) v[2] += pw;
  }
  block_sum<3, 256>(v, sh);
  double err2;  // Fourier-domain variance (pplib.py:2076-2079)
  if (a.noise) { const double nz = a.noise[ig]; err2 = nz * nz * (double)NH; }
  else err2 = v[2] / ((double)(2 * NH) * (double)(NH + 1 - kc)) * (double)NH;
  const double d_tot = v[0] / err2, p_tot = v[1] / err2;

  // ---- brute-force grid (scipy.optimize.brute over np.mgrid[-0.5:0.5:Ns j]) ----
  // phi_j = -1/2 + j/M, M = Ns - 1:  C_j = -Re sum_k Y_k e^{-i pi k} rho_j^k / err2 with rho_j = e^{2 pi i j/M}.
  // One grid point per lane; the phasors of the odd and of the even harmonics advance by rho_j^2
  // (two independent FP64 recurrences, no table look-up or index arithmetic in the loop); Y_k is a
  // shared-memory broadcast.  Harmonic N sits in slot 0.
  const int M = a.Ns - 1;
  const int NU = (nused > 0 && nused < N) ? (nused & ~1) : N;   // even
  double bv = CUDART_INF;
  int bi = 0x7fffffff;
  for (int j0 = w * 32; j0 < a.Ns; j0 += 256) {
    const int j = j0 + lane;
    if (j < a.Ns) {
      const double2 r1 = a.grid_general ? a.table[j] : a.table[j % M];
      const cx<double> rho = mk<double>(r1.x, r1.y), rho2 = csqr(rho);
      cx<double> po = rho, pe = rho2;                 // harmonics 1 and 2
      double acc_o = 0.0, acc_e = 0.0;
#pragma unroll 4
      for (int m = 0; m < NU / 2; ++m) {
        const double2 yo = Y[2 * m + 1];
        const double2 ye = Y[(2 * m + 2 == N) ? 0 : 2 * m + 2];
        acc_o = fma(yo.x, po.x, fma(-yo.y, po.y, acc_o));
        acc_e = fma(ye.x, pe.x, fma(-ye.y, pe.y, acc_e));
        po = cmul(po, rho2);
        pe = cmul(pe, rho2);
      }
      // default grid: e^{-i pi k} of phi = -1/2 + j/M, i.e. the odd harmonics change sign
      const double cj = a.grid_general ? -(acc_e + acc_o) / err2 : -(acc_e - acc_o) / err2;
      if (cj < bv) { bv = cj; bi = j; }                // j ascending within a lane: first index wins ties
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {                   // warp argmin, lowest index on ties
    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) { bestv[w] = bv; besti[w] = bi; }
  __syncthreads();
  if (tid == 0) {
    double b = bestv[0]; int ib = besti[0];
    for (int q = 1; q < 8; ++q)
      if (bestv[q] < b || (bestv[q] == b && besti[q] < ib)) { b = bestv[q]; ib = besti[q]; }
    besti[0] = ib;
  }
  __syncthreads();
  const int lagi = besti[0];
  const double h = a.grid_general ? a.phi_step : 1.0 / (double)M;
  double x = (a.grid_general ? a.phi_lo : -0.5) + (double)lagi * h;
  double lo = x - h, hi = x + h;
  double C0 = 0, C1 = 0, C2 = 0;
  // ---- exact polish: safeguarded Newton on C'(phi) = 0 inside the bracket ------
  for (int it = 0; it < 60; ++it) {
    double u[3] = {0.0, 0.0, 0.0};
    for (int i = tid; i < (NU < N ? NU + 1 : N); i += 256) {
      if (i == 0 && NU < N) continue;          // slot 0 is the Nyquist harmonic
      const int k = (i == 0) ? N : i;
      double c, sn;
      cis2pi((double)k * x, c, sn);
      const double re = Y[i].x * c - Y[i].y * sn;
      const double im = Y[i].x * sn + Y[i].y * c;
      const double wk = kTwoPi * (double)k;
      u[0] -= re;            // C   (pplib.py:1244-1256)
      u[1] += wk * im;       // C'  (1258-1268)
      u[2] += wk * wk * re;  // C'' (1270-1280)
    }
    block_sum<3, 256>(u, sh);
    C0 = u[0] / err2; C1 = u[1] / err2; C2 = u[2] / err2;
    if (tid == 0) {
      if (C1 < 0.0) lo = x; else hi = x;
      double xn = (C2 > 0.0) ? x - C1 / C2 : CUDART_NAN;
      if (!(xn > lo && xn < hi)) xn = 0.5 * (lo + hi);
      bc[0] = xn; bc[1] = lo; bc[2] = hi;
      bc[3] = (fabs(xn - x) < a.polish_tol || C1 == 0.0) ? 1.0 : 0.0;
    }
    __syncthreads();
    const bool stop = bc[3] != 0.0;
    const double xn = bc[0];
    if (!stop) { x = xn; lo = bc[1]; hi = bc[2]; }
    __syncthreads();
    if (stop) { if (a.x) x = xn; break; }   // start value of the solver: take the last (tiny) step too
  }
  if (tid == 0) {
    const double fmin = C0;
    const double scale = -fmin / p_tot;
    if (a.phase) a.phase[ig] = x;
    if (a.lag) a.lag[ig] = lagi;
    if (a.phase_err) a.phase_err[ig] = 1.0 / sqrt(scale * C2);       // pplib.py:2092-2093
    if (a.scale) a.scale[ig] = scale;
    if (a.scale_err) a.scale_err[ig] = 1.0 / sqrt(p_tot);
    if (a.red_chi2) a.red_chi2[ig] = (d_tot - fmin * fmin / p_tot) / (double)(2 * NH - 2);
    if (a.snr) a.snr[ig] = sqrt(scale * scale * p_tot);
    if (a.x) {
      const double dmg = a.DMg ? a.DMg[ig] : 0.0;
      const double nm = a.nu_mean[ig], nf = a.nu_fit[(size_t)ig * 3];
      // phase_transform(phi, DM_guess, nu_mean, nu_fit_DM, P, mod=True) (pptoas.py:456)
      double ph = x + kDconst * dmg / a.P[ig] * (1.0 / (nf * nf) - 1.0 / (nm * nm));
      ph = wrap_phase(ph);
      double* xs = a.x + (size_t)ig * 5;
      xs[0] = ph; xs[1] = dmg;
      xs[2] = a.init ? a.init[(size_t)ig * 5 + 2] : 0.0;
      xs[3] = a.init ? a.init[(size_t)ig * 5 + 3] : 0.0;
      xs[4] = a.init ? a.init[(size_t)ig * 5 + 4] : 0.0;
      if (a.scat) {                                  // pptoas.py:427-452
        double tg = a.scat[(size_t)ig * 2];
        if (a.log10_tau) { if (tg == 0.0) tg = 1.0 / (double)(2 * NH); tg = log10(tg); }
        xs[3] = tg; xs[4] = a.scat[(size_t)ig * 2 + 1];
      }
    }
  }
}

// ----------------------------------------------------------------------------
// Solver state (struct of arrays, global subint index)
// ----------------------------------------------------------------------------
struct SolverState {
  double* x;        // [nsub,5] current evaluation point (at nu_fit)
  double* xprev;    // [nsub,5] last accepted point
  double* step;     // [nsub,5] last proposed step
  double* fprev;    // [nsub]
  double* lam;      // [nsub] backtracking factor
  int* iter;        // [nsub] passes done
  int* iterc;       // [nsub] evaluations of the coarse objectives (general solver), not counted against max_iter
  int* done;        // [nsub] 0 running, 1 finished
};

// Box constraints on the parameters at the fit reference frequencies (scipy TNC bounds:
// pplib.py:2146-2148, pptoaslib.py:1008-1014).  Handled by the Newton solvers as an active set:
// a parameter that sits on a bound with the gradient pushing outwards is held for that step,
// steps are clipped to the box.
struct Box {
  double lo[5], hi[5];
  int on;
};
__device__ __forceinline__ bool box_holds(const Box& b, int p, double x, double g) {
  return b.on && ((x <= b.lo[p] && g > 0.0) || (x >= b.hi[p] && g < 0.0));
}
__device__ __forceinline__ double box_clip(const Box& b, int p, double xn, bool& clipped) {
  if (!b.on) return xn;
  if (xn < b.lo[p]) { clipped = true; return b.lo[p]; }
  if (xn > b.hi[p]) { clipped = true; return b.hi[p]; }
  return xn;
}

// ----------------------------------------------------------------------------
// k_pass2: K3 for (phi, DM).  8 lanes per channel row, 4 rows per warp,
// 8 warps per CTA: grid = (ceil(nchan/32), subints in chunk).
// ----------------------------------------------------------------------------
struct PassArgs {
  const float2* X;         // [chunk,nchan,N]
  const float2* Xlo;       // [chunk,nchan,LoK<N>]
  const double* nu2;       // [nchan]
  const double* P;         // [nsub]
  const double* nu_fit;    // [nsub,3]
  const double* Ssn;       // [nsub,nchan] (0 => unused channel)
  const double* sigma;     // [nsub,nchan]
  double* csum;            // [nsub,nchan,kNCsum]
  SolverState st;
  int s0, nchan, N;
  int nhalf;               // true nbin/2 of the noise normalisation (0: N; arbitrary nbin runs on N = Npad slots)
  const int* njn;          // [nchan] groups of 16 harmonics where the model has power (k_model_cutoff); N/16 = all
  ModelRows mr;            // nu2, njn of the subint's model
};

// streaming 16-byte load: read-only path, do not keep in L1
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// 16-byte asynchronous copy global -> shared (L2 only), thread-private use: the issuing thread alone reads the
// destination, after cp.async.wait_group
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int NPEND> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(NPEND) : "memory");
}

// k_pass2 / k_pass5 can keep D iterations of loads (16 bytes per thread each) in flight through a thread-private ring
// in shared memory instead of registers
template <int N> struct Pass2Ring {
  static constexpr int NJ = N / 16;
  static constexpr int D = NJ < 8 ? NJ : 8;
  static constexpr int KJ = LoK<N>::value / 16;
  static constexpr size_t kBytes = sizeof(float4) * 256 * (D + KJ);
  static constexpr int kMinBlocks = 4;   // CTAs per SM asked of the compiler
};
template <int N>
__global__ void __launch_bounds__(256, Pass2Ring<N>::kMinBlocks) k_pass2(PassArgs a) {
  const int sl = blockIdx.y, s = a.s0 + sl;
  if (a.st.done[s] == 1) return;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int sub = lane >> 3, l8 = lane & 7;
  const int ch = blockIdx.x * 32 + w * 4 + sub;
  const bool inrange = ch < a.nchan;
  const int chc = inrange ? ch : a.nchan - 1;
  const double Ssn = a.Ssn[(size_t)s * a.nchan + chc];
  const bool used = inrange && Ssn > 0.0;

  // C3, C4: sums for the third and fourth theta-derivatives; they let k_update2 follow the objective
  // along the Newton path without another pass over X
  double C = 0.0, C1 = 0.0, C2 = 0.0, C3 = 0.0, C4 = 0.0;
  if (used) {
    const int mb = a.mr.row0(s);   // the subint's model
    const double phi = a.st.x[(size_t)s * 5 + 0], DM = a.st.x[(size_t)s * 5 + 1];
    const double nf = a.nu_fit[(size_t)s * 3 + 0];
    const double g = kDconst * (a.nu2[mb + ch] - 1.0 / (nf * nf)) / a.P[s];
    double theta = phi + DM * g;               // pplib.py:1319-1320
    theta -= rint(theta);
    const float4* row = reinterpret_cast<const float4*>(a.X + ((size_t)sl * a.nchan + ch) * N);
    constexpr int NJ = N / 16;
    constexpr int KJ = LoK<N>::value / 16;                     // iterations that carry lo parts
    constexpr int D = Pass2Ring<N>::D;
    const int nj = a.njn[mb + ch];                             // groups of 16 harmonics the model has power in (>= KJ)
    const float4* lorow = reinterpret_cast<const float4*>(a.Xlo + ((size_t)sl * a.nchan + ch) * LoK<N>::value);
    // the X row pieces arrive through a thread-private ring in shared memory (cp.async, D iterations in flight);
    // the first copies go out before the phasor set-up so that its latency is hidden
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* rv = reinterpret_cast<float4*>(smem_raw) + tid;   // [D][256] X pieces
    float4* rl = rv + D * 256;                                // [KJ][256] float32 residuals of the low harmonics
    auto ring_issue = [&](int j) {                            // one commit group per iteration, empty past the end
      if (j < nj) cp_async16(rv + (j % D) * 256, row + j * 8 + l8);
      cp_async_commit();
    };
#pragma unroll
    for (int j = 0; j < KJ; ++j) cp_async16(rl + j * 256, lorow + j * 8 + l8);
#pragma unroll
    for (int j = 0; j < D - 1; ++j) ring_issue(j);
    // element (j, e): complex index 16 j + 2 l8 + e, harmonic k = index (slot 0 = Nyquist).
    // Phasors e^{2 pi i k theta} for k = 2 l8, 2 l8 + 1 and the step 16 from one sincospi and
    // repeated squaring (phase error ~1e-15 rad, far inside the chi^2 tolerance).
    double c0, s0, c1, s1, cw, sw;
    cx<double> e1, e2, e4, e8, e16;
    cis2pi(theta, e1.x, e1.y);
    e2 = csqr(e1); e4 = csqr(e2); e8 = csqr(e4); e16 = csqr(e8);
    {
      cx<double> z = mk<double>(1.0, 0.0);
      if (l8 & 1) z = e2;
      if (l8 & 2) z = cmul(z, e4);
      if (l8 & 4) z = cmul(z, e8);
      c0 = z.x; s0 = z.y;
      const cx<double> z1 = cmul(z, e1);
      c1 = z1.x; s1 = z1.y;
      cw = e16.x; sw = e16.y;
    }
    double k0 = (double)(2 * l8), k1 = (double)(2 * l8 + 1);
    auto accum = [&](double xr0, double xi0, double xr1, double xi1) {
      const double re0 = xr0 * c0 - xi0 * s0, im0 = xr0 * s0 + xi0 * c0;
      const double re1 = xr1 * c1 - xi1 * s1, im1 = xr1 * s1 + xi1 * c1;
      const double kk0 = k0 * k0, kk1 = k1 * k1;
      const double ki0 = k0 * im0, ki1 = k1 * im1;     // k Im z
      const double kr0 = kk0 * re0, kr1 = kk1 * re1;   // k^2 Re z
      C += re0 + re1;
      C1 += ki0 + ki1;
      C2 += kr0 + kr1;
      C3 = fma(kk0, ki0, C3); C3 = fma(kk1, ki1, C3);
      C4 = fma(kk0, kr0, C4); C4 = fma(kk1, kr1, C4);
      // advance both phasors by 16 harmonics
      const double t0 = c0 * cw - s0 * sw; s0 = c0 * sw + s0 * cw; c0 = t0;
      const double t1 = c1 * cw - s1 * sw; s1 = c1 * sw + s1 * cw; c1 = t1;
      k0 += 16.0; k1 += 16.0;
    };
    // iteration j: wait for its copy, read its slot, refill the slot read one iteration ago.
    // The first KJ iterations carry the float32 residuals of the low harmonics.
#pragma unroll
    for (int j = 0; j < KJ; ++j) {
      cp_async_wait<(D >= 2 ? D - 2 : 0)>();
      float4 v = rv[(j % D) * 256], lo = rl[j * 256];
      ring_issue(j + D - 1);
      if (j == 0 && l8 == 0) { v.x = 0.f; v.y = 0.f; lo.x = 0.f; lo.y = 0.f; }   // slot 0 is handled below
      accum((double)v.x + (double)lo.x, (double)v.y + (double)lo.y, (double)v.z + (double)lo.z, (double)v.w + (double)lo.w);
    }
#pragma unroll 4
    for (int j = KJ; j < nj; ++j) {
      cp_async_wait<(D >= 2 ? D - 2 : 0)>();
      const float4 v = rv[(j % D) * 256];
      ring_issue(j + D - 1);
      accum((double)v.x, (double)v.y, (double)v.z, (double)v.w);
    }
    if (l8 == 0 && nj == NJ) {  // Nyquist harmonic k = N stored in slot 0
      const float2 xh = __ldg(reinterpret_cast<const float2*>(row));
      const float2 xl = __ldg(reinterpret_cast<const float2*>(lorow));
      const double xnx = (double)xh.x + (double)xl.x, xny = (double)xh.y + (double)xl.y;
      cx<double> en = e16;          // e^{2 pi i N theta} = (e^{2 pi i 16 theta})^(N/16)
#pragma unroll
      for (int q = 16; q < N; q *= 2) en = csqr(en);
      const double cn = en.x, sn = en.y;
      const double re = xnx * cn - xny * sn;
      const double im = xnx * sn + xny * cn;
      const double n1 = (double)N, n2 = n1 * n1;
      C += re; C1 = fma(n1, im, C1); C2 = fma(n2, re, C2); C3 = fma(n2 * n1, im, C3); C4 = fma(n2 * n2, re, C4);
    }
  }
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) {
    C += __shfl_xor_sync(0xffffffffu, C, o);
    C1 += __shfl_xor_sync(0xffffffffu, C1, o);
    C2 += __shfl_xor_sync(0xffffffffu, C2, o);
    C3 += __shfl_xor_sync(0xffffffffu, C3, o);
    C4 += __shfl_xor_sync(0xffffffffu, C4, o);
  }
  if (inrange && l8 == 0) {
    double* o = a.csum + ((size_t)s * a.nchan + ch) * kNCsum;
    if (used) {
      const double sg = a.sigma[(size_t)s * a.nchan + ch];
      const double isF2 = 1.0 / (sg * sg * (double)(a.nhalf > 0 ? a.nhalf : N));
      o[0] = C * isF2;                         // C_n      (pplib.py:1322)
      o[1] = -kTwoPi * C1 * isF2;              // dC/dtheta  (1344)
      o[2] = -kTwoPi * kTwoPi * C2 * isF2;     // d2C/dtheta2 (1380)
      o[3] = kTwoPi * kTwoPi * kTwoPi * C3 * isF2;             // d3C/dtheta3 = Re sum (2 pi i k)^3 X e^{..}
      o[4] = kTwoPi * kTwoPi * kTwoPi * kTwoPi * C4 * isF2;    // d4C/dtheta4
    } else {
      o[0] = 0.0; o[1] = 0.0; o[2] = 0.0; o[3] = 0.0; o[4] = 0.0;
    }
  }
}

// ----------------------------------------------------------------------------
// k_update2: K3' for (phi, DM): one CTA of 128 threads per subint.
// ----------------------------------------------------------------------------
struct UpdateArgs {
  const double* csum;      // [nsub,nchan,kNCsum]
  const double* Ssn;       // [nsub,nchan]
  const double* Sdn;       // [nsub,nchan]
  const double* nu2;       // [nchan]
  const double* freqs;     // [nchan]
  const double* P;         // [nsub]
  const double* nu_fit;    // [nsub,3]
  const double* nu_outs;   // [nsub,3] or null
  const int* nok;          // [nsub]
  SolverState st;
  // outputs (device arrays, global subint index)
  double* params; double* param_errs; double* nu_out; double* cov; double* chi2; double* red_chi2;
  double* snr; int* nfeval; int* rc; double* scales; double* scale_errs; double* channel_snrs;
  int s0, nchan, nbin, max_iter, semantics, fit_phi, fit_dm, is_toa;
  int model_steps;         // Newton steps taken on the local fourth-order model per pass (<= 1: one step per pass)
  double tol;              // one step per pass: convergence when the step is below tol sigma
  double tol_model;        // model steps: step and estimated truncation shift below tol_model sigma
  Box box;
  ModelRows mr;            // nu2, freqs of the subint's model
};

// C_n, dC_n/dtheta, d2C_n/dtheta2 at theta + t from the derivatives c[0..4] at theta
struct Tay4 { double C, C1, C2; };
__device__ __forceinline__ Tay4 taylor4(const double* c, double t) {
  const double c0 = c[0], c1 = c[1], c2 = c[2], c3 = c[3], c4 = c[4];
  Tay4 y;
  y.C = c0 + t * (c1 + t * (0.5 * c2 + t * (c3 * (1.0 / 6.0) + t * c4 * (1.0 / 24.0))));
  y.C1 = c1 + t * (c2 + t * (0.5 * c3 + t * c4 * (1.0 / 6.0)));
  y.C2 = c2 + t * (c3 + t * 0.5 * c4);
  return y;
}

__global__ void __launch_bounds__(128) k_update2(UpdateArgs a) {
  const int s = a.s0 + blockIdx.x;
  if (a.st.done[s]) return;
  const int mb = a.mr.row0(s);   // the subint's model
  __shared__ double sh[8 * 4];
  const int tid = threadIdx.x;
  const int nchan = a.nchan;
  const double* cs = a.csum + (size_t)s * nchan * kNCsum;
  const double* Sv = a.Ssn + (size_t)s * nchan;
  const double P = a.P[s];
  const double nf = a.nu_fit[(size_t)s * 3];
  const double nf2 = 1.0 / (nf * nf);
  const double KP = kDconst / P;

  double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // f, g0, g1, h00, h01, h11, gmax(unused), Sd
  double gmax = 0.0;
  for (int n = tid; n < nchan; n += 128) {
    const double S = Sv[n];
    if (!(S > 0.0)) continue;
    const double C = cs[n * kNCsum], C1 = cs[n * kNCsum + 1], C2 = cs[n * kNCsum + 2];
    const double g = KP * (a.nu2[mb + n] - nf2);
    const double t = -2.0 * C * C1 / S;            // pplib.py:1348-1349
    const double W = (C1 * C1 + C * C2) / S;       // pplib.py:1385-1386
    v[0] -= C * C / S;
    v[1] += t; v[2] += t * g;
    v[3] -= 2.0 * W; v[4] -= 2.0 * W * g; v[5] -= 2.0 * W * g * g;
    v[7] += a.Sdn[(size_t)s * nchan + n];
    gmax = fmax(gmax, fabs(g));
  }
  block_sum<8, 128>(v, sh);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) gmax = fmax(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
  __syncthreads();
  if ((tid & 31) == 0) sh[tid >> 5] = gmax;
  __syncthreads();
  gmax = fmax(fmax(sh[0], sh[1]), fmax(sh[2], sh[3]));
  __syncthreads();

  double* x = a.st.x + (size_t)s * 5;
  double* xp = a.st.xprev + (size_t)s * 5;
  double* stp = a.st.step + (size_t)s * 5;
  // ---- safeguarded Newton.  Every thread holds the same sums and takes the same decisions;
  // thread 0 writes the state.  The per-channel derivatives up to the fourth order (k_pass2) give a
  // local model C_n(theta_n + t) of the objective; the Newton iteration runs on that model
  // (a few reductions over nchan numbers) instead of costing one pass over X per step, and the
  // fit finishes without another pass when the model's truncation error at the point reached is
  // far below the tolerance.  Otherwise the point reached is evaluated by the next pass.
  const int it = a.st.iter[s] + 1;
  const double f = v[0];
  const double fprev = a.st.fprev[s], lam_prev = a.st.lam[s];
  const double x0 = x[0], x1 = x[1], xp0 = xp[0], xp1 = xp[1], stp0 = stp[0], stp1 = stp[1];
  __syncthreads();                       // all reads of the state precede thread 0's writes
  int finish = 0, rc = 0;
  double d0 = 0.0, d1 = 0.0;             // displacement applied on top of the evaluated point
  if (!(f == f) || fabs(f) > 1e300) { finish = 1; rc = 3; }
  else if (a.max_iter < 0) { finish = 2; rc = 0; }   // evaluate-only (get_scales)
  else if (it > 1 && f > fprev + 1e-12 * fabs(fprev)) {
    // uphill: shrink the previous step and re-evaluate
    const double lam = lam_prev * 0.25;
    if (it >= a.max_iter || lam < 1e-6) { finish = 2; rc = 1; }  // give up: report this point
    if (tid == 0) {
      a.st.lam[s] = lam;
      if (!finish) { x[0] = xp0 + lam * stp0; x[1] = xp1 + lam * stp1; }
    }
  } else {
    double m[6] = {v[0], v[1], v[2], v[3], v[4], v[5]};   // f, g0, g1, h00, h01, h11 at x + (d0, d1)
    bool conv = false, clipped = false, pd = true, free0 = true, free1 = true;
    double sg0 = 0.0, sg1 = 0.0, cv01 = 0.0;
    const int n_inner = a.model_steps > 0 ? a.model_steps : 1;
    for (int inner = 0; inner < n_inner; ++inner) {
      if (inner > 0) {
        for (int i = 0; i < 6; ++i) m[i] = 0.0;
        for (int n = tid; n < nchan; n += 128) {
          const double S = Sv[n];
          if (!(S > 0.0)) continue;
          const double g = KP * (a.nu2[mb + n] - nf2);
          const Tay4 y = taylor4(cs + n * kNCsum, d0 + d1 * g);
          const double t = -2.0 * y.C * y.C1 / S;
          const double W = (y.C1 * y.C1 + y.C * y.C2) / S;
          m[0] -= y.C * y.C / S;
          m[1] += t; m[2] += t * g;
          m[3] -= 2.0 * W; m[4] -= 2.0 * W * g; m[5] -= 2.0 * W * g * g;
        }
        block_sum<6, 128>(m, sh);
        __syncthreads();
      }
      double h00 = m[3], h01 = m[4], h11 = m[5], g0 = m[1], g1 = m[2];
      free0 = a.fit_phi && !box_holds(a.box, 0, x0 + d0, g0);
      free1 = a.fit_dm && !box_holds(a.box, 1, x1 + d1, g1);
      if (!free1) { h01 = 0.0; h11 = 1.0; g1 = 0.0; }
      if (!free0) { h01 = 0.0; h00 = 1.0; g0 = 0.0; }
      const double det = h00 * h11 - h01 * h01;
      pd = h00 > 0.0 && h11 > 0.0 && det > 1e-14 * h00 * h11;
      double e0, e1;
      if (pd) {
        e0 = -(h11 * g0 - h01 * g1) / det;
        e1 = -(-h01 * g0 + h00 * g1) / det;
      } else if (inner == 0) {  // not convex here: scaled steepest descent
        e0 = -g0 / (fabs(h00) + 1e-300);
        e1 = -g1 / (fabs(h11) + 1e-300);
      } else break;             // the model left the convex region: evaluate where we are
      // keep every channel's rotation change below 0.1 turn per pass
      const double big = fmax(fabs(d0 + e0), fabs(d1 + e1) * gmax);
      bool limited = false;
      if (big > 0.1) {
        const double bstep = fmax(fabs(e0), fabs(e1) * gmax);
        if (inner == 0) { e0 *= 0.1 / bstep; e1 *= 0.1 / bstep; }
        else { e0 = 0.0; e1 = 0.0; }
        limited = true;
      }
      clipped = false;
      const double xn0 = box_clip(a.box, 0, x0 + d0 + e0, clipped), xn1 = box_clip(a.box, 1, x1 + d1 + e1, clipped);
      if (clipped) { e0 = xn0 - (x0 + d0); e1 = xn1 - (x1 + d1); }
      d0 += e0; d1 += e1;
      if (!pd || limited) break;
      // 1-sigma from cov = inv(H/2) (pplib.py:2187-2190)
      sg0 = sqrt(2.0 * h11 / det); sg1 = sqrt(2.0 * h00 / det); cv01 = -2.0 * h01 / det;
      const double tol_step = n_inner > 1 ? a.tol_model : a.tol;
      if (!clipped && (fabs(e0) <= tol_step * sg0 || !free0) && (fabs(e1) <= tol_step * sg1 || !free1)) { conv = true; break; }
    }
    if (conv && n_inner > 1) {
      // ---- is the model good enough at (d0, d1)?  The first neglected term of the gradient series
      // is estimated from the last one kept, c4 t^3/6, times r t/4 with r^2 = sum|c4| / sum|c2|
      // (~ (2 pi k_eff)^2); likewise for the objective.  Required: parameter shifts below
      // tol_model sigma, an objective error below 1e-9 |f| and a curvature error below 1e-5.
      double q[6] = {0, 0, 0, 0, 0, 0};   // sum|c2|, sum|c4|, gradient terms (phi, DM), objective term, Hessian term
      for (int n = tid; n < nchan; n += 128) {
        const double S = Sv[n];
        if (!(S > 0.0)) continue;
        const double* c = cs + n * kNCsum;
        const double g = KP * (a.nu2[mb + n] - nf2);
        const double t = fabs(d0 + d1 * g);
        const double e = 2.0 * fabs(c[0]) * fabs(c[4]) * t * t * t / (6.0 * S);
        q[0] += fabs(c[2]); q[1] += fabs(c[4]); q[2] += e; q[3] += e * fabs(g); q[4] += e * t * 0.25;
        q[5] += fabs(c[0]) * fabs(c[4]) * t * t / S;
      }
      block_sum<6, 128>(q, sh);
      __syncthreads();
      const double r = sqrt(q[1] / fmax(q[0], 1e-300));
      const double rt = r * (fabs(d0) + fabs(d1) * gmax);
      const double eg0 = free0 ? q[2] * rt * 0.25 : 0.0, eg1 = free1 ? q[3] * rt * 0.25 : 0.0;
      const double err0 = 0.5 * (sg0 * sg0 * eg0 + fabs(cv01) * eg1), err1 = 0.5 * (fabs(cv01) * eg0 + sg1 * sg1 * eg1);
      const bool good = rt < 0.5 && (err0 <= a.tol_model * sg0 || !free0) && (err1 <= a.tol_model * sg1 || !free1) &&
                        q[4] * rt * 0.2 <= 1e-9 * fabs(m[0]) &&
                        q[5] * rt * (1.0 / 3.0) <= 1e-5 * fabs(m[3]);   // curvature (error bars) to 1e-5
      if (!good) conv = false;
    }
    if (conv) { finish = 1; rc = 0; }
    else if (it >= a.max_iter) { finish = 2; rc = 1; }   // out of passes: report the evaluated point as it is
    if (tid == 0) {
      xp[0] = x0; xp[1] = x1;
      stp[0] = d0; stp[1] = d1;
      a.st.fprev[s] = f;
      a.st.lam[s] = 1.0;
      if (!finish) { x[0] = x0 + d0; x[1] = x1 + d1; }
    }
  }
  if (tid == 0) a.st.iter[s] = it;
  if (!finish) return;
  // ---- epilogue: sums are at x, the final point is x + (d0, d1) --------------------
  // finish == 2: back-tracking gave up, report the evaluated point without a step.
  if (finish != 1 || rc == 3) { d0 = 0.0; d1 = 0.0; }
  const double phi_fit = x0 + d0, DM_fit = x1 + d1;
  // the per-channel sums at the final point from their Taylor series
  double u[4] = {0, 0, 0, 0};  // f, sumW, sumW nu^-2, snr^2
  for (int n = tid; n < nchan; n += 128) {
    const double S = Sv[n];
    if (!(S > 0.0)) continue;
    const double g = KP * (a.nu2[mb + n] - nf2);
    const Tay4 y = taylor4(cs + n * kNCsum, d0 + d1 * g);
    const double W = (y.C1 * y.C1 + y.C * y.C2) / S;
    u[0] -= y.C * y.C / S;
    u[1] += W; u[2] += W * a.nu2[mb + n];
    u[3] += y.C * y.C / S;
  }
  block_sum<4, 128>(u, sh);
  __syncthreads();
  const double fmin = u[0];
  // zero-covariance frequency (pplib.py:1390; pptoaslib.py:746-752)
  double nu_zero = nf;
  if (a.fit_phi && a.fit_dm) nu_zero = sqrt(u[1] / u[2]);
  double nu_o = a.nu_outs ? a.nu_outs[(size_t)s * 3] : CUDART_NAN;
  if (!(nu_o == nu_o)) nu_o = nu_zero;
  const double no2 = 1.0 / (nu_o * nu_o);
  double hh[3] = {0, 0, 0};
  for (int n = tid; n < nchan; n += 128) {
    const double S = Sv[n];
    if (!(S > 0.0)) continue;
    const double g = KP * (a.nu2[mb + n] - nf2);
    const Tay4 y = taylor4(cs + n * kNCsum, d0 + d1 * g);
    const double W = (y.C1 * y.C1 + y.C * y.C2) / S;
    const double go = KP * (a.nu2[mb + n] - no2);
    hh[0] -= 2.0 * W; hh[1] -= 2.0 * W * go; hh[2] -= 2.0 * W * go * go;
  }
  block_sum<3, 128>(hh, sh);
  double h00 = hh[0], h01 = hh[1], h11 = hh[2];
  if (!a.fit_dm) { h01 = 0.0; h11 = 1.0; }
  if (!a.fit_phi) { h01 = 0.0; h00 = 1.0; }
  const double det = h00 * h11 - h01 * h01;
  // covariance = inv(H/2) = 2 inv(H)
  double c00 = 2.0 * h11 / det, c01 = -2.0 * h01 / det, c11 = 2.0 * h00 / det;
  if (!a.fit_dm) { c11 = 0.0; c01 = 0.0; }
  if (!a.fit_phi) { c00 = 0.0; c01 = 0.0; }
  const int nok = a.nok[s];
  const int nfit = (a.fit_phi ? 1 : 0) + (a.fit_dm ? 1 : 0);
  const double chi2 = v[7] + fmin;
  const double dof = (double)nok * a.nbin - (double)(nfit + nok);
  // per-channel outputs
  for (int n = tid; n < nchan; n += 128) {
    const double S = Sv[n];
    const size_t o = (size_t)s * nchan + n;
    double sc = 0.0, se = 0.0, csn = 0.0;
    if (S > 0.0) {
      const double g = KP * (a.nu2[mb + n] - nf2);
      const Tay4 y = taylor4(cs + n * kNCsum, d0 + d1 * g);
      const double C = y.C, C1 = y.C1;
      sc = C / S;                                         // pptoaslib.py:688
      csn = sc * sqrt(S);                                 // pptoaslib.py:1081
      if (a.semantics == 1) se = 1.0 / sqrt(S);           // pplib.py:2197
      else {
        // diag(2 LR), LR = Cinv + Cinv V Xinv U Cinv (pptoaslib.py:713-724)
        const double go = KP * (a.nu2[mb + n] - no2);
        const double U0 = a.fit_phi ? -2.0 * C1 : 0.0, U1 = a.fit_dm ? -2.0 * C1 * go : 0.0;
        // Xinv = inv(H_out) = cov/2
        const double q = 0.5 * (U0 * U0 * c00 + 2.0 * U0 * U1 * c01 + U1 * U1 * c11);
        se = sqrt(1.0 / S + q / (2.0 * S * S));
      }
    }
    if (a.scales) a.scales[o] = sc;
    if (a.scale_errs) a.scale_errs[o] = se;
    if (a.channel_snrs) a.channel_snrs[o] = csn;
  }
  if (tid == 0) {
    // phi at the output frequency (pplib.py:2182; pptoaslib.py:1052-1057)
    double phi_out = phi_fit + KP * DM_fit * (no2 - nf2);
    phi_out = wrap_phase(phi_out);
    double* po = a.params + (size_t)s * 5;
    po[0] = phi_out; po[1] = DM_fit; po[2] = x[2]; po[3] = x[3]; po[4] = x[4];
    double* pe = a.param_errs + (size_t)s * 5;
    pe[0] = sqrt(c00); pe[1] = sqrt(c11); pe[2] = 0; pe[3] = 0; pe[4] = 0;
    double* cv = a.cov + (size_t)s * 25;
    for (int i = 0; i < 25; ++i) cv[i] = 0.0;
    cv[0] = c00; cv[1] = c01; cv[5] = c01; cv[6] = c11;
    double* no = a.nu_out + (size_t)s * 3;
    no[0] = nu_o;
    no[1] = (a.is_toa && a.fit_dm) ? nu_o : a.nu_fit[(size_t)s * 3 + 1];   // pptoaslib.py:1048-1050
    no[2] = a.nu_fit[(size_t)s * 3 + 2];
    a.chi2[s] = chi2;
    a.red_chi2[s] = chi2 / dof;
    a.snr[s] = sqrt(u[3]);
    a.nfeval[s] = it;
    a.rc[s] = rc;
    x[0] = phi_fit; x[1] = DM_fit;
    a.st.done[s] = 1;
  }
}

// state initialisation when the caller supplies init params (no FFTFIT guess)
__global__ void k_init_state(SolverState st, const double* init, int s0, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = s0 + i;
  for (int q = 0; q < 5; ++q) {
    const double v = init ? init[(size_t)s * 5 + q] : 0.0;
    st.x[(size_t)s * 5 + q] = v; st.xprev[(size_t)s * 5 + q] = v; st.step[(size_t)s * 5 + q] = 0.0;
  }
  st.fprev[s] = 0.0; st.lam[s] = 1.0; st.iter[s] = 0; st.iterc[s] = 0; st.done[s] = 0;
}

// number of subints of [s0, s0+n) that are not finished yet
__global__ void k_count_running(SolverState st, int s0, int n, int* out) {
  __shared__ int cnt;
  if (threadIdx.x == 0) cnt = 0;
  __syncthreads();
  int c = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) c += (st.done[s0 + i] != 1);
  atomicAdd(&cnt, c);
  __syncthreads();
  if (threadIdx.x == 0) *out = cnt;
}

__global__ void k_reset_state(SolverState st, int s0, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = s0 + i;
  for (int q = 0; q < 5; ++q) { st.xprev[(size_t)s * 5 + q] = st.x[(size_t)s * 5 + q]; st.step[(size_t)s * 5 + q] = 0.0; }
  st.fprev[s] = 0.0; st.lam[s] = 1.0; st.iter[s] = 0; st.iterc[s] = 0; st.done[s] = 0;
}

// Coarse level of the general fit with several models: a running subint whose model has no such level (nj[model]
// = 0) waits in state kSitsOut, untouched by the level's kernels (on = 1), and runs again afterwards (on = 0).
constexpr int kSitsOut = 4;
__global__ void k_coarse_sitout(SolverState st, ModelRows mr, const int* nj, int s0, int n, int on) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = s0 + i;
  if (on) { if (st.done[s] == 0 && nj[mr.of(s)] == 0) st.done[s] = kSitsOut; }
  else if (st.done[s] == kSitsOut) st.done[s] = 0;
}

// end of the coarse stage of the general fit: every unfinished subint starts the full-resolution Newton
// iterations from where the coarse ones left it (the objective changes: no comparison with the old value)
__global__ void k_coarse_end(SolverState st, int s0, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = s0 + i;
  if (st.done[s] == 1 || st.done[s] == kSitsOut) return;
  st.done[s] = 0;
  st.fprev[s] = CUDART_INF;
  st.lam[s] = 1.0;
  for (int q = 0; q < 5; ++q) { st.xprev[(size_t)s * 5 + q] = st.x[(size_t)s * 5 + q]; st.step[(size_t)s * 5 + q] = 0.0; }
}

// number of subints of [s0, s0+n) still in the coarse stage
__global__ void k_count_coarse(SolverState st, int s0, int n, int* out) {
  __shared__ int cnt;
  if (threadIdx.x == 0) cnt = 0;
  __syncthreads();
  int c = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) c += (st.done[s0 + i] == 0);
  atomicAdd(&cnt, c);
  __syncthreads();
  if (threadIdx.x == 0) *out = cnt;
}

// Harmonic cut-off of a model channel: the objective sees the data only through X_nk = d_nk conj(m_nk), so the
// harmonics where the model has no power carry nothing.  njn[n] = the leading groups of 16 harmonics outside which
// the information-weighted model power, sum k^2 |m_nk|^2, is below eps2 (1e-20) of its total: by Cauchy-Schwarz the
// neglected part of C_n is below 1e-10 ||d_n|| ||m_n||, i.e. chi^2 moves by < 2e-10 relative and the parameters by
// ~1e-9 sigma (DESIGN 4).  Smooth templates (Gaussian / spline models) keep a fraction of the harmonics; a template
// with a noise floor keeps them all (njn = N/16, which also keeps the Nyquist term).  One CTA per channel.
__global__ void __launch_bounds__(256) k_model_cutoff(const double* mpow, int* njn, int N, int kj_min, double eps2) {
  __shared__ double grp[129];   // per group of 16 harmonics; [NJ] = the Nyquist term
  const int n = blockIdx.x, NJ = N / 16;
  const double* m = mpow + (size_t)n * N;
  for (int j = threadIdx.x; j <= NJ; j += blockDim.x) {
    double v = 0.0;
    if (j < NJ) {
      for (int q = 0; q < 16; ++q) { const int k = 16 * j + q; if (k > 0) v += (double)k * (double)k * m[k]; }
    } else v = (double)N * (double)N * m[0];
    grp[j] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int j = 0; j <= NJ; ++j) tot += grp[j];
    int keep = NJ;
    if (tot > 0.0 && tot < CUDART_INF) {
      double tail = grp[NJ];                       // dropping any group drops the Nyquist term as well
      while (keep > kj_min && tail + grp[keep - 1] <= eps2 * tot) { tail += grp[keep - 1]; --keep; }
      if (!(tail <= eps2 * tot)) keep = NJ;        // the Nyquist term alone is too much: keep everything
    }
    njn[n] = keep;
  }
}

// Where the phase information of the (scattered) model sits, per group of 16 harmonics:
//   info[j] = sum_n sum_{16 j <= k < 16 (j+1)} k^2 |m_nk|^2 |B_nk|^2,  |B_nk|^2 = 1 / (1 + (2 pi k tau_n)^2)
// with tau_n from the start values of subint s (x = null: no scattering).  The host accumulates the groups and
// takes the leading ones that hold coarse_frac of the total as the coarse objective of the general solver
// (the Nyquist term is left out).  grid.y: one model each, from its subint first[y] (global index: x, nu_fit and
// info [gridDim.y, N/16] then start at subint 0); first null: one model, x and nu_fit at subint s.
__global__ void k_model_info(const double* mpow, const double* lgf, const double* x, const double* nu_fit, int log10_tau,
                             double* info, int nchan, int N, ModelRows mr, const int* first) {
  const int j = blockIdx.x;
  if (first) {
    const int s = first[blockIdx.y];
    const size_t r = mr.row0(s);
    mpow += r * N; lgf += r;
    if (x) x += (size_t)s * 5;
    nu_fit += (size_t)s * 3;
    info += (size_t)blockIdx.y * (N / 16);
  }
  double tau = 0.0, alpha = 0.0, lg2nT = 0.0;
  if (x) {
    tau = log10_tau ? exp2(x[3] * 3.3219280948873623479) : x[3];
    alpha = x[4];
    lg2nT = log2(nu_fit[2]);
  }
  double v = 0.0;
  for (int n = threadIdx.x; n < nchan; n += blockDim.x) {
    const double wt = tau != 0.0 ? kTwoPi * tau * exp2(alpha * (lgf[n] - lg2nT)) : 0.0;
    const double* m = mpow + (size_t)n * N + j * 16;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int k = j * 16 + q;
      if (k == 0) continue;     // slot 0 holds the Nyquist harmonic
      const double b = (double)k * wt;
      v += (double)k * (double)k * m[q] / fma(b, b, 1.0);
    }
  }
  __shared__ double sh[32];
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) t += sh[q];
    info[j] = t;
  }
}

// start values are moved into the box, as scipy's TNC does with x0
__global__ void k_clamp_state(SolverState st, Box box, int s0, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int s = s0 + i;
  for (int q = 0; q < 5; ++q) {
    bool c = false;
    const double v = box_clip(box, q, st.x[(size_t)s * 5 + q], c);
    if (c) { st.x[(size_t)s * 5 + q] = v; st.xprev[(size_t)s * 5 + q] = v; }
  }
}

// ----------------------------------------------------------------------------
// k_pass5: K3 for (phi, DM, GM, tau, alpha) -- pptoaslib.py:181-523.
// Per channel the nine primitive sums with respect to (theta_n, tau_n):
//   C, C_th, C_thth, C_t, C_tt, C_tht  (Cdbp* family, 424-523)
//   S, S_t, S_tt                        (Sbp* family, 390-422)
// with B_nk = 1/(1 + i w tau_n), w = 2 pi k (pplib.py:4080-4095),
// dB/dtau_n = -i w B^2, d2B/dtau_n^2 = -2 w^2 B^3 (== B(B-1)/tau_n, 2B(B-1)^2/tau_n^2;
// pptoaslib.py:318-356).  Same lane mapping as k_pass2.
// ----------------------------------------------------------------------------
struct Pass5Args {
  const float2* X;         // [chunk,nchan,N]
  const float2* Xlo;       // [chunk,nchan,LoK<N>]
  const double* mpow;      // [nchan,N] |m|^2 (slot layout, double: S_n must not carry float rounding)
  const double* nu2;       // [nchan]
  const double* freqs;     // [nchan]
  const double* lgf;       // [nchan] log2(freqs)
  const double* P;         // [nsub]
  const double* nu_fit;    // [nsub,3]
  const double* Ssn;       // [nsub,nchan] (0 => unused channel)
  const double* sigma;     // [nsub,nchan]
  double* csum;            // [nsub,nchan,kNCsum]
  SolverState st;
  int s0, nchan, log10_tau;
  int nhalf;               // true nbin/2 (0: N)
  int nj;                  // groups of 16 harmonics summed: N/16 = all of them; fewer = the coarse objective, which
                           // also leaves the Nyquist term out and skips subints already coarse-converged (done == 3)
  int cstride;             // coarse objective: every cstride-th channel only (1: all)
  const int* njn;          // [nchan] groups of 16 harmonics where the model has power (k_model_cutoff)
  ModelRows mr;            // mpow, nu2, freqs, lgf, njn of the subint's model
  const int* njm;          // [nmodel] coarse level with several models: its groups per model (then nj = 0), or null
};

// k_pass5 keeps D iterations of loads (X row piece + |m|^2 piece, 16 bytes each per thread) in flight through a
// thread-private ring in shared memory: the kernel is FP64-bound with 128 registers per thread and 16 warps per SM,
// too few to cover the load latency from registers.
template <int N> struct Pass5Ring {
  static constexpr int NJ = N / 16;
  static constexpr int D = NJ < 8 ? NJ : 8;
  static constexpr int KJ = LoK<N>::value / 16;
  static constexpr size_t kBytes = sizeof(float4) * 256 * (2 * D + KJ);
  static constexpr int kMinBlocks = 2;   // CTAs per SM asked of the compiler
};

template <int N>
__global__ void __launch_bounds__(256, Pass5Ring<N>::kMinBlocks) k_pass5(Pass5Args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int sl = blockIdx.y, s = a.s0 + sl;
  constexpr int NJ = N / 16;
  const bool coarse = a.nj < NJ;
  {
    const int dn = a.st.done[s];
    if (dn == 1 || (coarse && dn >= 3)) return;
  }
  const int m = a.mr.of(s), mb = m * a.nchan;   // the subint's model
  const int lvnj = a.njm ? __ldg(a.njm + m) : a.nj;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int sub = lane >> 3, l8 = lane & 7;
  const int ch = (blockIdx.x * 32 + w * 4 + sub) * a.cstride;
  const bool inrange = ch < a.nchan;
  const int chc = inrange ? ch : a.nchan - 1;
  const bool used = inrange && a.Ssn[(size_t)s * a.nchan + chc] > 0.0;

  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  double taun = 0.0;
  if (used) {
    using R = Pass5Ring<N>;
    constexpr int D = R::D, KJ = R::KJ;
    float4* rv = reinterpret_cast<float4*>(smem_raw) + tid;   // [D][256] X pieces
    float4* rm = rv + D * 256;                                 // [D][256] |m|^2 pieces (double2)
    float4* rl = rm + D * 256;                                 // [KJ][256] float32 residuals of the low harmonics
    const float4* row = reinterpret_cast<const float4*>(a.X + ((size_t)sl * a.nchan + ch) * N) + l8;
    const float4* mrow = reinterpret_cast<const float4*>(a.mpow + (size_t)(mb + ch) * N) + l8;
    const float4* lorow = reinterpret_cast<const float4*>(a.Xlo + ((size_t)sl * a.nchan + ch) * LoK<N>::value) + l8;
    const int nj = min(lvnj, a.njn[mb + ch]);   // harmonics the model has power in (>= KJ groups), fewer on a coarse level
    auto issue = [&](int j) {            // one commit group per iteration, empty past the end
      if (j < nj) {
        cp_async16(rv + (j % D) * 256, row + j * 8);
        cp_async16(rm + (j % D) * 256, mrow + j * 8);
      }
      cp_async_commit();
    };
    // the first loads go out before the phasor set-up
#pragma unroll
    for (int j = 0; j < KJ; ++j) cp_async16(rl + j * 256, lorow + j * 8);
#pragma unroll
    for (int j = 0; j < D - 1; ++j) issue(j);

    const double* x = a.st.x + (size_t)s * 5;
    const double P = a.P[s];
    const double nD = a.nu_fit[(size_t)s * 3 + 0], nG = a.nu_fit[(size_t)s * 3 + 1], nT = a.nu_fit[(size_t)s * 3 + 2];
    const double n2 = a.nu2[mb + ch];
    const double gD = kDconst * (n2 - 1.0 / (nD * nD)) / P;                       // pptoaslib.py:206
    const double gG = kDconst * kDconst * (n2 * n2 - 1.0 / (nG * nG * nG * nG)) / P;  // :207
    double theta = x[0] + x[1] * gD + x[2] * gG;
    theta -= rint(theta);
    // tau_n = tau (nu_n/nu_tau)^alpha (pplib.py:4049-4053) as one exp2: log2(nu_n) is tabulated
    {
      const double lr = x[4] * (a.lgf[mb + ch] - log2(nT));
      taun = a.log10_tau ? exp2(fma(x[3], 3.3219280948873623479, lr)) : x[3] * exp2(lr);
    }
    // phasors for k = 2 l8, 2 l8 + 1 and the step 16 from one sincospi by repeated squaring (as k_pass2)
    double c0, s0, c1, s1, cw, sw;
    cx<double> e1, e2, e4, e8, e16;
    cis2pi(theta, e1.x, e1.y);
    e2 = csqr(e1); e4 = csqr(e2); e8 = csqr(e4); e16 = csqr(e8);
    {
      cx<double> z = mk<double>(1.0, 0.0);
      if (l8 & 1) z = e2;
      if (l8 & 2) z = cmul(z, e4);
      if (l8 & 4) z = cmul(z, e8);
      c0 = z.x; s0 = z.y;
      const cx<double> z1 = cmul(z, e1);
      c1 = z1.x; s1 = z1.y;
      cw = e16.x; sw = e16.y;
    }
    double k0 = (double)(2 * l8), k1 = (double)(2 * l8 + 1);
    const double wt = kTwoPi * taun;   // b = k * wt
    auto element = [&](double xr, double xi, double m, double c, double sn, double k) {
      const double zr = xr * c - xi * sn, zi = xr * sn + xi * c;      // X e^{i psi}
      const double b = k * wt;
      const double den = fma(b, b, 1.0);
      double q;                                                       // |B|^2 = 1/(1 + b^2)
      asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(q) : "d"(den));         // ~20 bits, then two Newton steps
      q = q * fma(-den, q, 2.0);
      q = q * fma(-den, q, 2.0);
      const double br = q, bi = b * q;                                // conj(B)
      const double a1r = zr * br - zi * bi, a1i = zr * bi + zi * br;  // Z conjB
      const double a2r = a1r * br - a1i * bi, a2i = a1r * bi + a1i * br;
      const double a3r = a2r * br - a2i * bi;
      const double k2 = k * k;
      acc[0] += a1r;
      acc[1] = fma(k, a1i, acc[1]);
      acc[2] = fma(k2, a1r, acc[2]);
      acc[3] = fma(k, a2i, acc[3]);
      acc[4] = fma(k2, a3r, acc[4]);
      acc[5] = fma(k2, a2r, acc[5]);
      const double qm = q * m;
      const double k2q2m = k2 * q * qm;
      acc[6] += qm;
      acc[7] += k2q2m;
      acc[8] = fma(k2q2m, fma(-4.0, q, 3.0), acc[8]);                 // 4 b^2 q - 1 = 3 - 4 q
    };
    auto advance = [&]() {
      const double t0 = c0 * cw - s0 * sw; s0 = c0 * sw + s0 * cw; c0 = t0;
      const double t1 = c1 * cw - s1 * sw; s1 = c1 * sw + s1 * cw; c1 = t1;
      k0 += 16.0; k1 += 16.0;
    };
    // iteration j: wait for its group, read its slot, refill the slot read one iteration ago
    auto fetch = [&](int j, float4& v, double2& mm) {
      cp_async_wait<(D >= 2 ? D - 2 : 0)>();
      v = rv[(j % D) * 256];
      mm = *reinterpret_cast<const double2*>(rm + (j % D) * 256);
      issue(j + D - 1);
    };
    // the first KJ iterations carry the float32 residuals of the low harmonics
#pragma unroll
    for (int j = 0; j < KJ; ++j) {
      float4 v; double2 mm;
      fetch(j, v, mm);
      const float4 lo = rl[j * 256];
      const bool z = (j == 0 && l8 == 0);
      element(z ? 0.0 : (double)v.x + (double)lo.x, z ? 0.0 : (double)v.y + (double)lo.y, z ? 0.0 : mm.x, c0, s0, k0);
      element((double)v.z + (double)lo.z, (double)v.w + (double)lo.w, mm.y, c1, s1, k1);
      advance();
    }
#pragma unroll 2
    for (int j = KJ; j < nj; ++j) {
      float4 v; double2 mm;
      fetch(j, v, mm);
      element((double)v.x, (double)v.y, mm.x, c0, s0, k0);
      element((double)v.z, (double)v.w, mm.y, c1, s1, k1);
      advance();
    }
    row -= l8; lorow -= l8;
    if (l8 == 0 && nj == NJ) {  // Nyquist harmonic k = N stored in slot 0
      const float2 xh = __ldg(reinterpret_cast<const float2*>(row));
      const float2 xl = __ldg(reinterpret_cast<const float2*>(lorow));
      const double mn = __ldg(a.mpow + (size_t)(mb + ch) * N);
      cx<double> en = e16;          // e^{2 pi i N theta} = (e^{2 pi i 16 theta})^(N/16)
#pragma unroll
      for (int q = 16; q < N; q *= 2) en = csqr(en);
      element((double)xh.x + (double)xl.x, (double)xh.y + (double)xl.y, mn, en.x, en.y, (double)N);
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  }
  if (inrange && l8 == 0) {
    double* o = a.csum + ((size_t)s * a.nchan + ch) * kNCsum;
    if (used) {
      const double sg = a.sigma[(size_t)s * a.nchan + ch];
      const double isF2 = 1.0 / (sg * sg * (double)(a.nhalf > 0 ? a.nhalf : N));
      const double p2 = kTwoPi * kTwoPi;
      o[0] = acc[0] * isF2;                        // C
      o[1] = -kTwoPi * acc[1] * isF2;              // C_th   = -sum w Im(A1)
      o[2] = -p2 * acc[2] * isF2;                  // C_thth = -sum w^2 Re(A1)
      o[3] = -kTwoPi * acc[3] * isF2;              // C_t    = -sum w Im(A2)
      o[4] = -2.0 * p2 * acc[4] * isF2;            // C_tt   = -2 sum w^2 Re(A3)
      o[5] = -p2 * acc[5] * isF2;                  // C_tht  = -sum w^2 Re(A2)
      o[6] = acc[6] * isF2;                        // S      = sum |B|^2 M
      o[7] = -2.0 * taun * p2 * acc[7] * isF2;     // S_t    = -2 tau_n sum w^2 q^2 M
      o[8] = 2.0 * p2 * acc[8] * isF2;             // S_tt   = sum 2 w^2 q^2 (4 b^2 q - 1) M
    } else {
#pragma unroll
      for (int i = 0; i < 9; ++i) o[i] = 0.0;
    }
  }
}

// ----------------------------------------------------------------------------
// small dense helpers for k_update5 (n <= 5, row-major 5x5 storage)
// ----------------------------------------------------------------------------
__device__ inline bool chol5(const double* A, int n, double* L) {
  for (int i = 0; i < n; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = A[i * 5 + j];
      for (int k = 0; k < j; ++k) s -= L[i * 5 + k] * L[j * 5 + k];
      if (i == j) {
        if (!(s > 0.0)) return false;
        L[i * 5 + i] = sqrt(s);
      } else L[i * 5 + j] = s / L[j * 5 + j];
    }
  return true;
}
__device__ inline void chol5_solve(const double* L, int n, const double* b, double* x) {
  double y[5];
  for (int i = 0; i < n; ++i) {
    double s = b[i];
    for (int k = 0; k < i; ++k) s -= L[i * 5 + k] * y[k];
    y[i] = s / L[i * 5 + i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double s = y[i];
    for (int k = i + 1; k < n; ++k) s -= L[k * 5 + i] * x[k];
    x[i] = s / L[i * 5 + i];
  }
}
__device__ inline void chol5_inverse(const double* L, int n, double* Inv) {
  for (int c = 0; c < n; ++c) {
    double e[5] = {0, 0, 0, 0, 0}, x[5];
    e[c] = 1.0;
    chol5_solve(L, n, e, x);
    for (int r = 0; r < n; ++r) Inv[r * 5 + c] = x[r];
  }
}

// Real positive roots of sum_i c[i] x^(deg-i) (np.roots convention), Aberth iteration in
// complex double; returns the count written to out[].
// Eigen-decomposition of a symmetric n x n matrix (n <= 5, row stride 5) by cyclic Jacobi rotations:
// A = V diag(w) V^T (V column k = eigenvector k).  Used where the Hessian is not positive definite.
__device__ inline void sym_eig5(const double* A_in, int n, double* V, double* w) {
  double A[25];
  for (int i = 0; i < n; ++i) for (int k = 0; k < n; ++k) { A[i * 5 + k] = A_in[i * 5 + k]; V[i * 5 + k] = (i == k) ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 12; ++sweep) {
    double off = 0.0, dg = 0.0;
    for (int i = 0; i < n; ++i) { dg += A[i * 5 + i] * A[i * 5 + i]; for (int k = i + 1; k < n; ++k) off += A[i * 5 + k] * A[i * 5 + k]; }
    if (off <= 1e-30 * dg) break;
    for (int p = 0; p < n; ++p)
      for (int q = p + 1; q < n; ++q) {
        const double apq = A[p * 5 + q];
        if (apq == 0.0) continue;
        const double th = (A[q * 5 + q] - A[p * 5 + p]) / (2.0 * apq);
        const double t = (th >= 0.0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < n; ++k) {   // columns p, q
          const double akp = A[k * 5 + p], akq = A[k * 5 + q];
          A[k * 5 + p] = c * akp - sn * akq; A[k * 5 + q] = sn * akp + c * akq;
        }
        for (int k = 0; k < n; ++k) {   // rows p, q
          const double apk = A[p * 5 + k], aqk = A[q * 5 + k];
          A[p * 5 + k] = c * apk - sn * aqk; A[q * 5 + k] = sn * apk + c * aqk;
        }
        for (int k = 0; k < n; ++k) {
          const double vkp = V[k * 5 + p], vkq = V[k * 5 + q];
          V[k * 5 + p] = c * vkp - sn * vkq; V[k * 5 + q] = sn * vkp + c * vkq;
        }
      }
  }
  for (int i = 0; i < n; ++i) w[i] = A[i * 5 + i];
}

__device__ inline int real_pos_roots(const double* c_in, int deg_in, double* out) {
  double c[8];
  int deg = deg_in, off = 0;
  while (deg > 0 && c_in[off] == 0.0) { ++off; --deg; }   // strip leading zeros
  if (deg <= 0) return 0;
  for (int i = 0; i <= deg; ++i) c[i] = c_in[off + i] / c_in[off];
  double zr[8], zi[8];
  double rad = 0.0;
  for (int i = 1; i <= deg; ++i) rad = fmax(rad, pow(fabs(c[i]), 1.0 / i));
  rad = rad > 0 ? 2.0 * rad : 1.0;
  for (int i = 0; i < deg; ++i) { double sn, cs; sincospi(2.0 * (i + 0.35) / deg, &sn, &cs); zr[i] = 0.6 * rad * cs; zi[i] = 0.6 * rad * sn; }
  for (int it = 0; it < 200; ++it) {
    double change = 0.0;
    for (int i = 0; i < deg; ++i) {
      double pr = 1.0, pi = 0.0, dr = 0.0, di = 0.0;   // Horner p and p'
      for (int k = 1; k <= deg; ++k) {
        const double ndr = dr * zr[i] - di * zi[i] + pr, ndi = dr * zi[i] + di * zr[i] + pi;
        dr = ndr; di = ndi;
        const double npr = pr * zr[i] - pi * zi[i] + c[k], npi = pr * zi[i] + pi * zr[i];
        pr = npr; pi = npi;
      }
      const double dd = dr * dr + di * di;
      if (dd == 0.0) continue;
      double nr = (pr * dr + pi * di) / dd, ni = (pi * dr - pr * di) / dd;  // p/p'
      double sr = 0.0, si = 0.0;
      for (int j = 0; j < deg; ++j) if (j != i) {
        const double er = zr[i] - zr[j], ei = zi[i] - zi[j];
        const double e2 = er * er + ei * ei;
        if (e2 > 0) { sr += er / e2; si -= ei / e2; }
      }
      const double qr = 1.0 - (nr * sr - ni * si), qi = -(nr * si + ni * sr);
      const double q2 = qr * qr + qi * qi;
      if (q2 == 0.0) continue;
      const double wr = (nr * qr + ni * qi) / q2, wi = (ni * qr - nr * qi) / q2;
      zr[i] -= wr; zi[i] -= wi;
      change = fmax(change, fabs(wr) + fabs(wi));
    }
    if (change < 1e-15 * rad) break;
  }
  int n = 0;
  for (int i = 0; i < deg; ++i)
    if (fabs(zi[i]) <= 1e-9 * fabs(zr[i]) && zr[i] > 0.0) out[n++] = zr[i];
  return n;
}

// ----------------------------------------------------------------------------
// k_update5: K3' for the general fit: chain rule to the five global parameters,
// gradient / Hessian (pptoaslib.py:544-643), safeguarded Newton on the fitted
// subset, and -- once converged and re-evaluated at the final point -- the
// epilogue: get_nu_zeros (733-906), re-referencing (1040-1065), covariance with
// the amplitude block (645-731 in closed form), scales, snr, chi2 (1069-1085).
// ----------------------------------------------------------------------------
struct Update5Args {
  const double* csum; const double* Sdn; const double* nu2; const double* freqs; const double* P;
  const double* lgf;       // [nchan] log2(freqs)
  const double* nu_fit; const double* nu_outs; const int* nok;
  SolverState st;
  double* params; double* param_errs; double* nu_out; double* cov; double* chi2; double* red_chi2;
  double* snr; int* nfeval; int* rc; double* scales; double* scale_errs; double* channel_snrs;
  int s0, nchan, nbin, max_iter, log10_tau, option, is_toa;
  int flags[5];
  int taylor_finish;   // finish a converged fit from the sums at the last evaluated point (no final pass)
  int cstride;         // coarse: the sums exist for every cstride-th channel only (else 1)
  int coarse;          // the sums are those of the low harmonics only (k_pass5 nj < N/16): Newton steps towards
                       // the start point of the full-resolution iterations, no epilogue; a subint whose step is
                       // <= ctol sigma waits in state done == 3
  double tol, ctol;
  Box box;
  ModelRows mr;        // nu2, freqs, lgf of the subint's model
};

// the per-channel sums c[0..8] = C, C_th, C_thth, C_t, C_tt, C_tht, S, S_t, S_tt carried from (theta_n, tau_n) to
// (theta_n + dth, tau_n + dta): values to second order, first derivatives to first order
__device__ __forceinline__ void chan_shift(double* c, double dth, double dta) {
  const double C = c[0] + c[1] * dth + c[3] * dta + 0.5 * (c[2] * dth * dth + 2.0 * c[5] * dth * dta + c[4] * dta * dta);
  const double Cth = c[1] + c[2] * dth + c[5] * dta;
  const double Ct = c[3] + c[5] * dth + c[4] * dta;
  const double S = c[6] + c[7] * dta + 0.5 * c[8] * dta * dta;
  const double St = c[7] + c[8] * dta;
  c[0] = C; c[1] = Cth; c[3] = Ct; c[6] = S; c[7] = St;
}

struct ChanJ {   // per-channel Jacobians of (theta_n, tau_n) w.r.t. the five parameters
  double Jth[3], Jt[2], Ktt, Kta, Kaa, lnf, taun;
};

// lg2r = log2(nu_n / nu_tau) from the tabulated log2(nu_n): tau_n is one exp2, as in k_pass5
__device__ __forceinline__ ChanJ chan_jac(double lg2r, double n2, double P, double nD, double nG, double tau_lin,
                                          double alpha, int log10_tau) {
  ChanJ j;
  j.Jth[0] = 1.0;
  j.Jth[1] = kDconst * (n2 - 1.0 / (nD * nD)) / P;                           // pptoaslib.py:222
  j.Jth[2] = kDconst * kDconst * (n2 * n2 - 1.0 / (nG * nG * nG * nG)) / P;  // :223
  j.lnf = lg2r * 0.69314718055994530942;
  j.taun = tau_lin * exp2(alpha * lg2r);
  const double ln10 = 2.302585092994045684;
  if (log10_tau) {                                                            // :246-274
    j.Jt[0] = ln10 * j.taun; j.Ktt = ln10 * j.Jt[0]; j.Kta = ln10 * j.lnf * j.taun;
  } else {
    j.Jt[0] = tau_lin != 0.0 ? j.taun / tau_lin : 0.0; j.Ktt = 0.0;
    j.Kta = tau_lin != 0.0 ? j.lnf * j.taun / tau_lin : 0.0;
  }
  j.Jt[1] = j.lnf * j.taun;
  j.Kaa = j.lnf * j.Jt[1];
  return j;
}

// first derivatives of C_n, S_n w.r.t. the five parameters
__device__ __forceinline__ void chan_first(const double* c, const ChanJ& j, double* dC, double* dS) {
  dC[0] = c[1] * j.Jth[0]; dC[1] = c[1] * j.Jth[1]; dC[2] = c[1] * j.Jth[2];
  dC[3] = c[3] * j.Jt[0]; dC[4] = c[3] * j.Jt[1];
  dS[0] = dS[1] = dS[2] = 0.0; dS[3] = c[7] * j.Jt[0]; dS[4] = c[7] * j.Jt[1];
}
__device__ __forceinline__ double chan_d2C(const double* c, const ChanJ& j, int a, int b) {
  if (a > b) { const int t = a; a = b; b = t; }
  if (b < 3) return c[2] * j.Jth[a] * j.Jth[b];
  if (a < 3) return c[5] * j.Jth[a] * j.Jt[b - 3];
  const double K = (a == 3 && b == 3) ? j.Ktt : ((a == 3) ? j.Kta : j.Kaa);
  return c[4] * j.Jt[a - 3] * j.Jt[b - 3] + c[3] * K;
}
__device__ __forceinline__ double chan_d2S(const double* c, const ChanJ& j, int a, int b) {
  if (a > b) { const int t = a; a = b; b = t; }
  if (a < 3) return 0.0;
  const double K = (a == 3 && b == 3) ? j.Ktt : ((a == 3) ? j.Kta : j.Kaa);
  return c[8] * j.Jt[a - 3] * j.Jt[b - 3] + c[7] * K;
}
// per-channel profile-likelihood Hessian entry (pptoaslib.py:624-628, written without 1/C)
__device__ __forceinline__ double chan_H(double C, double S, double d2C, double d2S, double dCa, double dCb, double dSa,
                                         double dSb) {
  const double iS = 1.0 / S;
  return -2.0 * (C * d2C * iS - 0.5 * C * C * d2S * iS * iS + dCa * dCb * iS + C * C * dSa * dSb * iS * iS * iS -
                 C * (dCa * dSb + dSa * dCb) * iS * iS);
}

// The same derivatives without the per-entry divisions: with r = C/S every gradient / Hessian entry of the
// channel's -C^2/S is one of five scalars times products of the Jacobians,
//   g_i = G1 Jth_i (i < 3), G2 Jt_i (i >= 3)
//   H_ik = A Jth_i Jth_k (i, k < 3), M Jth_i Jt_k (i < 3 <= k), T1 Jt_i Jt_k + G2 K_ik (i, k >= 3)
// (pptoaslib.py:572, 624-628 written out for dC_i = C_th Jth_i | C_t Jt_i, dS_i = 0 | S_t Jt_i).
struct ChanK { double f, G1, G2, A, M, T1, r; };
__device__ __forceinline__ ChanK chan_k(const double* c) {
  const double iS = 1.0 / c[6];
  const double r = c[0] * iS, r2 = r * r;
  const double e = c[3] - r * c[7];
  ChanK k;
  k.r = r;
  k.f = -c[0] * r;
  k.G1 = -2.0 * r * c[1];
  k.G2 = -2.0 * r * c[3] + r2 * c[7];
  k.A = -2.0 * (r * c[2] + c[1] * c[1] * iS);
  k.M = -2.0 * (r * c[5] + c[1] * iS * e);
  k.T1 = -2.0 * (r * c[4] - 0.5 * r2 * c[8] + iS * e * e);
  return k;
}
// adds the channel's Hessian (upper triangle, row-major: 00 01 02 03 04 11 12 13 14 22 23 24 33 34 44) to h
__device__ __forceinline__ void chan_hess(const ChanK& k, const ChanJ& j, double* h) {
  const double a1 = k.A * j.Jth[1], a2 = k.A * j.Jth[2];
  const double m0 = k.M * j.Jt[0], m1 = k.M * j.Jt[1];
  h[0] += k.A; h[1] += a1; h[2] += a2; h[3] += m0; h[4] += m1;
  h[5] = fma(a1, j.Jth[1], h[5]); h[6] = fma(a1, j.Jth[2], h[6]); h[7] = fma(m0, j.Jth[1], h[7]); h[8] = fma(m1, j.Jth[1], h[8]);
  h[9] = fma(a2, j.Jth[2], h[9]); h[10] = fma(m0, j.Jth[2], h[10]); h[11] = fma(m1, j.Jth[2], h[11]);
  const double t0 = k.T1 * j.Jt[0], t1 = k.T1 * j.Jt[1];
  h[12] += fma(t0, j.Jt[0], k.G2 * j.Ktt);
  h[13] += fma(t0, j.Jt[1], k.G2 * j.Kta);
  h[14] += fma(t1, j.Jt[1], k.G2 * j.Kaa);
}

template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) k_update5(Update5Args a) {
  const int s = a.s0 + blockIdx.x;
  const int state = a.st.done[s];
  if (state == 1 || state >= 3) return;   // finished, coarse-converged, or sitting a coarse level out
  const int mb = a.mr.row0(s);   // the subint's model
  __shared__ double sh[24 * (NT / 32)];
  __shared__ double bc[48];
  const int tid = threadIdx.x, nchan = a.nchan;
  const double* cs = a.csum + (size_t)s * nchan * kNCsum;
  const double P = a.P[s];
  const double nD = a.nu_fit[(size_t)s * 3], nG = a.nu_fit[(size_t)s * 3 + 1], nT = a.nu_fit[(size_t)s * 3 + 2];
  double* x = a.st.x + (size_t)s * 5;
  double* xp = a.st.xprev + (size_t)s * 5;
  double* stp = a.st.step + (size_t)s * 5;
  const double tau_lin = a.log10_tau ? pow(10.0, x[3]) : x[3];
  const double alpha = x[4];
  const double lg2nT = log2(nT);
  // The epilogue reports the point x + dx: dx = 0 when the sums in csum were evaluated at the
  // reported point (final pass), or the last (converged, <= tol sigma) Newton step, in which case
  // the per-channel sums are carried there by their second-order Taylor series (chan_shift) and the
  // final evaluation pass is saved.
  bool shifted = false;
  double dx[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  double tau_e = tau_lin, alpha_e = alpha;
  // mirror of the reference: with all tau_n == 0 the scattering derivatives are zero
  // (pptoaslib.py:325-330, 341-356)
  const bool scat_on = tau_lin != 0.0;
  int fl[5];
  int nfit = 0, idx[5];
  for (int i = 0; i < 5; ++i) { fl[i] = a.flags[i]; if (fl[i]) idx[nfit++] = i; }

  if (state == 0) {
    // ---- f, gradient, Hessian --------------------------------------------------------
    double v[23];
    for (int i = 0; i < 23; ++i) v[i] = 0.0;   // f, g[5], H upper [15], Sd, spare
    double gmax1 = -CUDART_INF, gmax2 = -CUDART_INF;   // max nu^-2, max -nu^-2
    const int cst = a.coarse ? a.cstride : 1;
    for (int n = tid * cst; n < nchan; n += NT * cst) {
      double c[9];
      for (int i = 0; i < 9; ++i) c[i] = cs[n * kNCsum + i];
      const double S = c[6];
      if (!(S > 0.0)) continue;
      if (!scat_on) { c[3] = c[4] = c[5] = c[7] = c[8] = 0.0; }
      const ChanJ j = chan_jac(a.lgf[mb + n] - lg2nT, a.nu2[mb + n], P, nD, nG, tau_lin, alpha, a.log10_tau);
      const ChanK k = chan_k(c);
      v[0] += k.f;
      v[1] += k.G1; v[2] = fma(k.G1, j.Jth[1], v[2]); v[3] = fma(k.G1, j.Jth[2], v[3]);   // :572
      v[4] = fma(k.G2, j.Jt[0], v[4]); v[5] = fma(k.G2, j.Jt[1], v[5]);
      chan_hess(k, j, v + 6);
      v[21] += a.Sdn[(size_t)s * nchan + n];
      gmax1 = fmax(gmax1, a.nu2[mb + n]);      // range of nu^-2 over the used channels (step limit below)
      gmax2 = fmax(gmax2, -a.nu2[mb + n]);
    }
    for (int i = 0; i < 5; ++i) v[1 + i] *= fl[i];
    {
      int q = 6;
      for (int i = 0; i < 5; ++i) for (int k = i; k < 5; ++k, ++q) v[q] *= fl[i] * fl[k];
    }
    block_sum<23, NT>(v, sh);
    double gm[2] = {gmax1, gmax2};
    for (int o = 16; o > 0; o >>= 1) { gm[0] = fmax(gm[0], __shfl_xor_sync(0xffffffffu, gm[0], o)); gm[1] = fmax(gm[1], __shfl_xor_sync(0xffffffffu, gm[1], o)); }
    __syncthreads();
    if ((tid & 31) == 0) { sh[tid >> 5] = gm[0]; sh[NT / 32 + (tid >> 5)] = gm[1]; }
    __syncthreads();
    gmax1 = gmax2 = -CUDART_INF;
#pragma unroll
    for (int q = 0; q < NT / 32; ++q) { gmax1 = fmax(gmax1, sh[q]); gmax2 = fmax(gmax2, sh[NT / 32 + q]); }
    if (tid == 0) {
      int it;
      if (a.coarse) { it = a.st.iterc[s] + 1; a.st.iterc[s] = it; }   // (the levels' objectives differ: fprev is reset between them)
      else { it = a.st.iter[s] + 1; a.st.iter[s] = it; }
      const double f = v[0];
      int action = 0;   // 0 continue, 1 go to final evaluation at x, 2 finish now (failure)
      int rc = 0;
      if (!(f == f) || fabs(f) > 1e300) { action = 2; rc = 3; }
      else if (a.max_iter < 0) { action = 3; rc = 0; }          // evaluate-only: epilogue at x now
      else if (it > 1 && f > a.st.fprev[s] + 1e-12 * fabs(a.st.fprev[s])) {
        const double lam = a.st.lam[s] * 0.25;
        a.st.lam[s] = lam;
        if (a.coarse) {   // the coarse stage only prepares a start point: give up early, at the best point seen
          if (lam < 1e-2) { for (int i = 0; i < 5; ++i) x[i] = xp[i]; a.st.done[s] = 3; }
          else for (int i = 0; i < 5; ++i) x[i] = xp[i] + lam * stp[i];
        }
        else if (it >= a.max_iter || lam < 1e-6) { action = 3; rc = 1; }
        else for (int i = 0; i < 5; ++i) x[i] = xp[i] + lam * stp[i];
      } else {
        double H[25], g[5], L[25], d[5] = {0, 0, 0, 0, 0}, dr[5];
        int q = 6;
        double Hf[25];
        for (int i = 0; i < 5; ++i) for (int k = i; k < 5; ++k, ++q) { Hf[i * 5 + k] = v[q]; Hf[k * 5 + i] = v[q]; }
        const int nfit_all = nfit;
        int idx_all[5];
        for (int i = 0; i < 5; ++i) idx_all[i] = idx[i];
        if (a.box.on) {   // active set: parameters held on a bound leave this step's system
          int nfree = 0;
          for (int i = 0; i < nfit; ++i) if (!box_holds(a.box, idx[i], x[idx[i]], v[1 + idx[i]])) idx[nfree++] = idx[i];
          nfit = nfree;
        }
        for (int i = 0; i < nfit; ++i) { g[i] = v[1 + idx[i]]; for (int k = 0; k < nfit; ++k) H[i * 5 + k] = Hf[idx[i] * 5 + idx[k]]; }
        bool pd = chol5(H, nfit, L);
        double Inv[25];
        if (pd) {
          double mg[5];
          for (int i = 0; i < nfit; ++i) mg[i] = -g[i];
          chol5_solve(L, nfit, mg, dr);
          chol5_inverse(L, nfit, Inv);
        } else {
          // Not convex here (a saddle or a flat valley of the tau / alpha / GM surface): Newton step on the
          // Hessian with its eigenvalues replaced by their moduli, in the coordinates scaled by the
          // diagonal (the parameters' natural scales differ by orders of magnitude, so an unscaled
          // Levenberg shift freezes the weakly constrained ones: 35 passes of crawling on a sigma = 1.5,
          // 32-channel, all-five-parameter golden).  Negative-curvature directions are descended at the
          // rate of their |curvature|; the objective-decrease test above backs a bad step off.
          double Dh[5], Hs[25], V[25], w[5], gs[5], y[5];
          for (int i = 0; i < nfit; ++i) { const double hd = fabs(H[i * 5 + i]); Dh[i] = hd > 0.0 ? 1.0 / sqrt(hd) : 1.0; }
          for (int i = 0; i < nfit; ++i) { gs[i] = g[i] * Dh[i]; for (int k = 0; k < nfit; ++k) Hs[i * 5 + k] = H[i * 5 + k] * Dh[i] * Dh[k]; }
          sym_eig5(Hs, nfit, V, w);
          for (int k = 0; k < nfit; ++k) {
            double pk = 0.0;
            for (int i = 0; i < nfit; ++i) pk += V[i * 5 + k] * gs[i];
            y[k] = -pk / fmax(fabs(w[k]), 1e-8);
          }
          for (int i = 0; i < nfit; ++i) {
            double di = 0.0;
            for (int k = 0; k < nfit; ++k) di += V[i * 5 + k] * y[k];
            dr[i] = di * Dh[i];
          }
        }
        for (int i = 0; i < nfit; ++i) d[idx[i]] = dr[i];
        // step limits: rotation of any channel <= 0.1 turn, log10(tau) <= 0.5, alpha <= 1,
        // linear tau: at most halve / grow by its own size
        double sc = 1.0;
        double rot;
        {
          // the rotation of channel n is the quadratic d0 + d1 K1 (nu_n^-2 - nu_D^-2) + d2 K2 (nu_n^-4 - nu_G^-4) in
          // nu_n^-2: its largest modulus over the band (DM and GM steps along their common valley nearly cancel,
          // the sum of the moduli would throttle them for many iterations)
          const double K1 = kDconst / P, K2 = kDconst * kDconst / P;
          const double q0 = d[0] - d[1] * K1 / (nD * nD) - d[2] * K2 / (nG * nG * nG * nG), q1 = d[1] * K1, q2 = d[2] * K2;
          const double lo = -gmax2, hi = gmax1;
          auto qv = [&](double t) { return fabs(fma(fma(q2, t, q1), t, q0)); };
          rot = fmax(qv(lo), qv(hi));
          if (q2 != 0.0) { const double tv = -0.5 * q1 / q2; if (tv > lo && tv < hi) rot = fmax(rot, qv(tv)); }
          if (!(rot == rot)) rot = CUDART_INF;
        }
        if (rot > 0.1) sc = fmin(sc, 0.1 / rot);
        if (a.log10_tau) { if (fabs(d[3]) > 0.5) sc = fmin(sc, 0.5 / fabs(d[3])); }
        else if (fl[3] && x[3] > 0.0 && fabs(d[3]) > 0.5 * x[3]) sc = fmin(sc, 0.5 * x[3] / fabs(d[3]));
        if (fabs(d[4]) > 1.0) sc = fmin(sc, 1.0 / fabs(d[4]));
        for (int i = 0; i < 5; ++i) d[i] *= sc;
        bool clipped = false;
        double xn[5];
        for (int i = 0; i < 5; ++i) xn[i] = box_clip(a.box, i, x[i] + d[i], clipped);
        if (clipped) for (int i = 0; i < 5; ++i) d[i] = xn[i] - x[i];
        bool conv = pd && sc == 1.0 && !clipped;
        bool tiny = conv;   // last step <= 0.1 tol sigma: the sums can be carried to the final point (chan_shift)
        bool cconv = conv;  // coarse stage: last step <= ctol sigma
        if (conv) for (int i = 0; i < nfit; ++i) {
          const double sg = sqrt(2.0 * Inv[i * 5 + i]);     // 1-sigma from inv(H/2)
          if (!(fabs(dr[i]) <= a.tol * sg)) conv = false;
          if (!(fabs(dr[i]) <= 0.1 * a.tol * sg)) tiny = false;
          if (!(fabs(dr[i]) <= a.ctol * sg)) cconv = false;
        }
        for (int i = 0; i < 5; ++i) { xp[i] = x[i]; stp[i] = d[i]; }
        a.st.fprev[s] = f;
        a.st.lam[s] = 1.0;
        for (int i = 0; i < 5; ++i) x[i] = xn[i];
        nfit = nfit_all;
        for (int i = 0; i < 5; ++i) idx[i] = idx_all[i];
        if (a.coarse) {   // no epilogue from the coarse sums: wait (state 3) for the full-resolution iterations
          if (cconv) a.st.done[s] = 3;
        }
        else if (conv && tiny && a.taylor_finish) {   // report x + d from the sums at x (no final pass)
          action = 4; rc = 0;
          for (int i = 0; i < 5; ++i) { bc[33 + i] = d[i]; bc[38 + i] = xn[i]; }
        }
        else if (conv) { action = 1; rc = 0; }
        else if (it >= a.max_iter) { action = 1; rc = 1; }
      }
      if (action == 1) a.st.done[s] = 2;   // one more pass at the final point, then the epilogue
      bc[0] = (double)action; bc[1] = (double)rc;
      if (action >= 1) a.rc[s] = rc;
      if (action == 2) {                    // non-finite objective: report what we have
        double* po = a.params + (size_t)s * 5;
        for (int i = 0; i < 5; ++i) po[i] = x[i];
        a.nfeval[s] = a.st.iter[s] + a.st.iterc[s]; a.st.done[s] = 1;
      }
    }
    __syncthreads();
    const int act = (int)bc[0];
    if (act != 3 && act != 4) return;   // 3: run the epilogue right now with the sums at x; 4: at x + d
    if (act == 4) {
      shifted = true;
      for (int i = 0; i < 5; ++i) dx[i] = bc[33 + i];
      tau_e = a.log10_tau ? pow(10.0, bc[38 + 3]) : bc[38 + 3];
      alpha_e = bc[38 + 4];
    }
  }
  // per-channel sums at the reported point
  auto load_c = [&](int n, double* c) {
    for (int i = 0; i < 9; ++i) c[i] = cs[n * kNCsum + i];
    if (!(c[6] > 0.0)) return;
    if (!scat_on) { c[3] = c[4] = c[5] = c[7] = c[8] = 0.0; }
    if (shifted) {
      const double n2 = a.nu2[mb + n];
      const double dth = dx[0] + dx[1] * (kDconst * (n2 - 1.0 / (nD * nD)) / P) +
                         dx[2] * (kDconst * kDconst * (n2 * n2 - 1.0 / (nG * nG * nG * nG)) / P);
      double dta = 0.0;
      if (scat_on) {
        const double lg2r = a.lgf[mb + n] - lg2nT;
        const double dl = (a.log10_tau ? 2.302585092994045684 * dx[3] : log1p(dx[3] / tau_lin)) + dx[4] * lg2r * 0.69314718055994530942;
        dta = tau_lin * exp2(alpha * lg2r) * expm1(dl);
      }
      chan_shift(c, dth, dta);
    }
  };

  // ======================= epilogue: sums in csum are at the final x =======================
  const double K1 = kDconst / P, K2 = kDconst * kDconst / P;
  // ---- get_nu_zeros (pptoaslib.py:733-906) at the fit reference frequencies ----------------
  int zfl[5];
  for (int i = 0; i < 5; ++i) zfl[i] = fl[i];
  if (fl[0] && fl[1] && fl[2] && fl[3] && fl[4]) zfl[2] = 0;      // [1,1,1,1,1] -> formulas of [1,1,0,1,1] (:893-901)
  double u[24];
  for (int i = 0; i < 24; ++i) u[i] = 0.0;
  // u[0..14]: for j=0..4: sum h_th(j), sum nu^-2 h_th(j), sum nu^-4 h_th(j)
  // u[15..20]: for j in {0,1,3}: sum h_ln(j), sum ln(nu) h_ln(j) ; u[21]: f ; u[22]: Sd ; u[23]: snr^2
  // (one loop: the theta_n- and alpha-rows for the nu_zero formulas and the full Hessian at the fit frequencies,
  // which some of those formulas need as well)
  double hv[15];
  for (int i = 0; i < 15; ++i) hv[i] = 0.0;
  double fmean = 0.0;
  for (int n = tid; n < nchan; n += NT) {
    double c[9];
    load_c(n, c);
    const double S = c[6];
    if (!(S > 0.0)) continue;
    if (!scat_on) { c[3] = c[4] = c[5] = c[7] = c[8] = 0.0; }
    const ChanJ j = chan_jac(a.lgf[mb + n] - lg2nT, a.nu2[mb + n], P, nD, nG, tau_e, alpha_e, a.log10_tau);
    const ChanK k = chan_k(c);
    const double n2 = a.nu2[mb + n], lnnu = a.lgf[mb + n] * 0.69314718055994530942;
    for (int p = 0; p < 5; ++p) {
      // Hessian row w.r.t. theta_n (= Hn[DM,p]/gDM_n etc.): d2C[theta,p], no S-dependence on theta
      const double h = (p < 3 ? k.A * j.Jth[p] : k.M * j.Jt[p - 3]) * zfl[p];
      u[3 * p] += h; u[3 * p + 1] += n2 * h; u[3 * p + 2] += n2 * n2 * h;
    }
    {
      // Hessian row w.r.t. alpha divided by ln(nu_n/nu_tau): d/dalpha = lnf * tau_n d/dtau_n
      const double k10 = a.log10_tau ? 2.302585092994045684 * j.taun : (tau_e != 0.0 ? j.taun / tau_e : 0.0);
      const double hs[3] = {k.M * j.taun * zfl[0], k.M * j.Jth[1] * j.taun * zfl[1],
                            (k.T1 * j.taun * j.Jt[0] + k.G2 * k10) * zfl[3]};
      for (int q = 0; q < 3; ++q) { u[15 + 2 * q] += hs[q]; u[16 + 2 * q] += lnnu * hs[q]; }
    }
    u[21] += k.f;
    u[22] += a.Sdn[(size_t)s * nchan + n];
    u[23] -= k.f;
    chan_hess(k, j, hv);
    fmean += a.freqs[mb + n];
  }
  {
    int q = 0;
    for (int i = 0; i < 5; ++i) for (int k = i; k < 5; ++k, ++q) hv[q] *= zfl[i] * zfl[k];
  }
  block_sum<24, NT>(u, sh);
  block_sum<15, NT>(hv, sh);
  double fm[1] = {fmean};
  block_sum<1, NT>(fm, sh);
  if (tid == 0) {
    double Hz[25];
    int q = 0;
    for (int i = 0; i < 5; ++i) for (int k = i; k < 5; ++k, ++q) { Hz[i * 5 + k] = hv[q]; Hz[k * 5 + i] = hv[q]; }
    double nzD = nD, nzG = nG, nzT = nT;
    const int code = fl[0] * 16 + fl[1] * 8 + fl[2] * 4 + fl[3] * 2 + fl[4];
    const double fbar = fm[0] / (double)a.nok[s];
    auto th = [&](int p, int m) { return u[3 * p + m]; };          // m: 0 sum, 1 nu^-2, 2 nu^-4
    auto ln = [&](int q2, int m) { return u[15 + 2 * q2 + m]; };    // q2: 0 phi, 1 DM, 2 tau
    if (code == 0b11000) {                                          // :746-752
      nzD = pow(th(0, 1) / th(0, 0), -0.5);
    } else if (code == 0b10100) {                                   // :753-760
      nzG = pow(th(0, 2) / th(0, 0), -0.25);
    } else if (code == 0b00011) {                                   // :761-767
      nzT = exp(ln(2, 1) / ln(2, 0));
    } else if (code == 0b11010) {                                   // :768-778
      const double H13 = Hz[3 * 5 + 0], H33 = Hz[3 * 5 + 3];
      nzD = pow((H13 * th(3, 1) - H33 * th(0, 1)) / (H13 * th(3, 0) - H33 * th(0, 0)), -0.5);
    } else if (code == 0b11011 || code == 0b11111) {                // :813-836 (and 893-901)
      // reduced indices (phi, DM, tau, alpha) = (0,1,3,4)
      const double H11 = Hz[0], H22 = Hz[6], H33 = Hz[18], H44 = Hz[24];
      const double H12 = Hz[1], H13 = Hz[3], H14 = Hz[4], H23 = Hz[8], H34 = Hz[19];
      (void)H22;
      const double c1 = H34 * H34 - H33 * H44, c2 = H13 * H44 - H14 * H34, c3 = H14 * H33 - H13 * H34;
      nzD = pow((c1 * th(0, 1) + c2 * th(3, 1) + c3 * th(4, 1)) / (c1 * th(0, 0) + c2 * th(3, 0) + c3 * th(4, 0)), -0.5);
      const double e1 = H13 * H22 - H12 * H23, e2 = H11 * H23 - H12 * H13, e3 = H12 * H12 - H11 * H22;
      nzT = exp((e1 * ln(0, 1) + e2 * ln(1, 1) + e3 * ln(2, 1)) / (e1 * ln(0, 0) + e2 * ln(1, 0) + e3 * ln(2, 0)));
    } else if (code == 0b11100 && (a.option == 0 || a.option == 1)) {   // :779-812
      double A, B, C_, D, E, F, G, Hh;
      if (a.option == 0) { A = th(0, 2); B = th(0, 0); C_ = th(2, 1); D = th(2, 0); E = th(2, 2); F = th(2, 0); G = th(0, 1); Hh = th(0, 0); }
      else { A = th(0, 2); B = th(0, 0); C_ = th(1, 1); D = th(1, 0); E = th(1, 2); F = th(1, 0); G = th(0, 1); Hh = th(0, 0); }
      const double cf[7] = {A * C_ - E * G, 0.0, E * Hh - A * D, 0.0, F * G - B * C_, 0.0, B * D - F * Hh};
      double r[8];
      const int nr = real_pos_roots(cf, 6, r);
      if (nr > 0) { double best = r[0]; for (int i = 1; i < nr; ++i) if (fabs(fbar - r[i]) < fabs(fbar - best)) best = r[i]; nzD = nzG = best; }
    } else if (code == 0b11110 && (a.option == 0 || a.option == 1)) {   // :837-892
      const double cD = K1, cG = K2;
      const double H14 = Hz[3 * 5 + 0], H44 = Hz[3 * 5 + 3];
      double cf[6]; int deg;
      if (a.option == 0) {
        const double A = cG * th(3, 2), a_ = cG * th(3, 0), B = cD * th(0, 1), b_ = cD * th(0, 0), C_ = cG * th(0, 2), c_ = cG * th(0, 0);
        const double D = cD * th(2, 1), d_ = cD * th(2, 0), E = cG * th(2, 2), e_ = cG * th(2, 0), F = cD * th(3, 1), f_ = cD * th(3, 0);
        cf[0] = A * A * B + H44 * C_ * D + H14 * E * F - H44 * B * E - A * C_ * F - H14 * A * D;
        cf[1] = -A * A * b_ - H44 * C_ * d_ - H14 * E * f_ + H44 * b_ * E + A * C_ * f_ + H14 * A * d_;
        cf[2] = -2 * A * a_ * B - H44 * c_ * D - H14 * e_ * F + H44 * B * e_ + (A * c_ + a_ * C_) * F + H14 * a_ * D;
        cf[3] = 2 * A * a_ * b_ + H44 * c_ * d_ + H14 * e_ * f_ - H44 * b_ * e_ - (A * c_ + a_ * C_) * f_ - H14 * a_ * d_;
        cf[4] = a_ * a_ * B - a_ * c_ * F;
        cf[5] = -a_ * a_ * b_ + a_ * c_ * f_;
        deg = 5;
      } else {
        const double A = cD * th(3, 1), a_ = cD * th(3, 0), B = cG * th(0, 2), b_ = cG * th(0, 0), C_ = cD * th(0, 1), c_ = cD * th(0, 0);
        const double D = cG * th(1, 2), d_ = cG * th(1, 0), E = cD * th(1, 1), e_ = cD * th(1, 0), F = cG * th(3, 2), f_ = cG * th(3, 0);
        cf[0] = A * A * B + H44 * C_ * D + H14 * E * F - H44 * B * E - A * C_ * F - H14 * A * D;
        cf[1] = -2 * A * a_ * B - H44 * c_ * D - H14 * e_ * F + H44 * B * e_ + (A * c_ + a_ * C_) * F + H14 * a_ * D;
        cf[2] = -(A * A * b_ - a_ * a_ * B) - H44 * C_ * d_ - H14 * E * f_ + H44 * b_ * E + (A * C_ * f_ - a_ * c_ * F) + H14 * A * d_;
        cf[3] = 2 * A * a_ * b_ + H44 * c_ * d_ + H14 * e_ * f_ - H44 * b_ * e_ - (A * c_ + a_ * C_) * f_ - H14 * a_ * d_;
        cf[4] = -a_ * a_ * b_ + a_ * c_ * f_;
        deg = 4;
      }
      double r[8];
      const int nr = real_pos_roots(cf, deg, r);
      if (nr > 0) {
        double best = sqrt(r[0]);
        for (int i = 1; i < nr; ++i) if (fabs(fbar - sqrt(r[i])) < fabs(fbar - best)) best = sqrt(r[i]);
        nzD = nzG = best;
      }
    }
    // requested output frequencies (NaN = zero-covariance value)          :1040-1050
    double noD = a.nu_outs ? a.nu_outs[(size_t)s * 3] : CUDART_NAN;
    double noG = a.nu_outs ? a.nu_outs[(size_t)s * 3 + 1] : CUDART_NAN;
    double noT = a.nu_outs ? a.nu_outs[(size_t)s * 3 + 2] : CUDART_NAN;
    if (!(noD == noD)) noD = nzD;
    if (!(noG == noG)) noG = nzG;
    if (!(noT == noT)) noT = nzT;
    if (a.is_toa) { if (fl[1]) noG = noD; else if (fl[2]) noD = noG; }
    bc[2] = noD; bc[3] = noG; bc[4] = noT;
  }
  __syncthreads();
  const double noD = bc[2], noG = bc[3], noT = bc[4];
  // ---- re-reference phi and tau (pptoaslib.py:1052-1065) -----------------------------------
  const double tau_out_lin = tau_e * pow(noT / nT, alpha_e);
  const double lg2noT = log2(noT);
  // ---- Hessian at the output frequencies, covariance incl. amplitudes (645-731) -------------
  double ho[15];
  for (int i = 0; i < 15; ++i) ho[i] = 0.0;
  for (int n = tid; n < nchan; n += NT) {
    double c[9];
    load_c(n, c);
    const double S = c[6];
    if (!(S > 0.0)) continue;
    if (!scat_on) { c[3] = c[4] = c[5] = c[7] = c[8] = 0.0; }
    const ChanJ j = chan_jac(a.lgf[mb + n] - lg2noT, a.nu2[mb + n], P, noD, noG, tau_out_lin, alpha_e, a.log10_tau);
    chan_hess(chan_k(c), j, ho);
  }
  {
    int q = 0;
    for (int i = 0; i < 5; ++i) for (int k = i; k < 5; ++k, ++q) ho[q] *= fl[i] * fl[k];
  }
  block_sum<15, NT>(ho, sh);
  if (tid == 0) {
    double Hf[25], H[25], L[25], Inv[25];
    int q = 0;
    for (int i = 0; i < 5; ++i) for (int k = i; k < 5; ++k, ++q) { Hf[i * 5 + k] = ho[q]; Hf[k * 5 + i] = ho[q]; }
    for (int i = 0; i < nfit; ++i) for (int k = 0; k < nfit; ++k) H[i * 5 + k] = Hf[idx[i] * 5 + idx[k]];
    bool ok = chol5(H, nfit, L);
    for (int i = 0; i < 25; ++i) Inv[i] = CUDART_NAN;
    if (ok) chol5_inverse(L, nfit, Inv);
    for (int i = 0; i < 25; ++i) bc[8 + i] = Inv[i];   // X^-1 = inv(H_out) over the fitted subset
  }
  __syncthreads();
  double Xinv[25];
  for (int i = 0; i < 25; ++i) Xinv[i] = bc[8 + i];
  for (int n = tid; n < nchan; n += NT) {
    double c[9];
    load_c(n, c);
    const double S = c[6];
    const size_t o = (size_t)s * nchan + n;
    double sc = 0.0, se = 0.0, csn = 0.0;
    if (S > 0.0) {
      if (!scat_on) { c[3] = c[4] = c[5] = c[7] = c[8] = 0.0; }
      const ChanJ j = chan_jac(a.lgf[mb + n] - lg2noT, a.nu2[mb + n], P, noD, noG, tau_out_lin, alpha_e, a.log10_tau);
      double dC[5], dS[5];
      chan_first(c, j, dC, dS);
      sc = c[0] / S;                                               // :688
      csn = sc * sqrt(S);                                          // :1081
      double U[5];
      for (int i = 0; i < nfit; ++i) U[i] = -2.0 * (dC[idx[i]] - sc * dS[idx[i]]);   // :690, 715
      double qf = 0.0;
      for (int i = 0; i < nfit; ++i) for (int k = 0; k < nfit; ++k) qf += U[i] * Xinv[i * 5 + k] * U[k];
      se = sqrt(1.0 / S + qf / (2.0 * S * S));                     // diag(2 LR), :721-724
    }
    if (a.scales) a.scales[o] = sc;
    if (a.scale_errs) a.scale_errs[o] = se;
    if (a.channel_snrs) a.channel_snrs[o] = csn;
  }
  if (tid == 0) {
    const double phi_inf = x[0] - K1 * x[1] / (nD * nD) - K2 * x[2] / (nG * nG * nG * nG);   // :1052-1053
    double phi_out = phi_inf + K1 * x[1] / (noD * noD) + K2 * x[2] / (noG * noG * noG * noG);
    phi_out = wrap_phase(phi_out);
    double* po = a.params + (size_t)s * 5;
    po[0] = phi_out; po[1] = x[1]; po[2] = x[2];
    po[3] = a.log10_tau ? log10(tau_out_lin) : tau_out_lin;
    po[4] = x[4];
    double* pe = a.param_errs + (size_t)s * 5;
    double* cv = a.cov + (size_t)s * 25;
    for (int i = 0; i < 5; ++i) pe[i] = 0.0;
    for (int i = 0; i < 25; ++i) cv[i] = 0.0;
    for (int i = 0; i < nfit; ++i) {
      pe[idx[i]] = sqrt(2.0 * Xinv[i * 5 + i]);
      for (int k = 0; k < nfit; ++k) cv[idx[i] * 5 + idx[k]] = 2.0 * Xinv[i * 5 + k];
    }
    double* no = a.nu_out + (size_t)s * 3;
    no[0] = noD; no[1] = noG; no[2] = noT;
    const int nok = a.nok[s];
    const double chi2 = u[22] + u[21];
    a.chi2[s] = chi2;
    a.red_chi2[s] = chi2 / ((double)nok * a.nbin - (double)(nfit + nok));
    a.snr[s] = sqrt(u[23]);
    a.nfeval[s] = a.st.iter[s] + a.st.iterc[s] + (state == 2 ? 1 : 0);
    a.st.done[s] = 1;
  }
}

// ----------------------------------------------------------------------------
// k_rfft_rows: half-spectra (slot layout, DC dropped) and/or get_noise_PS of
// independent rows.  Used by the batched 1-D FFTFIT (pplib.py:2073-2079) and
// by pp_get_noise_batch (pplib.py:2227-2245).
// ----------------------------------------------------------------------------
struct RowsArgs {
  const float* in;      // [nrows, 2N]
  float2* spec;         // [nrows, N] or null
  double* noise;        // [nrows] or null
  const void* twN;
  const void* tw2N;
  int nrows, conj;
  int kc;               // first harmonic of the noise estimate (get_noise_PS: int((1 - 1/frac) nharm), pplib.py:2244)
  double2* spec64;      // [nrows, N] FP64 spectra (slot layout) or null; dc64: [nrows] harmonic 0 (get_noise_fit)
  double* dc64;
};

template <int N, typename T>
__global__ void __launch_bounds__(256) k_rfft_rows(RowsArgs a) {
  using G = RowGeom<N>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufs = tw2N + (N / 2 + 2);
  __shared__ double red[8];
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  {
    const cx<T>* g1 = reinterpret_cast<const cx<T>*>(a.twN);
    const cx<T>* g2 = reinterpret_cast<const cx<T>*>(a.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  cx<T>* bufA = bufs + (size_t)r * 2 * N;
  cx<T>* bufB = bufA + N;
  const int row = blockIdx.x * G::kRows + r;
  const bool valid = row < a.nrows;
  const float4* src = reinterpret_cast<const float4*>(a.in + (size_t)(valid ? row : 0) * 2 * N);
#pragma unroll
  for (int m = 0; m < G::kLoads; ++m) {
    const int i4 = t_row + m * G::kTRow;
    const float4 v = valid ? __ldg(src + i4) : make_float4(0, 0, 0, 0);
    bufA[2 * i4] = mk<T>((T)v.x, (T)v.y);
    bufA[2 * i4 + 1] = mk<T>((T)v.z, (T)v.w);
  }
  __syncthreads();
  cx<T>* Z = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
  const int kc = a.kc;
  const int ntop = N + 1 - kc;
  double top = 0.0;
  float2* out = (a.spec && valid) ? a.spec + (size_t)row * N : nullptr;
  const float sgn = a.conj ? -1.f : 1.f;
  double2* out64 = (a.spec64 && valid) ? a.spec64 + (size_t)row * N : nullptr;
  auto put = [&](int k, cx<T> d) {
    if (k >= kc) top += (double)(d.x * d.x + d.y * d.y);
    if (out) out[(k == N) ? 0 : k] = make_float2((float)d.x, sgn * (float)d.y);
    if (out64) out64[(k == N) ? 0 : k] = make_double2((double)d.x, (double)d.y);
  };
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) {
    const int p = t_row + 1 + i * G::kTRow;
    if (p <= N / 2) {
      cx<T> dp, dq;
      unpack_pair<T>(Z, tw2N, N, p, dp, dq);
      put(p, dp);
      if (p < N / 2) put(N - p, dq);
    }
  }
  if (t_row == 0) {
    put(N, mk<T>(Z[0].x - Z[0].y, 0));
    if (kc == 0) { const double d0 = (double)(Z[0].x + Z[0].y); top += d0 * d0; }   // frac = 1: the DC term counts
    if (a.dc64 && valid) a.dc64[row] = (double)(Z[0].x + Z[0].y);
  }
  if (a.noise) {
#pragma unroll
    for (int o = (G::kTRow < 32 ? G::kTRow : 32) / 2; o > 0; o >>= 1) top += __shfl_xor_sync(0xffffffffu, top, o);
    if (G::kTRow > 32) {
      if ((tid & 31) == 0) red[tid >> 5] = top;
      __syncthreads();
      double st = 0.0;
#pragma unroll
      for (int w = 0; w < G::kTRow / 32; ++w) st += red[r * (G::kTRow / 32) + w];
      top = st;
    }
    if (t_row == 0 && valid) a.noise[row] = sqrt(top / ((double)(2 * N) * (double)ntop));
  }
}

// ----------------------------------------------------------------------------
// k_gauss_model: evolving-Gaussian model portrait (gen_gaussian_portrait,
// pplib.py:853-930) with evolve_parameter (996-1046) and gaussian_profile
// (770-825, norm=False).  One CTA per channel.  Scattering (params[1] != 0) is
// applied afterwards by k_rotate with the taus written here.
// ----------------------------------------------------------------------------
struct GaussModelArgs {
  const double* params;   // [2 + 6 ngauss]: DC, tau [bin], (loc, m_loc, wid, m_wid, amp, m_amp) per component
  const double* freqs;    // [nchan]
  float* out;             // [nchan, nbin]
  double* out64;          // the same in double when non-null (then `out` is unused)
  double* taus;           // [nchan] out: (tau/nbin) (nu/nu_ref)^alpha [rot]
  double nu_ref, alpha;
  int ngauss, nchan, nbin;
  int code_loc, code_wid, code_amp;   // 0 power law, 1 linear
};

__device__ __forceinline__ double evolve_param(double f, double nu_ref, double p, double m, int code) {
  if (code == 0) return exp((log(f) - log(nu_ref)) * m + log(p));   // pplib.py:1034-1037
  return (f - nu_ref) * m + p;                                       // pplib.py:1038-1041
}

constexpr int kMaxGauss = 64;

// bin centres: np.linspace(lo + d/(2 nbin), hi - d/(2 nbin), nbin) (pplib.py:671-684)
struct BinCentres {
  double lo, hi, dx;
  int nbin;
  __device__ explicit BinCentres(int n)
      : lo(1.0 / (2.0 * n)), hi(1.0 - 1.0 / (2.0 * n)), dx(n > 1 ? (hi - lo) / (double)(n - 1) : 0.0), nbin(n) {}
  __device__ double operator()(int i) const { return i == nbin - 1 ? hi : lo + (double)i * dx; }
};

// phases wrapped once around the component's centre (pplib.py:805-808)
__device__ __forceinline__ double gauss_wrapx(double x, double mean) {
  if (mean < 0.5) return x > mean + 0.5 ? x - 1.0 : x;
  return x < mean - 0.5 ? x + 1.0 : x;
}

// One component of gaussian_profile(norm=False) in one channel: value at bin centre x is
// scale * exp(-z^2/2) with z = gauss_z(x), where |z| < 20 (pplib.py:770-825).  renorm = scale / amp is
// the reference's peak renormalisation: 1 while loc lies in [0, 1), ~0 for a component centred outside.
// An invalid component (wid <= 0, or no bin within |z| < 20) has scale = renorm = 0.
struct GaussComp {
  double mean, isig, scale, renorm;
  __device__ double z(double x) const { return (gauss_wrapx(x, mean) - mean) * isig; }
};

__device__ __forceinline__ GaussComp gauss_comp(double loc, double wid, double amp, const BinCentres& xbin) {
  GaussComp c{0.0, 0.0, 0.0, 0.0};
  if (wid > 0.0) {
    const int nbin = xbin.nbin;
    const double sigma = wid / (2.0 * sqrt(2.0 * log(2.0)));
    c.mean = loc - floor(loc);                      // loc % 1
    c.isig = 1.0 / sigma;
    // the peak bin (argmax of the profile = smallest |z|, first index on ties) fixes the
    // amplitude: value exp(-0.5 ((x[ipk] - loc)/sigma)^2) at the peak bin (pplib.py:820-823)
    int i0 = (int)floor(c.mean * nbin);
    double best = CUDART_INF; int ipk = -1;
    for (int d = -1; d <= 1; ++d) {
      const int i = ((i0 + d) % nbin + nbin) % nbin;
      const double z = fabs((gauss_wrapx(xbin(i), c.mean) - c.mean) * c.isig);
      if (z < best || (z == best && i < ipk)) { best = z; ipk = i; }
    }
    if (best < 20.0) {
      const double xp = gauss_wrapx(xbin(ipk), c.mean);
      const double zl = (xp - loc) * c.isig;
      const double el = exp(-0.5 * zl * zl), eb = exp(-0.5 * best * best);
      c.scale = amp * el / eb;
      c.renorm = el / eb;
    }
  }
  return c;
}

__global__ void __launch_bounds__(256) k_gauss_model(GaussModelArgs a) {
  __shared__ GaussComp comp[kMaxGauss];
  const int ch = blockIdx.x, tid = threadIdx.x, nbin = a.nbin;
  const double f = a.freqs[ch];
  const BinCentres xbin(nbin);
  for (int g = tid; g < a.ngauss; g += 256) {
    const double* q = a.params + 2 + 6 * g;
    const double loc = evolve_param(f, a.nu_ref, q[0], q[1], a.code_loc);
    const double wid = evolve_param(f, a.nu_ref, q[2], q[3], a.code_wid);
    const double amp = evolve_param(f, a.nu_ref, q[4], q[5], a.code_amp);
    comp[g] = gauss_comp(loc, wid, amp, xbin);
  }
  if (tid == 0) a.taus[ch] = (a.params[1] / (double)nbin) * pow(f / a.nu_ref, a.alpha);   // pplib.py:4049-4053
  __syncthreads();
  const double dc = a.params[0];
  for (int i = tid; i < nbin; i += 256) {
    const double x = xbin(i);
    double v = dc;
    for (int g = 0; g < a.ngauss; ++g) {
      const GaussComp& c = comp[g];
      if (c.scale == 0.0) continue;
      const double z = c.z(x);
      if (fabs(z) < 20.0) v += c.scale * exp(-0.5 * z * z);
    }
    if (a.out64) a.out64[(size_t)ch * nbin + i] = v;
    else a.out[(size_t)ch * nbin + i] = (float)v;
  }
}

// float32 -> float64 (a scattered model is formed in float32 rows by k_rotate)
__global__ void __launch_bounds__(256) k_cvt_f32_f64(const float* __restrict__ in, double* __restrict__ out, size_t n) {
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) out[i] = (double)in[i];
}

// ----------------------------------------------------------------------------
// k_spline_model: B-spline (PCA) model portrait, gen_spline_portrait
// (pplib.py:932-956): port[n, :] = mean_prof + sum_c s_c(nu_n) eigvec[:, c] with
// s_c the parametric B-spline of scipy.interpolate.splev(freqs, tck, ext=0)
// (knots t, coefficients c, degree k <= 5; outside the knot range the end
// polynomials extrapolate, as FITPACK's splev does).  One CTA per channel.
// ----------------------------------------------------------------------------
struct SplineModelArgs {
  const double* mean_prof;  // [nbin]
  const double* eigvec;     // [nbin, ncomp]
  const double* knots;      // [nknots]
  const double* coefs;      // [ncomp, nknots - degree - 1]
  const double* freqs;      // [nchan]
  float* out;               // [nchan, nbin]
  int ncomp, nknots, degree, nchan, nbin;
};

constexpr int kMaxSplineComp = 32;

__global__ void __launch_bounds__(256) k_spline_model(SplineModelArgs a) {
  __shared__ double proj[kMaxSplineComp];
  const int ch = blockIdx.x, tid = threadIdx.x;
  const int k = a.degree, n = a.nknots - k - 1;        // n coefficients per component
  if (tid < a.ncomp) {
    const double x = a.freqs[ch];
    const double* t = a.knots;
    // knot span l with t[l] <= x < t[l+1], clamped to the first / last polynomial piece
    int l = k;
    while (l < n - 1 && x >= t[l + 1]) ++l;
    // de Boor: d_j = c[l-k+j], j = 0..k
    double d[6];
    const double* c = a.coefs + (size_t)tid * n;
    for (int j = 0; j <= k; ++j) d[j] = c[l - k + j];
    for (int r = 1; r <= k; ++r)
      for (int j = k; j >= r; --j) {
        const double tl = t[j + l - k], tr = t[j + 1 + l - r];
        const double al = (x - tl) / (tr - tl);
        d[j] = (1.0 - al) * d[j - 1] + al * d[j];
      }
    proj[tid] = d[k];
  }
  __syncthreads();
  for (int b = tid; b < a.nbin; b += 256) {
    double v = a.mean_prof[b];
    const double* e = a.eigvec + (size_t)b * a.ncomp;
    for (int c = 0; c < a.ncomp; ++c) v = fma(proj[c], e[c], v);
    a.out[(size_t)ch * a.nbin + b] = (float)v;
  }
}

// ----------------------------------------------------------------------------
// k_rotate: rfft -> multiply harmonic k by e^{2 pi i k theta} -> irfft
// (pplib.py:2338-2460).  One row-slot per channel row; rows = nsub*nchan.
// ----------------------------------------------------------------------------
struct RotateArgs {
  const float* in;      // [nsub,nchan,2N]
  float* out;           // [nsub,nchan,2N]
  const double* phase;  // [nsub]
  const double* DM;     // [nsub]
  const double* P;      // [nsub]
  const double* nu_ref; // [nsub]
  const double* GM;     // [nsub] or null (pptoaslib.rotate_portrait_full, pptoaslib.py:52-81)
  const double* nu_GM;  // [nsub] or null
  const double* nu2;    // [nchan]
  const double* taus;   // [nchan] scattering times [rot] or null: multiply harmonic k by 1/(1 + 2 pi i k tau_n)
                        // (scattering_portrait_FT, pplib.py:4080-4095)
  const double* resp;   // [nchan,N+1] real per-harmonic response or null: multiply harmonic k of channel n by resp[n][k]
                        // (instrumental_response_port_FT, pptoaslib.py:147-179; pptoas.py:388-394)
  const void* twN;
  const void* tw2N;
  int nsub, nchan;
};

// (c + i s) / (1 + i b): the rotation phasor times the scattering kernel B_nk
__device__ __forceinline__ void scatter_factor(double& c, double& s, double b) {
  const double q = 1.0 / (1.0 + b * b);
  const double cr = (c + s * b) * q, ci = (s - c * b) * q;
  c = cr; s = ci;
}

// theta_n = phase + Dconst DM (nu^-2 - nu_ref^-2)/P + Dconst^2 GM (nu^-4 - nu_GM^-4)/P
__device__ __forceinline__ double rot_theta(const RotateArgs& a, int s, int ch) {
  double theta = a.phase[s];
  const double dm = a.DM[s];
  const double n2 = a.nu2[ch];
  if (dm != 0.0) {
    const double nr = a.nu_ref[s];
    theta += kDconst * dm / a.P[s] * (n2 - 1.0 / (nr * nr));   // pplib.py:2381-2411
  }
  if (a.GM) {
    const double gm = a.GM[s];
    if (gm != 0.0) {
      const double ng = a.nu_GM[s];
      theta += kDconst * kDconst * gm / a.P[s] * (n2 * n2 - 1.0 / (ng * ng * ng * ng));   // pptoaslib.py:207
    }
  }
  return theta - rint(theta);
}

template <int N, typename T>
__global__ void __launch_bounds__(256) k_rotate(RotateArgs a) {
  using G = RowGeom<N>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufs = tw2N + (N / 2 + 2);
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  {
    const cx<T>* g1 = reinterpret_cast<const cx<T>*>(a.twN);
    const cx<T>* g2 = reinterpret_cast<const cx<T>*>(a.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  cx<T>* bufA = bufs + (size_t)r * 2 * N;
  cx<T>* bufB = bufA + N;
  const long nrows = (long)a.nsub * a.nchan;
  const long row = (long)blockIdx.x * G::kRows + r;
  const bool valid = row < nrows;
  const long rowc = valid ? row : 0;
  const int s = (int)(rowc / a.nchan), ch = (int)(rowc % a.nchan);
  const float4* src = reinterpret_cast<const float4*>(a.in + (size_t)rowc * 2 * N);
#pragma unroll
  for (int m = 0; m < G::kLoads; ++m) {
    const int i4 = t_row + m * G::kTRow;
    const float4 v = valid ? src[i4] : make_float4(0, 0, 0, 0);
    bufA[2 * i4] = mk<T>((T)v.x, (T)v.y);
    bufA[2 * i4 + 1] = mk<T>((T)v.z, (T)v.w);
  }
  __syncthreads();
  cx<T>* Z = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
  cx<T>* other = (Z == bufA) ? bufB : bufA;
  const double theta = rot_theta(a, s, ch);
  const double wtau = a.taus ? kTwoPi * a.taus[ch] : 0.0;
  const double* const resp = a.resp ? a.resp + (size_t)ch * (N + 1) : nullptr;
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) {
    const int p = t_row + 1 + i * G::kTRow;
    if (p <= N / 2) {
      cx<T> dp, dq;
      unpack_pair<T>(Z, tw2N, N, p, dp, dq);
      double c, sn;
      cis2pi((double)p * theta, c, sn);
      if (wtau != 0.0) scatter_factor(c, sn, wtau * (double)p);
      if (resp) { const double g = resp[p]; c *= g; sn *= g; }
      dp = cmul(dp, mk<T>((T)c, (T)sn));
      if (p < N / 2) {
        cis2pi((double)(N - p) * theta, c, sn);
        if (wtau != 0.0) scatter_factor(c, sn, wtau * (double)(N - p));
        if (resp) { const double g = resp[N - p]; c *= g; sn *= g; }
        dq = cmul(dq, mk<T>((T)c, (T)sn));
      } else {
        dq = dp;
      }
      cx<T> zp, zq;
      pack_pair<T>(dp, dq, tw2N[p], zp, zq);
      Z[p] = cconj(zp);           // conj for the inverse transform
      if (p < N / 2) Z[N - p] = cconj(zq);
    }
  }
  if (t_row == 0) {
    T d0 = Z[0].x + Z[0].y;
    double c, sn;
    cis2pi((double)N * theta, c, sn);
    if (wtau != 0.0) scatter_factor(c, sn, wtau * (double)N);
    if (resp) { d0 *= (T)resp[0]; c *= resp[N]; }
    const T dN = (Z[0].x - Z[0].y) * (T)c;   // irfft keeps the real part of the Nyquist term
    Z[0] = mk<T>(T(0.5) * (d0 + dN), -T(0.5) * (d0 - dN));
  }
  __syncthreads();
  cx<T>* Y = fft_forward<N, G::kTRow, T>(Z, other, twN, t_row);
  if (valid) {
    float4* dst = reinterpret_cast<float4*>(a.out + (size_t)row * 2 * N);
    const T sc = T(1) / T(N);
#pragma unroll
    for (int m = 0; m < G::kLoads; ++m) {
      const int i4 = t_row + m * G::kTRow;
      const cx<T> y0 = Y[2 * i4], y1 = Y[2 * i4 + 1];
      dst[i4] = make_float4((float)(y0.x * sc), (float)(-y0.y * sc), (float)(y1.x * sc), (float)(-y1.y * sc));
    }
  }
}

// ----------------------------------------------------------------------------
// k_align_accum: K5, the inner loop of ppalign.align_archives (ppalign.py:160-213):
// aligned[n] = sum_s w_sn * rotate(data_sn, phi_s, DM_s), accumulated in the
// Fourier domain in double and inverse transformed once per channel.  One row
// slot per channel, looping over the subints.
// ----------------------------------------------------------------------------
struct AlignArgs {
  RotateArgs r;            // in = data [nsub,nchan,2N]; out unused
  const double* weights;   // [nsub,nchan] (scales / sigma^2, ppalign.py:202); 0 skips the row
  double* aligned;         // [nchan,2N] sum (not normalised)
  double* wsum;            // [nchan] sum of the weights used
};

template <int N>
__global__ void __launch_bounds__(256) k_align_accum(AlignArgs a) {
  using G = RowGeom<N>;
  using T = double;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufs = tw2N + (N / 2 + 2);
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  {
    const cx<T>* g1 = reinterpret_cast<const cx<T>*>(a.r.twN);
    const cx<T>* g2 = reinterpret_cast<const cx<T>*>(a.r.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  cx<T>* bufA = bufs + (size_t)r * 2 * N;
  cx<T>* bufB = bufA + N;
  const int ch = blockIdx.x * G::kRows + r;
  const bool valid = ch < a.r.nchan;
  const int chc = valid ? ch : 0;
  cx<T> accp[G::kPairs], accq[G::kPairs];
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) { accp[i] = mk<T>(0, 0); accq[i] = mk<T>(0, 0); }
  T acc0 = 0, accN = 0, wtot = 0;
  for (int s = 0; s < a.r.nsub; ++s) {
    const double w = valid ? a.weights[(size_t)s * a.r.nchan + chc] : 0.0;
    const bool use = w != 0.0 && fabs(w) < 1e300;   // negative weights (negative fitted amplitudes) count, ppalign.py:202-209
    const float4* src = reinterpret_cast<const float4*>(a.r.in + ((size_t)s * a.r.nchan + chc) * 2 * N);
    __syncthreads();   // previous iteration's reads of the buffers are done
#pragma unroll
    for (int m = 0; m < G::kLoads; ++m) {
      const int i4 = t_row + m * G::kTRow;
      const float4 v = use ? __ldg(src + i4) : make_float4(0, 0, 0, 0);
      bufA[2 * i4] = mk<T>((T)v.x, (T)v.y);
      bufA[2 * i4 + 1] = mk<T>((T)v.z, (T)v.w);
    }
    __syncthreads();
    cx<T>* Z = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
    if (use) {
      const double theta = rot_theta(a.r, s, chc);
#pragma unroll
      for (int i = 0; i < G::kPairs; ++i) {
        const int p = t_row + 1 + i * G::kTRow;
        if (p <= N / 2) {
          cx<T> dp, dq;
          unpack_pair<T>(Z, tw2N, N, p, dp, dq);
          double c, sn;
          cis2pi((double)p * theta, c, sn);
          dp = cmul(dp, mk<T>(c * w, sn * w));
          accp[i] = cadd(accp[i], dp);
          if (p < N / 2) {
            cis2pi((double)(N - p) * theta, c, sn);
            dq = cmul(dq, mk<T>(c * w, sn * w));
            accq[i] = cadd(accq[i], dq);
          }
        }
      }
      if (t_row == 0) {
        double c, sn;
        cis2pi((double)N * theta, c, sn);
        acc0 += w * (Z[0].x + Z[0].y);
        accN += w * (Z[0].x - Z[0].y) * c;
        wtot += w;
      }
    }
  }
  __syncthreads();
  // pack the accumulated half spectrum and inverse transform (conj / FFT / conj / N)
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) {
    const int p = t_row + 1 + i * G::kTRow;
    if (p <= N / 2) {
      cx<T> zp, zq;
      pack_pair<T>(accp[i], (p < N / 2) ? accq[i] : accp[i], tw2N[p], zp, zq);
      bufA[p] = cconj(zp);
      if (p < N / 2) bufA[N - p] = cconj(zq);
    }
  }
  if (t_row == 0) bufA[0] = mk<T>(T(0.5) * (acc0 + accN), -T(0.5) * (acc0 - accN));
  __syncthreads();
  cx<T>* Y = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
  if (valid) {
    double* dst = a.aligned + (size_t)ch * 2 * N;
    const T sc = T(1) / T(N);
    for (int j = t_row; j < N; j += G::kTRow) {
      dst[2 * j] = Y[j].x * sc;
      dst[2 * j + 1] = -Y[j].y * sc;
    }
    if (t_row == 0) a.wsum[ch] = wtot;
  }
}

// ----------------------------------------------------------------------------
// Fused ppalign accumulation (ppalign.py:197-213) from the spectra k_spectra kept:
//   acc[n,k] += sum_s w_sn d_snk e^{2 pi i k theta_sn},  w_sn = scales_sn / sigma_sn^2,
// theta_sn from the FITTED phi_s, DM_s about nu_out_s.  k_align_spec streams the float2
// spectra once (as k_pass2 streams X): grid (nchan, nsplit) x N/8 threads, thread t owns
// slots 8t..8t+7; the phasor of slot 8t comes from e^{2 pi i theta} by squaring and a
// binary product, the next seven by recurrence.  k_align_finish packs the sums and
// inverse transforms one channel per row slot.
// ----------------------------------------------------------------------------
struct AlignSpecArgs {
  const float2* D;         // [chunk,nchan,N]
  const double* Ddc;       // [chunk,nchan]
  const double* params;    // [nsub,5] fitted, phi at nu_out
  const double* nu_out;    // [nsub,3]
  const double* P;         // [nsub]
  const double* scales;    // [nsub,nchan]
  const double* sigma;     // [nsub,nchan] (0 = unused channel)
  const int* rc;           // [nsub] return codes (3 = non-finite fit: skipped)
  const double* nu2;       // [nchan]
  double2* acc;            // [nsplit,nchan,N] slot layout (slot 0: x = Nyquist sum, y = DC sum): one slice
  double* wsum;            // [nsplit,nchan]     per blockIdx.y, added to by one CTA only (deterministic)
  int s0, ns, nchan;
};

template <int N>
__global__ void __launch_bounds__(N / 8) k_align_spec(AlignSpecArgs a) {
  constexpr int T = N / 8;
  static_assert(T >= 4 && (T & (T - 1)) == 0, "row size");
  constexpr int LOGT = Log2<T>::value;
  const int n = blockIdx.x, t = threadIdx.x;
  const int per = (a.ns + gridDim.y - 1) / gridDim.y;
  const int sb = blockIdx.y * per, se = min(a.ns, sb + per);
  cx<double> acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = mk<double>(0.0, 0.0);
  double wtot = 0.0, dcsum = 0.0;
  const double n2 = a.nu2[n];
  auto row_ptr = [&](int sl) { return reinterpret_cast<const float4*>(a.D + ((size_t)sl * a.nchan + n) * N) + 4 * t; };
  float4 q[4], qn[4];
  if (sb < se) {
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = ld_stream(row_ptr(sb) + j);
  }
  for (int sl = sb; sl < se; ++sl) {
    if (sl + 1 < se) {
#pragma unroll
      for (int j = 0; j < 4; ++j) qn[j] = ld_stream(row_ptr(sl + 1) + j);
    }
    const int s = a.s0 + sl;
    const double sg = a.sigma[(size_t)s * a.nchan + n];
    const double sc = a.scales[(size_t)s * a.nchan + n];
    const double w = (sg > 0.0 && a.rc[s] != 3) ? sc / (sg * sg) : 0.0;       // ppalign.py:202
    if (w != 0.0 && fabs(w) < 1e300) {    // uniform over the CTA; negative amplitudes weigh in as in the reference
      const double nr = a.nu_out[(size_t)s * 3];
      double theta = a.params[(size_t)s * 5] + kDconst * a.params[(size_t)s * 5 + 1] * (n2 - 1.0 / (nr * nr)) / a.P[s];
      theta -= rint(theta);
      cx<double> e1, f;
      cis2pi(theta, e1.x, e1.y);
      f = csqr(csqr(csqr(e1)));                     // e^{2 pi i 8 theta}
      cx<double> ph = mk<double>(1.0, 0.0);
#pragma unroll
      for (int b = 0; b < LOGT; ++b) {              // e^{2 pi i 8 t theta}
        if ((t >> b) & 1) ph = cmul(ph, f);
        f = csqr(f);
      }
      // f is now e^{2 pi i 8 T theta} = e^{2 pi i N theta}: the Nyquist phasor
      const float2 d[8] = {make_float2(q[0].x, q[0].y), make_float2(q[0].z, q[0].w), make_float2(q[1].x, q[1].y),
                           make_float2(q[1].z, q[1].w), make_float2(q[2].x, q[2].y), make_float2(q[2].z, q[2].w),
                           make_float2(q[3].x, q[3].y), make_float2(q[3].z, q[3].w)};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double wx = w * (double)d[j].x, wy = w * (double)d[j].y;
        if (j == 0 && t == 0) {
          // slot 0 = Nyquist (real): irfft keeps Re(d_N e^{i N theta}); y carries the DC sum
          acc[0].x = fma(wx, f.x, acc[0].x);
        } else {
          acc[j].x += wx * ph.x - wy * ph.y;
          acc[j].y += wx * ph.y + wy * ph.x;
        }
        ph = cmul(ph, e1);
      }
      if (t == 0) { dcsum = fma(w, a.Ddc[(size_t)sl * a.nchan + n], dcsum); wtot += w; }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = qn[j];
  }
  double2* o = a.acc + ((size_t)blockIdx.y * a.nchan + n) * N + 8 * t;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    o[j].x += acc[j].x;
    o[j].y += (j == 0 && t == 0) ? dcsum : acc[j].y;
  }
  if (t == 0) a.wsum[(size_t)blockIdx.y * a.nchan + n] += wtot;
}

struct AlignFinishArgs {
  const double2* acc;      // [nsplit,nchan,N] from k_align_spec
  const double* wsum_parts;// [nsplit,nchan]
  double* aligned;         // [nchan,2N] out (not normalised by the weights)
  double* wsum;            // [nchan] out
  const void* twN;
  const void* tw2N;
  int nchan, nsplit;
};

template <int N>
__global__ void __launch_bounds__(256) k_align_finish(AlignFinishArgs a) {
  using G = RowGeom<N>;
  using T = double;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufs = tw2N + (N / 2 + 2);
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  {
    const cx<T>* g1 = reinterpret_cast<const cx<T>*>(a.twN);
    const cx<T>* g2 = reinterpret_cast<const cx<T>*>(a.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  __syncthreads();
  cx<T>* bufA = bufs + (size_t)r * 2 * N;
  cx<T>* bufB = bufA + N;
  const int ch = blockIdx.x * G::kRows + r;
  const bool valid = ch < a.nchan;
  const double2* src0 = a.acc + (size_t)(valid ? ch : 0) * N;
  const size_t part = (size_t)a.nchan * N;
  auto total = [&](int slot_i) {        // the slices in a fixed order
    double2 v = make_double2(0.0, 0.0);
    for (int q = 0; q < a.nsplit; ++q) { const double2 u = src0[q * part + slot_i]; v.x += u.x; v.y += u.y; }
    return v;
  };
  if (valid && t_row == 0) {
    double w = 0.0;
    for (int q = 0; q < a.nsplit; ++q) w += a.wsum_parts[(size_t)q * a.nchan + ch];
    a.wsum[ch] = w;
  }
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) {
    const int p = t_row + 1 + i * G::kTRow;
    if (p <= N / 2) {
      const double2 vp = total(p), vq = total((p < N / 2) ? N - p : p);
      cx<T> zp, zq;
      pack_pair<T>(mk<T>(vp.x, vp.y), mk<T>(vq.x, vq.y), tw2N[p], zp, zq);
      bufA[p] = cconj(zp);
      if (p < N / 2) bufA[N - p] = cconj(zq);
    }
  }
  if (t_row == 0) {
    const double2 v0 = total(0);   // x = Nyquist sum, y = DC sum
    bufA[0] = mk<T>(T(0.5) * (v0.y + v0.x), -T(0.5) * (v0.y - v0.x));
  }
  __syncthreads();
  cx<T>* Y = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
  if (valid) {
    double* dst = a.aligned + (size_t)ch * 2 * N;
    const T sc = T(1) / T(N);
    for (int j = t_row; j < N; j += G::kTRow) {
      dst[2 * j] = Y[j].x * sc;
      dst[2 * j + 1] = -Y[j].y * sc;
    }
  }
}

// ----------------------------------------------------------------------------
// Arbitrary nbin (bluestein.cuh): element-wise kernels on the FP64 spectrum scratch the Bluestein row
// transforms write / read.  Rows have Npad slots, slot k = harmonic k for 1 <= k <= L = nbin/2.
// ----------------------------------------------------------------------------
// conj(m), |m|^2, p_n of the model from its spectra (k_model for any nbin): one CTA per channel
__global__ void __launch_bounds__(256) k_model_from_spec(const cx<double>* __restrict__ spec, cx<float>* mconj32,
                                                          cx<double>* mconj64, double* mpow, double* pn, int Npad) {
  __shared__ double sh[8];
  const int ch = blockIdx.x, tid = threadIdx.x;
  double v[1] = {0.0};
  for (int k = tid; k < Npad; k += 256) {
    const cx<double> d = spec[(size_t)ch * Npad + k];
    const double pw = d.x * d.x + d.y * d.y;
    v[0] += pw;
    mconj64[(size_t)ch * Npad + k] = cconj(d);
    mconj32[(size_t)ch * Npad + k] = mk<float>((float)d.x, (float)(-d.y));
    mpow[(size_t)ch * Npad + k] = pw;
  }
  block_sum<1, 256>(v, sh);
  if (tid == 0) pn[ch] = v[0];
}

// float spectra (optionally conjugated) and the noise level of transformed rows (k_rfft_rows for any nbin)
__global__ void __launch_bounds__(256) k_rows_from_spec(const cx<double>* __restrict__ spec, const double* __restrict__ dc,
                                                         float2* out, double* noise, int Npad, int L, int kc, int conj) {
  __shared__ double sh[8];
  const long row = blockIdx.x;
  const int tid = threadIdx.x;
  double v[1] = {0.0};
  const float sgn = conj ? -1.f : 1.f;
  for (int k = tid; k < Npad; k += 256) {
    const cx<double> d = spec[(size_t)row * Npad + k];
    if (k >= kc && k >= 1) v[0] += d.x * d.x + d.y * d.y;
    if (out) out[(size_t)row * Npad + k] = make_float2((float)d.x, sgn * (float)d.y);
  }
  if (tid == 0 && kc == 0) v[0] += dc[row] * dc[row];     // frac = 1: the DC term counts
  block_sum<1, 256>(v, sh);
  if (tid == 0 && noise) noise[row] = sqrt(v[0] / ((double)(2 * L) * (double)(L + 1 - kc)));
}

// harmonic k of row (s, ch) times e^{2 pi i k theta} [/(1 + 2 pi i k tau_n)] [resp_n(k)] (k_rotate's multiply)
__global__ void __launch_bounds__(256) k_rot_mul(RotateArgs a, cx<double>* spec, double* dc, int Npad, int L) {
  const long row = blockIdx.x;
  const int s = (int)(row / a.nchan), ch = (int)(row % a.nchan);
  const double theta = rot_theta(a, s, ch);
  const double wtau = a.taus ? kTwoPi * a.taus[ch] : 0.0;
  const double* const resp = a.resp ? a.resp + (size_t)ch * (L + 1) : nullptr;
  for (int k = threadIdx.x + 1; k <= L; k += 256) {
    double c, sn;
    cis2pi((double)k * theta, c, sn);
    if (wtau != 0.0) scatter_factor(c, sn, wtau * (double)k);
    if (resp) { c *= resp[k]; sn *= resp[k]; }
    cx<double>& d = spec[(size_t)row * Npad + k];
    d = (k < L) ? cmul(d, mk<double>(c, sn)) : mk<double>(d.x * c, 0.0);   // irfft keeps the real part of the Nyquist term
  }
  if (threadIdx.x == 0 && resp) dc[row] *= resp[0];
}

// acc[n] += sum_s w[s,n] spec[s,n] over the rotated spectrum rows (slot layout) and dc[n] likewise, in double,
// subints in order: the accumulation of ppalign.py:202-208 for any nbin (one inverse transform of acc follows)
__global__ void __launch_bounds__(256) k_wsum_spec(const cx<double>* __restrict__ spec, const double* __restrict__ dc,
                                                    const double* __restrict__ w, cx<double>* acc, double* acc_dc, double* wsum,
                                                    int nsub, int nchan, int Npad, int first_call) {
  const int ch = blockIdx.x;
  for (int k = threadIdx.x; k < Npad; k += 256) {
    cx<double> v = first_call ? mk<double>(0.0, 0.0) : acc[(size_t)ch * Npad + k];
    for (int s = 0; s < nsub; ++s) {
      const double ws = w[(size_t)s * nchan + ch];
      if (ws != 0.0 && fabs(ws) < 1e300) {
        const cx<double> d = spec[((size_t)s * nchan + ch) * Npad + k];
        v.x = fma(ws, d.x, v.x);
        v.y = fma(ws, d.y, v.y);
      }
    }
    acc[(size_t)ch * Npad + k] = v;
  }
  if (threadIdx.x == 0) {
    double t = first_call ? 0.0 : wsum[ch], d0 = first_call ? 0.0 : acc_dc[ch];
    for (int s = 0; s < nsub; ++s) {
      const double ws = w[(size_t)s * nchan + ch];
      if (ws != 0.0 && fabs(ws) < 1e300) { t += ws; d0 = fma(ws, dc[(size_t)s * nchan + ch], d0); }
    }
    wsum[ch] = t;
    acc_dc[ch] = d0;
  }
}

// the slices of the fused ppalign sum (k_align_spec) added in a fixed order into spectrum rows + DC terms
__global__ void __launch_bounds__(256) k_align_reduce_any(const double2* __restrict__ acc, const double* __restrict__ wparts,
                                                           cx<double>* spec, double* dc, double* wsum, int nchan, int Npad, int nsplit) {
  const int ch = blockIdx.x;
  const size_t part = (size_t)nchan * Npad;
  for (int k = threadIdx.x; k < Npad; k += 256) {
    double2 v = make_double2(0.0, 0.0);
    for (int q = 0; q < nsplit; ++q) { const double2 u = acc[q * part + (size_t)ch * Npad + k]; v.x += u.x; v.y += u.y; }
    if (k == 0) { dc[ch] = v.y; v = make_double2(0.0, 0.0); }      // slot 0: y carries the DC sum
    spec[(size_t)ch * Npad + k] = mk<double>(v.x, v.y);
  }
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int q = 0; q < nsplit; ++q) t += wparts[(size_t)q * nchan + ch];
    wsum[ch] = t;
  }
}

// ----------------------------------------------------------------------------
// k_noise_fit: get_noise_fit (pplib.py:2255-2284) -- the noise floor of a row's power spectrum starts
// at fact * kc, kc from find_kc (pplib.py:1465-1495): scipy.optimize.brute (20 x 20 x 20 grid, no polish)
// of chi2(a, b, dc) = sum_k (log10 pows_k - b e^{-a k} - dc)^2 over a in [1/nharm, 1], b in
// [0, max - min], dc in [min, max] of log10 pows; the first k with e^{-a k} < 0.005.  One CTA per row:
// the table e^{-a k} of one a at a time in shared memory, the 400 (b, dc) points of that slice spread over
// the threads.  The grid values are np.mgrid's, i * step + start rounded twice, and the model term is
// b e^{-a k} + dc rounded twice, as numpy evaluates them.  The flat argmin in scipy's C order (a slowest)
// follows np.argmin (noise_argmin_before).
// ----------------------------------------------------------------------------
// np.argmin's order over the flat grid: a NaN chi2 wins, the first one; otherwise the lowest chi2, the lowest
// index on ties.  A row with an exactly zero harmonic has log10 pows = -inf, which makes every chi2 NaN: then
// grid point 0 (a = 1/nharm) is the minimiser, as in the reference.
__device__ __forceinline__ bool noise_argmin_before(double c, int i, double best, int besti) {
  if (isnan(c)) return !isnan(best) || i < besti;
  if (isnan(best)) return false;
  return c < best || (c == best && i < besti);
}

// find_kc of one row, called by all 256 threads of the CTA after y[0 .. nh) (the row's log10 powers, shared memory)
// is written and synchronised; ek [nh] is shared scratch.  Returns k_crit, the first k with e^{-a k} < 0.005 at the
// grid minimiser (nh - 1 if there is none), in every thread.  k_noise_fit and the low-pass of make_spline_model
// (k_lowpass, k_lowpass_spec) both take their cut-off from here.
__device__ int find_kc(const double* y, double* ek, int nh) {
  __shared__ double shv[8];
  __shared__ int shi[8];
  __shared__ double lim[2];
  __shared__ int kc_sh;
  const int tid = threadIdx.x;
  if (tid < 32) {   // min / max of y
    double lo = CUDART_INF, hi = -CUDART_INF;
    for (int k = tid; k < nh; k += 32) { lo = fmin(lo, y[k]); hi = fmax(hi, y[k]); }
    for (int o = 16; o > 0; o >>= 1) { lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o)); }
    if (tid == 0) { lim[0] = lo; lim[1] = hi; }
  }
  __syncthreads();
  const double ymin = lim[0], ymax = lim[1];
  const double a_lo = 1.0 / (double)nh, a_st = (1.0 - a_lo) / 19.0, b_st = (ymax - ymin) / 19.0, d_st = (ymax - ymin) / 19.0;
  auto mgrid = [](int i, double st, double lo) { return __dadd_rn(__dmul_rn((double)i, st), lo); };
  // every thread evaluates at least one point (400 per a, 256 threads), so besti is a grid index after the loop
  double best = CUDART_INF;
  int besti = 0x7fffffff;
  for (int ia = 0; ia < 20; ++ia) {
    const double av = mgrid(ia, a_st, a_lo);
    __syncthreads();
    for (int k = tid; k < nh; k += 256) ek[k] = exp(-av * (double)k);
    __syncthreads();
    for (int q = tid; q < 400; q += 256) {
      const int ib = q / 20, id = q % 20;
      const double bv = mgrid(ib, b_st, 0.0), dv = mgrid(id, d_st, ymin);
      double c2 = 0.0;
      for (int k = 0; k < nh; ++k) { const double r = y[k] - __dadd_rn(__dmul_rn(bv, ek[k]), dv); c2 = fma(r, r, c2); }
      const int flat = ia * 400 + q;
      if (noise_argmin_before(c2, flat, best, besti)) { best = c2; besti = flat; }
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
    if (noise_argmin_before(ov, oi, best, besti)) { best = ov; besti = oi; }
  }
  if ((tid & 31) == 0) { shv[tid >> 5] = best; shi[tid >> 5] = besti; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < 8; ++w) if (noise_argmin_before(shv[w], shi[w], best, besti)) { best = shv[w]; besti = shi[w]; }
    const int ia = besti / 400;
    const double av = mgrid(ia, a_st, a_lo);
    int kcrit = nh - 1;
    for (int k = 0; k < nh; ++k) if (exp(-av * (double)k) < 0.005) { kcrit = k; break; }
    kc_sh = kcrit;
  }
  __syncthreads();
  return kc_sh;
}

__global__ void __launch_bounds__(256) k_noise_fit(const double2* __restrict__ spec, const double* __restrict__ dc, double* noise,
                                                    int nslot, int L, int nyq_slot, double fact) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* y = reinterpret_cast<double*>(smem_raw);     // [L + 1] log10 pows
  double* pw = y + (L + 1);                            // [L + 1] pows
  double* ek = pw + (L + 1);                           // [L + 1] e^{-a k}
  const long row = blockIdx.x;
  const int tid = threadIdx.x, nh = L + 1;
  const double inv_n = 1.0 / (double)(2 * L);
  for (int k = tid; k < nh; k += 256) {
    double p;
    if (k == 0) p = dc[row] * dc[row];
    else { const double2 d = spec[(size_t)row * nslot + (k == L ? nyq_slot : k)]; p = d.x * d.x + d.y * d.y; }
    p *= inv_n;
    pw[k] = p;
    y[k] = log10(p);
  }
  __syncthreads();
  const int kcrit = find_kc(y, ek, nh);
  if (tid == 0) {
    double kf = fact * (double)kcrit;
    if (kf >= (double)nh) kf = fmin((double)(int)(0.99 * nh), kf);
    const int k0 = (int)kf;
    double sum = 0.0;
    for (int k = k0; k < nh; ++k) sum += pw[k];
    noise[row] = sqrt(sum / (double)(nh - k0));
  }
}

// ----------------------------------------------------------------------------
// Simulated archives (pp_simulate_batch): row (s, n) is
//   Y_k = S_sn M_mnk e^{-2 pi i k theta_sn} B_snk,  out = irfft(Y) + sigma_sn z(seed, s_global, n, b)
// with m = model_index[s], theta_sn = rot_theta (the injected phi, DM, GM: pp_fit_batch recovers them) and
// B_snk = 1/(1 + 2 pi i k tau_sn), tau_sn = tau_s (nu_n/nu_tau_s)^alpha_s [rot].  The model spectra M are float64
// rows computed once per call; the inverse transform is FP64.
//
// Noise: Philox4x32-10 (Salmon et al. 2011, the Random123 constants) with key (seed lo, seed hi) and counter
// (q, n, s_global lo, s_global hi) gives four uint32 for bins 4q .. 4q+3 of channel n of subint s_global; each is
// mapped to u = f32((x >> 8) 2^-24 + 2^-25) in (0, 1] (exact below 1/2, rounded to nearest even above) and pairs
// go through Box-Muller in float32 with the accurate logf / sqrtf / sincospif:
//   (z0, z1) = sqrt(-2 ln u0) (cos 2 pi u1, sin 2 pi u1), (z2, z3) likewise from (u2, u3);  |z| <= 5.89.
// A subint's samples depend on (seed, its global index, its model and parameters) only, not on the batch, the
// chunk or the device.
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    if (i) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

__device__ __forceinline__ float sim_uniform(unsigned x) {
  return __fadd_rn((float)(x >> 8) * 5.9604644775390625e-8f, 2.98023223876953125e-8f);   // 2^-24, 2^-25
}

__device__ __forceinline__ void box_muller(unsigned a, unsigned b, float& z0, float& z1) {
  const float r = sqrtf(-2.0f * logf(sim_uniform(a)));
  float sn, cs;
  sincospif(2.0f * sim_uniform(b), &sn, &cs);
  z0 = r * cs;
  z1 = r * sn;
}

struct SimArgs {
  RotateArgs r;               // phase, DM, P, nu_ref (= nu_DM), GM, nu_GM of the chunk's subints; nu2 [nmodel * nchan]
  const cx<double>* mspec;    // [nmodel * nchan, sstride] model spectra: slot k = harmonic k, 1..nbin/2; slot 0 = the DC
                              // term (power-of-two nbin) or unused (mdc)
  const double* mdc;          // [nmodel * nchan] DC terms (other nbin) or null
  const double* freqs;        // [nmodel * nchan]
  const int* index;           // [nsub] model of each subint or null (model 0)
  const double* tau;          // [nsub] or null (unscattered); alpha, nu_tau with it
  const double* alpha;
  const double* nu_tau;
  const double* scales;       // [nsub, nchan] or null (1)
  const double* sigma;        // [nsub, nchan] or null (0)
  float* out;                 // [nsub, nchan, nbin] float32 or null
  int16_t* raw;               // [nsub, nchan, nbin] or null; dat_scl, dat_offs [nsub, nchan] with it
  float* dat_scl;
  float* dat_offs;
  long long s_first;          // global index of subint 0 of the chunk (first_subint + chunk start)
  unsigned key0, key1;
  int nchan, nbin, sstride;
};

// row geometry shared by the simulate kernels: the model row, theta, the scattering and the scale of row (s, ch)
struct SimRow {
  const cx<double>* M;
  double theta, wtau, S, sigma;
  int mrow;
};
__device__ __forceinline__ SimRow sim_row(const SimArgs& a, int s, int ch) {
  SimRow w;
  const int m = a.index ? __ldg(a.index + s) : 0;
  w.mrow = m * a.nchan + ch;
  w.M = a.mspec + (size_t)w.mrow * a.sstride;
  w.theta = rot_theta(a.r, s, w.mrow);
  w.wtau = a.tau ? kTwoPi * a.tau[s] * pow(a.freqs[w.mrow] / a.nu_tau[s], a.alpha[s]) : 0.0;
  const size_t sc = (size_t)s * a.nchan + ch;
  w.S = a.scales ? a.scales[sc] : 1.0;
  w.sigma = a.sigma ? a.sigma[sc] : 0.0;
  return w;
}

// S e^{-2 pi i k theta} / (1 + 2 pi i k tau) times M_k
__device__ __forceinline__ cx<double> sim_harmonic(const SimRow& w, int k) {
  double c, sn;
  cis2pi((double)k * w.theta, c, sn);
  sn = -sn;
  if (w.wtau != 0.0) scatter_factor(c, sn, w.wtau * (double)k);
  return cmul(w.M[k], mk<double>(w.S * c, w.S * sn));
}

// samples 4q .. 4q+3 (the first n of them) of row (s, ch): clean values y plus sigma z, rounded to float32
__device__ __forceinline__ void sim_noise(const SimArgs& a, const SimRow& w, int q, int ch, int s, const double (&y)[4],
                                          float (&v)[4]) {
  float z[4] = {0.f, 0.f, 0.f, 0.f};
  if (w.sigma != 0.0) {
    const unsigned long long sg = (unsigned long long)(a.s_first + s);
    const uint4 x = philox4x32_10(make_uint4((unsigned)q, (unsigned)ch, (unsigned)sg, (unsigned)(sg >> 32)),
                                  make_uint2(a.key0, a.key1));
    box_muller(x.x, x.y, z[0], z[1]);
    box_muller(x.z, x.w, z[2], z[3]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = (float)fma(w.sigma, (double)z[i], y[i]);
}

// pptoas.quantize_subints of one row, given its float32 min / max: raw = clip(rint((x - offs) / scl)) in double,
// offs = f32((hi + lo) / 2), scl = f32((hi - lo) / 65000) (1 for a constant row)
struct SimQuant {
  double offs, scl;
  __device__ __forceinline__ SimQuant(float lo, float hi) {
    offs = (double)(float)(0.5 * ((double)hi + (double)lo));
    scl = hi > lo ? (double)(float)(((double)hi - (double)lo) / 65000.0) : 1.0;
  }
  __device__ __forceinline__ int16_t operator()(float x) const {
    const double r = rint(((double)x - offs) / scl);
    return (int16_t)fmin(fmax(r, -32768.0), 32767.0);
  }
};

// Power-of-two nbin: one row slot per output row: the spectrum row (L2-resident) times the phasor and scattering
// factor, packed for the inverse, one FP64 inverse transform, then noise and the store (float32 and / or int16 after
// a row-slot min / max).  Half of k_rotate's transforms, and no input portrait.
template <int N>
__global__ void __launch_bounds__(256) k_simulate(SimArgs a, int nsub) {
  using G = RowGeom<N>;
  using T = double;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* twN = reinterpret_cast<cx<T>*>(smem_raw);
  cx<T>* tw2N = twN + N;
  cx<T>* bufs = tw2N + (N / 2 + 2);
  __shared__ float red[2][8];
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  {
    const cx<T>* g1 = reinterpret_cast<const cx<T>*>(a.r.twN);
    const cx<T>* g2 = reinterpret_cast<const cx<T>*>(a.r.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  __syncthreads();   // the packing below reads tw2N[p], stored by other warps (no input load barrier here)
  cx<T>* bufA = bufs + (size_t)r * 2 * N;
  cx<T>* bufB = bufA + N;
  const long nrows = (long)nsub * a.nchan;
  const long row = (long)blockIdx.x * G::kRows + r;
  const bool valid = row < nrows;
  const long rowc = valid ? row : 0;
  const int s = (int)(rowc / a.nchan), ch = (int)(rowc % a.nchan);
  const SimRow w = sim_row(a, s, ch);
#pragma unroll
  for (int i = 0; i < G::kPairs; ++i) {
    const int p = t_row + 1 + i * G::kTRow;
    if (p <= N / 2) {
      const cx<T> dp = sim_harmonic(w, p);
      const cx<T> dq = p < N / 2 ? sim_harmonic(w, N - p) : dp;
      cx<T> zp, zq;
      pack_pair<T>(dp, dq, tw2N[p], zp, zq);
      bufA[p] = cconj(zp);           // conj for the inverse transform
      if (p < N / 2) bufA[N - p] = cconj(zq);
    }
  }
  if (t_row == 0) {
    const T d0 = w.S * w.M[0].x;
    const T dN = sim_harmonic(w, N).x;   // irfft keeps the real part of the Nyquist term
    bufA[0] = mk<T>(T(0.5) * (d0 + dN), -T(0.5) * (d0 - dN));
  }
  __syncthreads();
  const cx<T>* Y = fft_forward<N, G::kTRow, T>(bufA, bufB, twN, t_row);
  const T sc = T(1) / T(N);
  float v[G::kLoads][4];
  float lo = CUDART_INF_F, hi = -CUDART_INF_F;
#pragma unroll
  for (int m = 0; m < G::kLoads; ++m) {
    const int q = t_row + m * G::kTRow;
    const cx<T> y0 = Y[2 * q], y1 = Y[2 * q + 1];
    const double y[4] = {y0.x * sc, -y0.y * sc, y1.x * sc, -y1.y * sc};
    sim_noise(a, w, q, ch, s, y, v[m]);
#pragma unroll
    for (int i = 0; i < 4; ++i) { lo = fminf(lo, v[m][i]); hi = fmaxf(hi, v[m][i]); }
    if (a.out && valid)
      reinterpret_cast<float4*>(a.out + (size_t)row * 2 * N)[q] = make_float4(v[m][0], v[m][1], v[m][2], v[m][3]);
  }
  if (!a.raw) return;   // (uniform over the grid)
#pragma unroll
  for (int o = (G::kTRow < 32 ? G::kTRow : 32) / 2; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if (G::kTRow > 32) {
    if ((tid & 31) == 0) { red[0][tid >> 5] = lo; red[1][tid >> 5] = hi; }
    __syncthreads();
#pragma unroll
    for (int ww = 0; ww < G::kTRow / 32; ++ww) {
      lo = fminf(lo, red[0][r * (G::kTRow / 32) + ww]);
      hi = fmaxf(hi, red[1][r * (G::kTRow / 32) + ww]);
    }
  }
  if (!valid) return;
  const SimQuant qz(lo, hi);
#pragma unroll
  for (int m = 0; m < G::kLoads; ++m) {
    const int q = t_row + m * G::kTRow;
    short4 o4;
    o4.x = qz(v[m][0]); o4.y = qz(v[m][1]); o4.z = qz(v[m][2]); o4.w = qz(v[m][3]);
    reinterpret_cast<short4*>(a.raw + (size_t)row * 2 * N)[q] = o4;
  }
  if (t_row == 0) { a.dat_scl[row] = (float)qz.scl; a.dat_offs[row] = (float)qz.offs; }
}

// Other even nbin, step 1: the spectrum rows Y of a chunk into the any-nbin scratch (slot k = harmonic k, 1..L;
// dc = harmonic 0), for k_inv_any.  One CTA per row.
__global__ void __launch_bounds__(256) k_sim_mul(SimArgs a, cx<double>* spec, double* dc, int Npad, int L) {
  const long row = blockIdx.x;
  const int s = (int)(row / a.nchan), ch = (int)(row % a.nchan);
  const SimRow w = sim_row(a, s, ch);
  for (int k = threadIdx.x + 1; k <= L; k += 256) {
    const cx<double> d = sim_harmonic(w, k);
    spec[(size_t)row * Npad + k] = (k < L) ? d : mk<double>(d.x, 0.0);   // irfft keeps the real part of the Nyquist term
  }
  if (threadIdx.x == 0) dc[row] = w.S * a.mdc[w.mrow];
}

// Other even nbin, step 2: the noise and store epilogue of k_simulate on the float64 rows of k_inv_any.  One CTA per
// row; the row's float32 values wait in shared memory for the int16 pass.
__global__ void __launch_bounds__(256) k_sim_store(SimArgs a, const double* __restrict__ y) {
  __shared__ float vrow[4096];
  __shared__ float red[2][8];
  const long row = blockIdx.x;
  const int s = (int)(row / a.nchan), ch = (int)(row % a.nchan), tid = threadIdx.x, nbin = a.nbin;
  const SimRow w = sim_row(a, s, ch);
  const double* yr = y + (size_t)row * nbin;
  float lo = CUDART_INF_F, hi = -CUDART_INF_F;
  for (int q = tid; 4 * q < nbin; q += 256) {
    const int n = min(4, nbin - 4 * q);   // the last quad is partial when 4 does not divide nbin
    double yq[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = 0; i < n; ++i) yq[i] = yr[4 * q + i];
    float v[4];
    sim_noise(a, w, q, ch, s, yq, v);
    for (int i = 0; i < n; ++i) {
      vrow[4 * q + i] = v[i];
      lo = fminf(lo, v[i]); hi = fmaxf(hi, v[i]);
      if (a.out) a.out[(size_t)row * nbin + 4 * q + i] = v[i];
    }
  }
  if (!a.raw) return;
  for (int o = 16; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((tid & 31) == 0) { red[0][tid >> 5] = lo; red[1][tid >> 5] = hi; }
  __syncthreads();
  for (int ww = 0; ww < 8; ++ww) { lo = fminf(lo, red[0][ww]); hi = fmaxf(hi, red[1][ww]); }
  const SimQuant qz(lo, hi);
  for (int j = tid; j < nbin; j += 256) a.raw[(size_t)row * nbin + j] = qz(vrow[j]);
  if (tid == 0) { a.dat_scl[row] = (float)qz.scl; a.dat_offs[row] = (float)qz.offs; }
}

}  // namespace ppb
