// k_spectra16: K1 + K2 for nbin = 2048 (N = 1024), the configuration the headline metric is quoted on, and the
// only kernel that transforms rows of that size.  The same work as k_spectra (kernels.cuh) on the radix-16 plan
// of fft16.cuh, written around what bounds it on B200: the warp schedulers' issue slots.  An FP64 instruction
// holds the dispatch port of its SM sub-partition for two cycles and every other instruction for one
// (tools/micro/cvt_probe.cu), so a row costs 2 * n_fp64 + n_other slots per thread.  Run inside the generic
// k_spectra, this plan spent ~790 non-FP64 instructions per thread and row, a third of them on shared-memory
// addresses and on predicated-off code.  Here
//   * every shared-memory address is a per-thread base plus an immediate: the XOR swizzle of a pass is split
//     into its per-thread part (folded into a handful of base offsets, recomputed once per row) and its
//     compile-time part,
//   * unused (masked / out of range) rows take one uniform branch instead of predicated zero fills,
//   * the kernel is specialised at compile time on what the call needs (FFTFIT guess accumulators, kept data
//     spectra for the fused ppalign sum, 16-bit samples), the DM_guess rotation stays a rare uniform branch,
//   * the per-row power sums go to a small per-row table in shared memory (no latch code in the row loop),
//   * the conj(model) row of the channel arrives by its own TMA bulk copy into shared memory instead of
//     16 L2 loads per thread held in 32 registers across the last transform pass (those loads alone cost
//     12 % of the kernel: profiles/r02_spectra_experiments.md); the raw row is single buffered (its copy
//     for row r + 1 is issued as soon as row r sits in registers, a whole row time before it is needed),
//     so the shared-memory footprint and the 6 CTAs per SM stay as they were.
// Layout of the twiddle table and of the outputs: exactly SpecPlan16's (spectra_plan.cuh, tw_host.h).
#pragma once

namespace ppb {

constexpr int kSpec16MaxRows = 32;   // rows per CTA (host: rows_per_cta <= 32)

// element index -> position in the row buffer (16-byte elements): i ^ ((i >> 4) & 7), as phys16()
//   pass 1 writes  i = 16 t + k        -> 16 t + (k ^ (t & 7))
//   pass 2 reads   i = t + 64 r        -> ((t ^ (t >> 4)) ^ 4 (r & 1)) + 64 r
//   pass 2 writes  i = 256 b + k + 16 r (b = t >> 4, k = t & 15) -> 256 b + 16 r + (k ^ (r & 7))
//   split reads    i = p + 256 c       -> (p ^ ((p >> 4) & 7)) + 256 c

template <bool I16, bool GUESS, bool KEEPD>
__global__ void __launch_bounds__(64, SpecPlan16::kMinBlocks) k_spectra16(SpectraArgs a) {
  using F = double;
  using PL = SpecPlan16;
  constexpr int N = 1024, T = 64, kLo = LoK<N>::value;
  static_assert(kLo == T, "every thread owns exactly one lo slot (slot t)");
  constexpr unsigned kRowBytes = 2 * N * (I16 ? sizeof(short) : sizeof(float));
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<F>* tw = reinterpret_cast<cx<F>*>(smem_raw);                       // [16] e^{-2 pi i k/256}, [129] e^{-2 pi i p/2048}
  cx<F>* buf = tw + ((PL::kTwTotal + 1) & ~1);                          // [N]
  float* stage = reinterpret_cast<float*>(buf + N);                     // [2N] raw row
  cx<float>* mstage = reinterpret_cast<cx<float>*>(stage + 2 * N);      // [N] conj(model spectrum) of the row's channel
  __shared__ double2 rowsum[kSpec16MaxRows][2];                         // per row and warp: sum |d|^2, top-quarter sum
  __shared__ __align__(8) unsigned long long mbar[2];
  const int t = threadIdx.x;
  for (int i = t; i < PL::kTwTotal; i += T) tw[i] = a.tw8[i];
  if (t == 0) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); }
  mbar_fence_init();
  __syncthreads();

  const int sl = blockIdx.y, s = a.s0 + sl;
  const int mb = KEEPD ? 0 : a.mr.row0(s);   // the subint's model (the fused ppalign sum takes one model)
  const int ch_begin = blockIdx.x * a.G;
  const int ch_end = min(ch_begin + a.G, a.nchan);
  const int nsteps = ch_end - ch_begin;
  constexpr int ntop = N + 1 - 3 * (N / 4);            // harmonics >= int(0.75 nharm), pplib.py:2244
  double Dfac = 0.0, numean2 = 0.0;
  if constexpr (GUESS) {
    const double dmg = a.DMg ? a.DMg[s] : 0.0;
    Dfac = dmg != 0.0 ? kDconst * dmg / a.P[s] : 0.0;  // pplib.py:2381
    const double numean = a.nu_mean[s];
    numean2 = 1.0 / (numean * numean);
  }
  float2 acc[GUESS ? 16 : 1];
  if constexpr (GUESS) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = make_float2(0.f, 0.f);
  }
  const bool first = (t == 0);
  auto row_used = [&](int step) -> bool {
    if (step >= nsteps) return false;
    return a.mask ? (a.mask[(size_t)s * a.nchan + ch_begin + step] != 0) : true;
  };
  auto fetch = [&](int step) {   // TMA producer: bulk-copy the raw row into the staging buffer
    if (t == 0 && row_used(step)) {
      mbar_expect_tx(&mbar[0], kRowBytes);
      bulk_g2s(stage, static_cast<const char*>(a.data) + ((size_t)s * a.nchan + ch_begin + step) * kRowBytes, kRowBytes, &mbar[0]);
    }
  };
  auto fetch_model = [&](int ch) {   // ... and the float conj(model) row of channel ch
    if (t == 0) {
      mbar_expect_tx(&mbar[1], N * (unsigned)sizeof(cx<float>));
      bulk_g2s(mstage, a.mconj32 + (size_t)(mb + ch) * N, N * (unsigned)sizeof(cx<float>), &mbar[1]);
    }
  };
  fetch(0);
  unsigned ph0 = 0u, ph1 = 0u;
  const int kk = t & 15, bb = t >> 4;

  for (int step = 0; step < nsteps; ++step) {
    const int ch = ch_begin + step;
    const size_t row = (size_t)sl * a.nchan + ch;
    float2* const Xrow = a.X + row * N;
    if (!row_used(step)) {          // uniform over the CTA: zeros for the solver, nothing else
      if (a.X != nullptr) {
#pragma unroll
        for (int r = 0; r < 16; ++r) Xrow[t + 64 * r] = make_float2(0.f, 0.f);
        a.Xlo[row * kLo + t] = make_float2(0.f, 0.f);
      }
      if constexpr (KEEPD) {        // k_align_spec prefetches every row of the chunk: keep the skipped ones defined
#pragma unroll
        for (int r = 0; r < 16; ++r) a.D[row * N + t + 64 * r] = make_float2(0.f, 0.f);
        if (t == 0) a.Ddc[row] = 0.0;
      }
      if (t < 2) rowsum[step][t] = make_double2(0.0, 0.0);
      fetch(step + 1);              // the staging buffer is free (nothing was copied for this row)
      continue;
    }
    mbar_wait(&mbar[0], ph0); ph0 ^= 1u;

    // ---- pass 1: 16 samples t + 64 r of the packed row -> registers -> DFT16 -> buf[16 t + k] --------
    cx<F> v[16];
    {
      const float* graw = stage;
      if constexpr (I16) {
        const size_t o = (size_t)s * a.nchan + ch;
        const float scl = a.dat_scl[o], offs = a.dat_offs[o];
        const short2* g = reinterpret_cast<const short2*>(graw) + t;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          const short2 x = g[64 * r];
          v[r] = mk<F>((F)__fadd_rn(__fmul_rn((float)x.x, scl), offs), (F)__fadd_rn(__fmul_rn((float)x.y, scl), offs));
        }
      } else {
        const float2* g = reinterpret_cast<const float2*>(graw) + t;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          const float2 x = g[64 * r];
          v[r] = mk<F>((F)x.x, (F)x.y);
        }
      }
    }
    __syncthreads();   // staged row consumed; the previous row's split reads of buf and of the model row are done
    fetch(step + 1);
    const bool doX = a.X != nullptr;
    const int kcut = a.njn ? 16 * a.njn[mb + ch] : N;
    if (doX) fetch_model(ch);
    dft16(v);
    {
      cx<F>* const w0 = buf + 16 * t;
      const int c = t & 7;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        cx<F>* const wj = w0 + (j ^ c);        // 8 per-thread offsets; k and k + 8 share one
        wj[0] = v[dft16_at(j)];
        wj[8] = v[dft16_at(j + 8)];
      }
    }
    __syncthreads();
    // ---- pass 2: buf[t + 64 r] -> twiddles w^r, DFT16 -> buf[256 b + k + 16 r] -------------------------
    {
      const int te = t ^ bb;                    // per-thread part of the swizzle; odd r flips bit 2
      const cx<F>* const re = buf + te;
      const cx<F>* const ro = buf + (te ^ 4);
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = ((r & 1) ? ro : re)[64 * r];
    }
    __syncthreads();
    // conj(model spectrum) of this thread's harmonics: L2 loads issued here so that their latency hides
    // behind the butterflies.  Output q = 2 j of unit i is harmonic p + 256 j, q = 2 j + 1 is N - p - 256 j
    // (p = t + 64 i; the special unit of thread 0 uses p = 0 / 128).
    cx<F> mc64 = mk<F>(0.5, 0.25);
    const int po0 = first ? 128 : t;           // the odd outputs of unit 0
    if (doX) mc64 = a.mconj64[(size_t)(mb + ch) * N + t];   // the one double-precision factor (lo slot t)
    float wgt = 0.f;
    double shift = 0.0;
    if constexpr (GUESS) {
      wgt = (float)(a.weights ? a.weights[(size_t)s * a.nchan + ch] : 1.0);
      shift = Dfac != 0.0 ? Dfac * (a.nu2[mb + ch] - numean2) : 0.0;
    }
    twiddle16(v, tw[kk]);
    dft16(v);
    {
      cx<F>* const w0 = buf + 256 * bb;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        cx<F>* const wj = w0 + (kk ^ j);        // rows r = j and r = j + 8 share the offset k ^ (r & 7)
        wj[16 * j] = v[dft16_at(j)];
        wj[16 * (j + 8)] = v[dft16_at(j + 8)];
      }
    }
    __syncthreads();

    // ---- last radix-4 pass fused with the real-FFT split; power sums; X; guess accumulators -------------
    double s_all = 0.0, s_top = 0.0;
    float wrow = wgt;
    if (doX) { mbar_wait(&mbar[1], ph1); ph1 ^= 1u; }   // the model row has landed long ago
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int p = t + 64 * i;
      cx<F> d[8];
      F dc_term = F(0);
      if (i == 0 && first) dc_term = split_oct0<F>(buf, tw + PL::kSplitOff, d);
      else {
        const int q0 = 256 - p;
        split16_general<F>(buf + (p ^ ((p >> 4) & 7)), buf + (q0 ^ ((q0 >> 4) & 7)), tw[PL::kSplitOff + p], d);
      }
      // a NaN / Inf sample makes every harmonic of the row non-finite: such a row must not enter the
      // profile for the FFTFIT guess (its sigma comes out non-finite, so the fit skips it too)
      if constexpr (GUESS) { if (i == 0 && !(isfinite(d[0].x) && isfinite(d[0].y))) wrow = 0.f; }
      float vx[8], vy[8];
      double sa0 = 0.0, sa1 = 0.0;      // two chains: the power sum is latency, not throughput, bound
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        double& sa = (q & 1) ? sa1 : sa0;
        if (q == 1 || q == 6 || q == 0) {           // outputs that can be in the top quarter
          const double pw = fma(d[q].x, d[q].x, d[q].y * d[q].y);
          sa += pw;
          if (PL::top(i, q, first)) s_top += pw;    // harmonics >= 3N/4
        } else {
          sa = fma(d[q].x, d[q].x, sa);
          sa = fma(d[q].y, d[q].y, sa);
        }
        vx[q] = (float)d[q].x; vy[q] = (float)d[q].y;
      }
      s_all += sa0 + sa1;
      const int po = (i == 0) ? po0 : p;
      if (doX) {
        float2* const Xe = Xrow + p;
        float2* const Xo = Xrow + (N - po);
        const cx<float>* const Me = mstage + p;
        const cx<float>* const Mo = mstage + (N - po);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float2* const dst = (q & 1) ? Xo - 256 * (q >> 1) : Xe + 256 * (q >> 1);
          // slots at and above the model's harmonic cut-off are never read (slot 0 of the special unit is the
          // Nyquist term: read only when nothing is cut)
          if (((q & 1) ? N - po - 256 * (q >> 1) : p + 256 * (q >> 1)) >= kcut) continue;
          if (i == 0 && q == 0) {                   // slot t < 64: double product, float value + float residual
            const cx<F> pr = cmul(d[0], mc64);
            const float2 xv = make_float2((float)pr.x, (float)pr.y);
            *dst = xv;
            a.Xlo[row * kLo + t] = make_float2((float)(pr.x - (double)xv.x), (float)(pr.y - (double)xv.y));
          } else {
            const cx<float> m = *((q & 1) ? Mo - 256 * (q >> 1) : Me + 256 * (q >> 1));
            *dst = make_float2(fmaf(vx[q], m.x, -vy[q] * m.y), fmaf(vx[q], m.y, vy[q] * m.x));
          }
        }
      }
      if constexpr (KEEPD) {     // raw spectra for k_align_spec (unused rows are skipped there)
        float2* const De = a.D + row * N + p;
        float2* const Do = a.D + row * N + (N - po);
#pragma unroll
        for (int q = 0; q < 8; ++q) *((q & 1) ? Do - 256 * (q >> 1) : De + 256 * (q >> 1)) = make_float2(vx[q], vy[q]);
        if (i == 0 && first) a.Ddc[row] = dc_term;
      }
      if constexpr (GUESS) {
        if (shift != 0.0) {           // rotate_data with DM_guess (pptoas.py:422); uniform, rare
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const int sk = (q & 1) ? N - po - 256 * (q >> 1) : p + 256 * (q >> 1);
            const float2 r = rot2pi(vx[q], vy[q], (double)(sk == 0 ? N : sk) * shift);
            vx[q] = r.x; vy[q] = sk == 0 ? 0.f : r.y;   // the Nyquist term keeps its real part (irfft of rotate_data)
          }
        }
        if (wrow != 0.f) {   // uniform: 0 when the row is not finite
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            acc[8 * i + q].x = fmaf(wrow, vx[q], acc[8 * i + q].x);
            acc[8 * i + q].y = fmaf(wrow, vy[q], acc[8 * i + q].y);
          }
        }
      }
    }
    s_all = warp_sum(s_all); s_top = warp_sum(s_top);
    if ((t & 31) == 0) rowsum[step][t >> 5] = make_double2(s_all, s_top);
  }
  // ---- noise, Sd, S: one row per thread, so that the sqrt and the two divisions are off the per-row
  // critical path ------------------------------------------------------------------------------------
  __syncthreads();
  if (t < nsteps) {
    const int fch = ch_begin + t;
    const bool fused = row_used(t);
    const double keep_all = rowsum[t][0].x + rowsum[t][1].x, keep_top = rowsum[t][0].y + rowsum[t][1].y;
    double sig;
    if (a.errs) sig = fused ? a.errs[(size_t)s * a.nchan + fch] : 0.0;
    else sig = sqrt(keep_top / ((double)(2 * N) * (double)ntop));      // pplib.py:2243-2245
    const double sF2 = sig * sig * (double)N;                           // sigma^2 * nbin/2
    const bool ok = fused && (sF2 > 0.0) && (sF2 < 1e300);
    const size_t o = (size_t)s * a.nchan + fch;
    a.sigma[o] = ok ? sig : 0.0;
    a.Ssn[o] = ok ? a.pn[mb + fch] / sF2 : 0.0;
    a.Sdn[o] = ok ? keep_all / sF2 : 0.0;
  }
  if constexpr (GUESS) {
    float2* const pr = a.partial + ((size_t)sl * a.nparts + blockIdx.x) * N;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int p = t + 64 * i, po = (i == 0 && first) ? 128 : p;
#pragma unroll
      for (int q = 0; q < 8; ++q) pr[(q & 1) ? N - po - 256 * (q >> 1) : p + 256 * (q >> 1)] = acc[8 * i + q];
    }
  }
}

}  // namespace ppb
