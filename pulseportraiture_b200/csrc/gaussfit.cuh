// Weighted least-squares fit of evolving-Gaussian model portraits (pplib.fit_gaussian_portrait,
// pplib.py:1924-2052), batched over portraits, in FP64 throughout.
//
//   k_gfit_pass<N>   one (portrait, channel) row at a time: the model row g_n and its analytic
//                    local derivative rows are transformed with the double row FFT of fft.cuh,
//                    scattered (and rotated, with join parameters) in the Fourier domain, and the
//                    channel's local normal matrix, J^T r and chi^2 are summed over harmonics in a
//                    fixed order
//   k_gfit_reduce    chain rule: local sums of every channel -> the global P x P system, summed
//                    over channels in channel order (one thread per entry)
//   k_gfit_update    Levenberg-Marquardt with Marquardt scaling, an active set for the bounds,
//                    damped Cholesky, accept / reject by chi^2, and the epilogue (errors, cov)
//
// Parameter vector (P = 3 + 6 ngauss + 2 njoin): [DC, tau [bin at nu_ref], (loc, m_loc, wid, m_wid, amp,
// m_amp) x ngauss, alpha, (phi_j, DM_j) x njoin]; alpha is entry ia = 2 + 6 ngauss.  Local columns of
// channel n (L = 2 + 3 ngauss, plus 1 with joins): 0 = DC, 1 + 3g + q with q = 0 loc_n, 1 wid_n, 2 amp_n
// of component g, 1 + 3 ngauss = tau_n and, with joins, 2 + 3 ngauss = theta_n.
//
// Objective (Parseval, N = nbin/2): chi^2 = sum_n (R_0^2 + 2 sum_{0<k<N} |R_k|^2 + R_N^2) / (nbin sigma_n^2)
// with R = rfft(d) - M, M_0 = G_0, M_k = E_k B_k G_k, M_N = cos(2 pi N theta_n) Re(B_N) G_N,
// B_k = 1 / (1 + 2 pi i k tau_n), E_k = e^{2 pi i k theta_n}: what irfft(B rfft(g)) of gen_gaussian_portrait
// (pplib.py:921-927) does with each harmonic, followed by rotate_data(., phi_j, DM_j, P, freqs, nu_ref) on the
// channels of join group j.  theta_n = phi_j + Dconst DM_j / P (nu_n^-2 - nu_ref^-2) for a channel of group j
// (join_chan[n] = j) and 0 for a channel in no group; dM_k/dtheta_n = 2 pi i k M_k, and at the Nyquist term
// -2 pi N sin(2 pi N theta_n) Re(B_N) G_N.  The restatement is tests/test_cpu_gaussjoin.py.
//
// Size caps: ngauss <= 16, njoin <= 8, so P <= kGfitMaxP = 3 + 6 * 16 + 2 * 8 = 115.  k_gfit_update holds two
// P x P double matrices in dynamic shared memory (2 * 115^2 * 8 = 211600 bytes at the cap) next to its static
// arrays (idx, D, g, dx and flags: 3248 bytes): within the 227 KB a block may opt in to.
#pragma once
#include "kernels.cuh"

namespace ppb {

constexpr int kGfitMaxGauss = 16;
constexpr int kGfitMaxJoin = 8;
constexpr int kGfitMaxP = 3 + 6 * kGfitMaxGauss + 2 * kGfitMaxJoin;   // 115

struct GfitArgs {
  const double* data;    // [nc, nchan, nbin], or null when only the model is written
  const double* errs;    // [nc, nchan]
  const double* freqs;   // [nchan]
  const double* xt;      // [nc, P] point to evaluate
  const int* done;       // [nc] or null: rows of finished portraits are skipped
  double* rec;           // [nc * nchan, S]: packed upper triangle of the (L+1)^2 sums over rows
                         // (r, J_0 .. J_{L-1}), then the P chain coefficients c_n(i)
  double2* slab;         // [gridDim.x, L + 1, N + 1] per-CTA spectrum rows
  double* model;         // [nc, nchan, nbin] or null: write the model portrait at xt instead of sums
  const void* twN;
  const void* tw2N;
  const int* join_chan;  // [nchan] join group of each channel, -1 = none (null when njoin = 0)
  double nu_ref;
  double P_period;       // spin period [s] of the DM chain (njoin > 0)
  int nc, nchan, ngauss, P, L, S;
  int ia;                // index of alpha: 2 + 6 ngauss; the join pairs follow it
  int njoin;
  int code[3];           // loc, wid, amp: 0 power law, 1 linear
};

// index of (u, v), u <= v, in the packed upper triangle of an n x n symmetric matrix
__host__ __device__ __forceinline__ int tri_index(int u, int v, int n) { return u * n - u * (u - 1) / 2 + (v - u); }

// the local column global parameter i maps to (ia = index of alpha = 2 + 6 ngauss; tau_n is local column
// ia / 2 = 1 + 3 ngauss, theta_n the one after it)
__device__ __forceinline__ int gfit_local(int i, int ia) {
  if (i == 0) return 0;
  if (i == 1 || i == ia) return ia / 2;
  if (i > ia) return ia / 2 + 1;           // phi_j, DM_j: through theta_n
  const int j = i - 2;                      // (g, q, e) = component, quantity, evolution term
  return 1 + 3 * (j / 6) + (j % 6) / 2;
}

// kJoin: a.njoin > 0 (a separate instance, so that the unjoined fit carries no join code).  Two CTAs per SM:
// without the bound ptxas caps some instances at 80 registers and spills.
template <int N, bool kJoin>
__global__ void __launch_bounds__(256, 2) k_gfit_pass(GfitArgs a) {
  using G = RowGeom<N>;
  constexpr int nbin = 2 * N;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<double>* twN = reinterpret_cast<cx<double>*>(smem_raw);
  cx<double>* tw2N = twN + N;
  cx<double>* bufs = tw2N + (N / 2 + 2);
  __shared__ double p[kGfitMaxP];
  __shared__ GaussComp comp[kGfitMaxGauss];
  __shared__ double cval[kGfitMaxGauss][3];   // loc_n, wid_n, amp_n
  __shared__ double sh_tau, sh_theta;
  const int tid = threadIdx.x, r = tid / G::kTRow, t_row = tid % G::kTRow;
  const int lane = tid & 31, warp = tid >> 5;
  {
    const cx<double>* g1 = reinterpret_cast<const cx<double>*>(a.twN);
    const cx<double>* g2 = reinterpret_cast<const cx<double>*>(a.tw2N);
    for (int i = tid; i < N; i += 256) twN[i] = g1[i];
    for (int i = tid; i <= N / 2; i += 256) tw2N[i] = g2[i];
  }
  cx<double>* bufA = bufs + (size_t)r * 2 * N;
  cx<double>* bufB = bufA + N;
  const int P = a.P, L = a.L, ng = a.ngauss, ia = a.ia;
  const int Lt = ia / 2 + 1;   // slab row of the tau_n column (L without joins)
  constexpr bool join = kJoin;
  const BinCentres xbin(nbin);
  cx<double>* slab = reinterpret_cast<cx<double>*>(a.slab) + (size_t)blockIdx.x * (L + 1) * (N + 1);
  const long nunits = (long)a.nc * a.nchan;
  for (long unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
    const int s = (int)(unit / a.nchan), ch = (int)(unit % a.nchan);
    if (a.done && a.done[s]) continue;
    const double f = a.freqs[ch];
    const int jg = join ? a.join_chan[ch] : -1;                      // join group of the channel
    const double kdm = join ? kDconst / a.P_period * (1.0 / (f * f) - 1.0 / (a.nu_ref * a.nu_ref)) : 0.0;
    __syncthreads();   // the previous unit is finished with p, comp and the slab
    for (int i = tid; i < P; i += 256) p[i] = a.xt[(size_t)s * P + i];
    __syncthreads();
    for (int g = tid; g < ng; g += 256) {
      const double* q = p + 2 + 6 * g;
      const double loc = evolve_param(f, a.nu_ref, q[0], q[1], a.code[0]);
      const double wid = evolve_param(f, a.nu_ref, q[2], q[3], a.code[1]);
      const double amp = evolve_param(f, a.nu_ref, q[4], q[5], a.code[2]);
      comp[g] = gauss_comp(loc, wid, amp, xbin);
      cval[g][0] = loc; cval[g][1] = wid; cval[g][2] = amp;
    }
    if (tid == 0) {
      sh_tau = (p[1] / (double)nbin) * pow(f / a.nu_ref, p[ia]);   // pplib.py:4049-4053
      double th = 0.0;
      if (jg >= 0) { th = p[ia + 1 + 2 * jg] + p[ia + 2 + 2 * jg] * kdm; th -= rint(th); }
      sh_theta = th;
    }
    __syncthreads();
    // time-domain rows, transformed kRows at a time: j = 0 data -> slab row 0, j = 1 model g -> row L
    // (replaced by the tau_n column, or with joins the theta_n column, below), j = 2 + 3g + q -> row
    // 2 + 3g + q (local column 1 + 3g + q)
    const int nfft = 2 + 3 * ng;
    const double* drow = a.data ? a.data + ((size_t)s * a.nchan + ch) * nbin : nullptr;
    for (int base = 0; base < nfft; base += G::kRows) {
      const int j = base + r;
      auto sample = [&](int t) -> double {
        if (j >= nfft) return 0.0;
        if (j == 0) return drow ? drow[t] : 0.0;
        const double x = xbin(t);
        if (j == 1) {
          double v = p[0];
          for (int g = 0; g < ng; ++g) {
            const GaussComp& c = comp[g];
            if (c.scale == 0.0) continue;
            const double z = c.z(x);
            if (fabs(z) < 20.0) v += c.scale * exp(-0.5 * z * z);
          }
          return v;
        }
        const int g = (j - 2) / 3, q = (j - 2) % 3;
        const GaussComp& c = comp[g];
        if (c.renorm == 0.0) return 0.0;
        const double z = c.z(x);
        if (!(fabs(z) < 20.0)) return 0.0;
        const double e = exp(-0.5 * z * z);
        if (q == 0) return c.scale * e * z * c.isig;      // d/d loc_n
        if (q == 1) return c.scale * e * z * z / cval[g][1];   // d/d wid_n
        return c.renorm * e;                              // d/d amp_n
      };
      for (int m = t_row; m < N; m += G::kTRow) bufA[m] = mk<double>(sample(2 * m), sample(2 * m + 1));
      __syncthreads();
      cx<double>* Z = fft_forward<N, G::kTRow, double>(bufA, bufB, twN, t_row);
      if (j < nfft) {
        cx<double>* out = slab + (size_t)(j == 0 ? 0 : j == 1 ? L : j) * (N + 1);
        for (int pp = t_row + 1; pp <= N / 2; pp += G::kTRow) {
          cx<double> dp, dq;
          unpack_pair<double>(Z, tw2N, N, pp, dp, dq);
          out[pp] = dp;
          if (pp < N / 2) out[N - pp] = dq;
        }
        if (t_row == 0) {
          out[0] = mk<double>(Z[0].x + Z[0].y, 0.0);
          out[N] = mk<double>(Z[0].x - Z[0].y, 0.0);
        }
      }
      __syncthreads();
    }
    // scattering, rotation, residual and weights, harmonic by harmonic
    const double tau_n = sh_tau, theta_n = sh_theta;
    const double sig = a.errs ? a.errs[(size_t)s * a.nchan + ch] : 1.0;   // null: model only
    const double s_mid = sqrt(2.0 / (double)nbin) / sig, s_end = sqrt(1.0 / (double)nbin) / sig;
    for (int k = tid; k <= N; k += 256) {
      cx<double> fB = mk<double>(1.0, 0.0), fT = mk<double>(0.0, 0.0);   // M_k / G_k and dM_k/dtau_n / G_k
      if (k > 0) {
        const double b = kTwoPi * (double)k * tau_n, q = 1.0 / (1.0 + b * b);
        fB = mk<double>(q, -b * q);                                        // 1 / (1 + i b)
        const cx<double> B2 = cmul(fB, fB);
        fT = mk<double>(kTwoPi * (double)k * B2.y, -kTwoPi * (double)k * B2.x);   // -2 pi i k B^2
        if (k == N) { fB.y = 0.0; fT.y = 0.0; }                            // irfft keeps Re of the Nyquist term
      }
      cx<double> fH = mk<double>(0.0, 0.0);                                // dM_k/dtheta_n / G_k
      if (join) {   // E_k = e^{2 pi i k theta_n}; the rotated real row keeps cos(2 pi N theta_n) at the Nyquist term
        double c, sn;
        cis2pi((double)k * theta_n, c, sn);
        const double w = kTwoPi * (double)k;
        if (k == N) {
          fH = mk<double>(-w * sn * fB.x, 0.0);
          fB.x *= c; fT.x *= c;
        } else {
          const cx<double> E = mk<double>(c, sn);
          fB = cmul(fB, E); fT = cmul(fT, E);
          fH = mk<double>(-w * fB.y, w * fB.x);                            // 2 pi i k E_k B_k
        }
      }
      const double sc = (k == 0 || k == N) ? s_end : s_mid;
      const cx<double> Gk = slab[(size_t)L * (N + 1) + k];
      const cx<double> M = cmul(fB, Gk);
      if (a.model) { slab[(size_t)L * (N + 1) + k] = M; continue; }
      const cx<double> D = slab[k];
      slab[k] = mk<double>((D.x - M.x) * sc, (D.y - M.y) * sc);
      const cx<double> T = cmul(fT, Gk);
      slab[(size_t)Lt * (N + 1) + k] = mk<double>(T.x * sc, T.y * sc);
      if (join) {
        const cx<double> H = cmul(fH, Gk);
        slab[(size_t)L * (N + 1) + k] = mk<double>(H.x * sc, H.y * sc);
      }
      slab[(size_t)(N + 1) + k] = mk<double>(k == 0 ? (double)nbin * sc : 0.0, 0.0);   // DC: rfft(1) = nbin at k = 0
      for (int c = 1; c < Lt - 1; ++c) {
        const cx<double> J = cmul(fB, slab[(size_t)(c + 1) * (N + 1) + k]);
        slab[(size_t)(c + 1) * (N + 1) + k] = mk<double>(J.x * sc, J.y * sc);
      }
    }
    __syncthreads();
    if (a.model) {   // irfft of M (as k_rotate): packed conj spectrum, forward transform, conj / N
      const cx<double>* Mr = slab + (size_t)L * (N + 1);
      for (int pp = t_row + 1; pp <= N / 2; pp += G::kTRow) {
        cx<double> zp, zq;
        pack_pair<double>(Mr[pp], pp < N / 2 ? Mr[N - pp] : Mr[pp], tw2N[pp], zp, zq);
        bufA[pp] = cconj(zp);
        if (pp < N / 2) bufA[N - pp] = cconj(zq);
      }
      if (t_row == 0) {
        const double d0 = Mr[0].x, dN = Mr[N].x;
        bufA[0] = mk<double>(0.5 * (d0 + dN), -0.5 * (d0 - dN));
      }
      __syncthreads();
      cx<double>* Y = fft_forward<N, G::kTRow, double>(bufA, bufB, twN, t_row);
      if (r == 0) {
        double* out = a.model + ((size_t)s * a.nchan + ch) * nbin;
        const double inv = 1.0 / (double)N;
        for (int m = t_row; m < N; m += G::kTRow) { out[2 * m] = Y[m].x * inv; out[2 * m + 1] = -Y[m].y * inv; }
      }
      continue;
    }
    // sums over harmonics of Re(conj(row_u) row_v), u <= v, rows (r, J_0, .., J_{L-1}): one warp per
    // entry, lanes in a fixed order, then the warp's fixed-order reduction
    double* rec = a.rec + (size_t)unit * a.S;
    const int nsum = (L + 1) * (L + 2) / 2;
    for (int e = warp; e < nsum; e += 8) {
      int u = 0, rem = e;
      while (rem >= L + 1 - u) { rem -= L + 1 - u; ++u; }
      const int v = u + rem;
      const cx<double>* ru = slab + (size_t)u * (N + 1);
      const cx<double>* rv = slab + (size_t)v * (N + 1);
      double acc = 0.0;
      for (int k = lane; k <= N; k += 32) acc = fma(ru[k].x, rv[k].x, fma(ru[k].y, rv[k].y, acc));
      acc = warp_sum(acc);
      if (lane == 0) rec[e] = acc;
    }
    // chain coefficients d(local column) / d(global parameter) of this channel
    for (int i = tid; i < P; i += 256) {
      const double lr = log(f) - log(a.nu_ref);
      double c;
      if (i == 0) c = 1.0;
      else if (i == 1) c = pow(f / a.nu_ref, p[ia]) / (double)nbin;
      else if (i == ia) c = tau_n * lr;
      else if (i > ia) {   // phi_j, DM_j: d theta_n on the channels of group j, 0 elsewhere
        const int jj = (i - ia - 1) / 2;
        c = jg != jj ? 0.0 : ((i - ia - 1) % 2 == 0 ? 1.0 : kdm);
      } else {
        const int j = i - 2, g = j / 6, q = (j % 6) / 2, ev = j % 2;
        if (a.code[q] == 1) c = ev ? f - a.nu_ref : 1.0;
        else c = ev ? cval[g][q] * lr : exp(lr * p[i + 1]);   // (nu/nu_ref)^m, x_n ln(nu/nu_ref)
      }
      rec[nsum + i] = c;
    }
  }
}

struct GfitState {
  double* x;       // [nc, P] current (accepted) point
  double* xt;      // [nc, P] trial point (evaluated by the next pass)
  double* jtj_t;   // [nc, P, P] at the trial point (k_gfit_reduce)
  double* jtr_t;   // [nc, P]
  double* chi2_t;  // [nc]
  double* jtj;     // [nc, P, P] at x
  double* jtr;     // [nc, P]
  double* chi2;    // [nc]
  double* lam;     // [nc]
  int* nfev;       // [nc]
  int* done;       // [nc]
};

// global normal matrix, J^T r and chi^2 at the trial point of every running portrait; entries of fixed
// parameters are 0.  Thread e of portrait s sums entry e over the channels in channel order.
__global__ void __launch_bounds__(256) k_gfit_reduce(GfitArgs a, GfitState st, const uint8_t* free_) {
  const int s = blockIdx.y, P = a.P, L = a.L;
  if (st.done[s]) return;
  const int e = blockIdx.x * 256 + threadIdx.x;
  const int npair = P * (P + 1) / 2;
  if (e > npair + P) return;
  const int nsum = (L + 1) * (L + 2) / 2;
  const double* rec = a.rec + (size_t)s * a.nchan * a.S;
  double acc = 0.0;
  if (e == npair + P) {
    for (int n = 0; n < a.nchan; ++n) acc += rec[(size_t)n * a.S];
    st.chi2_t[s] = acc;
    return;
  }
  if (e >= npair) {
    const int i = e - npair;
    if (free_[i]) {
      const int t = tri_index(0, 1 + gfit_local(i, a.ia), L + 1);
      for (int n = 0; n < a.nchan; ++n) { const double* rn = rec + (size_t)n * a.S; acc += rn[nsum + i] * rn[t]; }
    }
    st.jtr_t[(size_t)s * P + i] = acc;
    return;
  }
  int i = 0, rem = e;
  while (rem >= P - i) { rem -= P - i; ++i; }
  const int j = i + rem;
  if (free_[i] && free_[j]) {
    const int u = 1 + gfit_local(i, a.ia), v = 1 + gfit_local(j, a.ia);
    const int t = u <= v ? tri_index(u, v, L + 1) : tri_index(v, u, L + 1);
    for (int n = 0; n < a.nchan; ++n) {
      const double* rn = rec + (size_t)n * a.S;
      acc += rn[nsum + i] * rn[nsum + j] * rn[t];
    }
  }
  st.jtj_t[((size_t)s * P + i) * P + j] = acc;
  st.jtj_t[((size_t)s * P + j) * P + i] = acc;
}

// ---- dense symmetric solves of one CTA on shared memory (n <= kGfitMaxP) ----

// in-place Cholesky A = L L^T of the n x n matrix A (row stride n, lower triangle used); false if A is
// not positive definite.  Each element is updated in the same order whatever the thread count.
__device__ bool gfit_chol(double* A, int n, int* flag) {
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int k = 0; k < n; ++k) {
    if (tid == 0) {
      const double d = A[k * n + k];
      *flag = d > 0.0 && isfinite(d);
      A[k * n + k] = sqrt(d);
    }
    __syncthreads();
    if (!*flag) return false;
    const double lkk = A[k * n + k];
    for (int i = k + 1 + tid; i < n; i += nt) A[i * n + k] /= lkk;
    __syncthreads();
    const int m = n - k - 1;
    for (int e = tid; e < m * m; e += nt) {
      const int i = k + 1 + e / m, j = k + 1 + e % m;
      if (j <= i) A[i * n + j] -= A[i * n + k] * A[j * n + k];
    }
    __syncthreads();
  }
  return true;
}

// B = L^{-1} (lower triangle, row stride n) from the factor in A: thread i solves for column i
__device__ void gfit_linv(const double* A, double* B, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    for (int r = 0; r < i; ++r) B[r * n + i] = 0.0;
    B[i * n + i] = 1.0 / A[i * n + i];
    for (int r = i + 1; r < n; ++r) {
      double acc = 0.0;
      for (int k = i; k < r; ++k) acc = fma(A[r * n + k], B[k * n + i], acc);
      B[r * n + i] = -acc / A[r * n + r];
    }
  }
  __syncthreads();
}

// x = (L L^T)^{-1} b by forward and back substitution (one thread; O(n^2))
__device__ void gfit_solve(const double* A, int n, const double* b, double* x) {
  for (int i = 0; i < n; ++i) {
    double acc = b[i];
    for (int k = 0; k < i; ++k) acc -= A[i * n + k] * x[k];
    x[i] = acc / A[i * n + i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double acc = x[i];
    for (int k = i + 1; k < n; ++k) acc -= A[k * n + i] * x[k];
    x[i] = acc / A[i * n + i];
  }
}

struct GfitUpdateArgs {
  const uint8_t* free_;   // [P]
  const double* lo;       // [P] lower bounds (-inf: none)
  const double* hi;       // [P]
  int P, max_iter;
  double tol, ndata;      // ndata = nchan * nbin
  int* running;           // count of portraits still running after this update
  // outputs for the chunk's portraits (row s of each)
  double *params, *errs, *cov, *chi2, *red_chi2, *jtr, *jtj;
  int *nfeval, *rc;
};

constexpr double kGfitLam0 = 1e-3;
constexpr double kGfitChi2Slack = 1e-12;

// one CTA per SM (up to 211600 bytes of dynamic shared memory); the bound lets ptxas keep it free of spills
__global__ void __launch_bounds__(256, 1) k_gfit_update(GfitState st, GfitUpdateArgs u) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int s = blockIdx.x, P = u.P, tid = threadIdx.x;
  if (st.done[s]) return;
  double* A = reinterpret_cast<double*>(smem_raw);   // [P, P]
  double* B = A + P * P;                             // [P, P]
  __shared__ int idx[kGfitMaxP];
  __shared__ double D[kGfitMaxP], g[kGfitMaxP], dx[kGfitMaxP];
  __shared__ int n_sh, flag, accept_sh, finish_sh;
  double* x = st.x + (size_t)s * P;
  double* xt = st.xt + (size_t)s * P;
  double* jtj = st.jtj + (size_t)s * P * P;
  double* jtr = st.jtr + (size_t)s * P;
  int nfree = 0;
  for (int i = 0; i < P; ++i) nfree += u.free_[i] ? 1 : 0;
  const int nfev = st.nfev[s] + 1;
  const double chi2t = st.chi2_t[s];
  if (tid == 0) {
    const bool first = nfev == 1;
    st.nfev[s] = nfev;
    // a trial may raise chi^2 by its own rounding (~1e-13 relative over nchan * nbin terms): near the optimum
    // the change a 1e-4 sigma step makes is no larger, and rejecting on rounding would stall the fit
    int acc = isfinite(chi2t) && (first || chi2t <= st.chi2[s] + kGfitChi2Slack * fabs(st.chi2[s]));
    int fin = -1;                                    // return code when the fit ends in this update
    if (first && !isfinite(chi2t)) { fin = 3; acc = 1; }
    if (u.max_iter < 0) { fin = 0; acc = 1; }
    if (acc) {
      if (!first) st.lam[s] = fmax(st.lam[s] * 0.1, 1e-12);
    } else {
      st.lam[s] *= 10.0;
    }
    accept_sh = acc; finish_sh = fin;
  }
  __syncthreads();
  if (accept_sh) {
    for (int i = tid; i < P; i += 256) { x[i] = xt[i]; jtr[i] = st.jtr_t[(size_t)s * P + i]; }
    for (int i = tid; i < P * P; i += 256) jtj[i] = st.jtj_t[(size_t)s * P * P + i];
    if (tid == 0) st.chi2[s] = chi2t;
  }
  __syncthreads();
  const double chi2 = st.chi2[s];
  const double red = chi2 / (u.ndata - (double)nfree);
  int fin = finish_sh;
  // the system of the free parameters that may move: a parameter on a bound whose gradient pushes
  // outwards (J^T r points out of the box) is held there for this step.  A parameter whose Jacobian
  // column is zero at x (alpha while tau = 0, the parameters of a component of zero width or amplitude
  // under a power law) is left out of the step and of the covariance, whose row and column for it stay 0
  // (MINPACK's covar convention for columns of zero norm)
  auto build = [&](bool active_only, double lam) {
    if (tid == 0) {
      int n = 0;
      for (int i = 0; i < P; ++i) {
        if (!u.free_[i] || !(jtj[i * P + i] > 0.0)) continue;
        if (active_only && ((x[i] <= u.lo[i] && jtr[i] < 0.0) || (x[i] >= u.hi[i] && jtr[i] > 0.0))) continue;
        idx[n++] = i;
      }
      n_sh = n;
    }
    __syncthreads();
    const int n = n_sh;
    for (int a = tid; a < n; a += 256) {
      const double d = jtj[idx[a] * P + idx[a]];
      D[a] = 1.0 / sqrt(d);                            // Marquardt scaling: unit diagonal
      g[a] = jtr[idx[a]] * D[a];
    }
    __syncthreads();
    for (int e = tid; e < n * n; e += 256) {
      const int a = e / n, b = e % n;
      A[e] = jtj[idx[a] * P + idx[b]] * D[a] * D[b] + (a == b ? lam : 0.0);
    }
    __syncthreads();
    return n;
  };
  if (fin < 0 && accept_sh) {   // converged when every Gauss-Newton step is below tol x its sigma
    const int n = build(true, 0.0);
    if (n == 0) fin = 0;
    else if (gfit_chol(A, n, &flag)) {
      if (tid == 0) gfit_solve(A, n, g, dx);
      gfit_linv(A, B, n);
      if (tid == 0) {
        bool conv = true;
        for (int a = 0; a < n; ++a) {
          double vi = 0.0;
          for (int r = a; r < n; ++r) vi += B[r * n + a] * B[r * n + a];
          const double step = fabs(dx[a] * D[a]), sigma = D[a] * sqrt(vi * red);
          if (!(step < u.tol * sigma || step <= 4e-16 * fabs(x[idx[a]]))) conv = false;
        }
        flag = conv;
      }
      __syncthreads();
      if (flag) fin = 0;
    }
  }
  if (fin < 0 && nfev >= u.max_iter) fin = 1;
  if (fin < 0) {   // damped step, clipped to the box
    double lam = st.lam[s];
    for (int tries = 0; tries < 8; ++tries, lam *= 10.0) {
      const int n = build(true, lam);
      if (gfit_chol(A, n, &flag)) {
        if (tid == 0) {
          gfit_solve(A, n, g, dx);
          for (int i = 0; i < P; ++i) xt[i] = x[i];
          for (int a = 0; a < n; ++a) {
            const int i = idx[a];
            xt[i] = fmin(fmax(x[i] + dx[a] * D[a], u.lo[i]), u.hi[i]);
          }
          st.lam[s] = lam;
          flag = 1;
        }
        __syncthreads();
        break;
      }
      if (tid == 0) flag = 0;
      __syncthreads();
    }
    if (!flag) fin = 3;
    if (fin < 0) {
      if (tid == 0) atomicAdd(u.running, 1);
      return;
    }
  }
  // epilogue at x: errors and covariance from the normal matrix of every free parameter, scaled by
  // red_chi2 (lmfit's scale_covar)
  const int n = build(false, 0.0);
  const bool ok = n > 0 && gfit_chol(A, n, &flag);
  if (ok) gfit_linv(A, B, n);
  double* cov = u.cov ? u.cov + (size_t)s * P * P : nullptr;
  if (cov) for (int e = tid; e < P * P; e += 256) cov[e] = 0.0;
  if (u.jtj) for (int e = tid; e < P * P; e += 256) u.jtj[(size_t)s * P * P + e] = jtj[e];
  __syncthreads();
  for (int e = tid; e < n * n; e += 256) {
    const int a = e / n, b = e % n;
    double c = CUDART_NAN;
    if (ok) {
      c = 0.0;
      for (int r = a > b ? a : b; r < n; ++r) c = fma(B[r * n + a], B[r * n + b], c);
      c *= D[a] * D[b] * red;
    }
    if (cov) cov[idx[a] * P + idx[b]] = c;
    if (a == b && u.errs) u.errs[(size_t)s * P + idx[a]] = sqrt(c);
  }
  for (int i = tid; i < P; i += 256) {
    if (u.params) u.params[(size_t)s * P + i] = x[i];
    if (u.errs && !(u.free_[i] && jtj[i * P + i] > 0.0)) u.errs[(size_t)s * P + i] = 0.0;
    if (u.jtr) u.jtr[(size_t)s * P + i] = jtr[i];
  }
  if (tid == 0) {
    if (u.chi2) u.chi2[s] = chi2;
    if (u.red_chi2) u.red_chi2[s] = red;
    if (u.nfeval) u.nfeval[s] = nfev;
    if (u.rc) u.rc[s] = fin;
    st.done[s] = 1;
  }
}

}  // namespace ppb
