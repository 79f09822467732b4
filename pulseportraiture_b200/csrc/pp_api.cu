// C-ABI implementation (see include/ppb200.h).  Host orchestration of the
// sm_100a kernels in kernels.cuh: plan / workspace management, chunked
// pipeline, pointer staging, timing.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ppb200.h"
#include "kernels.cuh"
#include "gaussfit.cuh"
#include "pca.cuh"
#include "tw_host.h"

using namespace ppb;

// ----------------------------------------------------------------------------
// error handling
// ----------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess)                                                               \
      return fail(-2, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

extern "C" const char* pp_last_error(void) { return g_err.c_str(); }

extern "C" void* pp_host_alloc(uint64_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    fail(-2, "cudaHostAlloc(%llu) failed", (unsigned long long)bytes);
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
extern "C" void pp_host_free(void* p) { if (p) cudaFreeHost(p); }
extern "C" int pp_abi_version(void) { return PPB200_ABI_VERSION; }

// ----------------------------------------------------------------------------
// device buffer that grows on demand
// ----------------------------------------------------------------------------
struct DBuf {
  void* p = nullptr;
  size_t cap = 0;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  DBuf(DBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  ~DBuf() { release(); }
  cudaError_t need(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    release();
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <typename T> T* as() { return reinterpret_cast<T*>(p); }
};

struct pp_plan {
  int nchan = 0, nbin = 0, N = 0, device = 0;
  // arbitrary (even, non power-of-two) nbin: rows are transformed by Bluestein kernels (bluestein.cuh) into an
  // FP64 spectrum scratch of N = Npad slots per row; L = nbin/2 is the true number of harmonics, M the FFT length
  // pageable host input: pieces are copied into a ring of page-locked buffers by several host threads
  // and sent from there (a plain cudaMemcpyAsync from pageable memory stages through one thread: ~10 GB/s)
  static const int kPinSlots = 4;
  static const size_t kPinPiece = 32u << 20;
  void* pin_ring[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t pin_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned long pin_count = 0;
  bool anyn = false;
  int L = 0, M = 0;
  DBuf any_chirp, any_B, any_twM, any_tw2n, any_twL, any_spec, any_dc, any_spec2, any_dc2;
  std::vector<int> any_rad;   // radices of the direct transform of length L (empty: Bluestein)
  cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev_copy[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  int chunk_req = 0;
  int l2_bytes = 0, sm_count = 0;
  bool model_set = false;
  int nmodel = 0;   // models set (pp_set_models): the model-side buffers hold nmodel * nchan rows (kernels.cuh ModelRows)
  // tables + model
  DBuf tw8, twN32, tw2N32, twN64, tw2N64, freqs, nu2, lgf, gm_params, gm_taus, gm_zero, gm_one, mconj32, mconj64, mpow, pn, mmean, mmean_sub, model_stage, model_stage64;
  int fft_precision = 0;   // 0 auto, 32, 64
  int model_steps = 8;     // (phi, DM) solver: Newton steps on the local fourth-order model per pass
  double cutoff_eps2 = 1e-20;  // harmonics outside which the model holds less than this share of its k^2-weighted power are skipped
  std::vector<int> kmax_used;  // per model: 16 x the largest per-channel cut-off
  DBuf kmax_dev;               // ... on the device (the FFTFIT guess of a batch with several models)
  double x_keep = 1.0;         // ... which leaves this share of the cross-spectrum to compute, store and stream
  double coarse_frac = 0.99;   // general solver: share of the model's phase information the coarse objective keeps
  std::vector<double> model_info;   // per group of 16 harmonics (scratch of the per-chunk choice)
  bool freqs_set = false;
  // FFTFIT grid tables keyed by Ns
  std::vector<std::pair<int, DBuf>> grid_tables;
  DBuf grid_general;   // table of the last grid with bounds other than [-0.5, 0.5]
  // per-batch staging of small inputs and per-subint / per-channel workspace
  DBuf running, minfo, njn, coarse_first, coarse_njm, in_scat, in_scl, in_offs, in_P, in_errs, in_mask, in_w, in_init, in_dmg, in_snrs, in_nufits, in_nuouts, in_noise, in_models;
  DBuf nu_fit, nu_mean, wsum, nok, sigma, Ssn, Sdn, csum;
  DBuf st_x, st_xprev, st_step, st_fprev, st_lam, st_iter, st_iterc, st_done;
  DBuf o_params, o_perrs, o_nuout, o_cov, o_chi2, o_rchi2, o_snr, o_nfev, o_rc, o_scales, o_serrs, o_csnr, o_lag, o_phig;
  DBuf resp, rot_gm, rot_nugm, al_w, al_out, al_wsum, ps_phase, ps_perr, ps_scale, ps_serr, ps_snr, ps_rchi2, ps_lag, ps_spec, ps_mspec, ps_noise, rot_in, rot_out,
      rot_phase, rot_dm, rot_P, rot_nuref;
  // chunk-sized
  DBuf X, Xlo, partial, data_stage[2], data_stage64[2], Dspec, Ddc, al_acc, al_wparts, al_dc;
  // evolving-Gaussian portrait fit (pp_fit_gaussian_portraits): per-chunk state and outputs, per-CTA slabs
  DBuf gf_data, gf_errs, gf_rec, gf_slab, gf_state, gf_out, gf_model, gf_par;
  // simulated archives (pp_simulate_batch): the call's models, spectra and tables, staged inputs, chunk scratch
  DBuf sim_models, sim_freqs, sim_nu2, sim_mspec, sim_mdc, sim_index, sim_par[9], sim_scales, sim_sigma, sim_spec, sim_dc,
      sim_rows, sim_out, sim_raw, sim_scl, sim_offs;
  // PCA model building (pp_pca_moments, pp_pca_project, pp_lowpass_rows)
  DBuf pca_x, pca_w, pca_mu, pca_rw, pca_wsum, pca_vecs, pca_out, lp_in, lp_out, lp_kc;
  // timing
  bool timing = false;
  std::vector<cudaEvent_t> ev_chunk;   // "chunk finished" events for the overlapped result copies
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  struct Span { int kind; cudaEvent_t a, b; };
  std::vector<Span> spans;
  pp_stats_t stats;
  // the DBuf members free themselves after this; `stream` may be the caller's (pp_plan_set_stream)
  ~pp_plan() {
    for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : ev_chunk) cudaEventDestroy(e);
    for (cudaEvent_t e : {ev_copy[0], ev_copy[1], ev_free[0], ev_free[1], pin_ev[0], pin_ev[1], pin_ev[2], pin_ev[3]})
      if (e) cudaEventDestroy(e);
    for (void* h : pin_ring) if (h) cudaFreeHost(h);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
  }
};

enum { SP_SPECTRA = 0, SP_GUESS = 1, SP_PASS = 2, SP_UPDATE = 3, SP_TOTAL = 4, SP_COARSE = 5 };

static cudaEvent_t get_event(pp_plan* pl) {
  if (pl->ev_used == pl->ev_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    pl->ev_pool.push_back(e);
  }
  return pl->ev_pool[pl->ev_used++];
}

struct SpanGuard {
  pp_plan* pl; int kind; cudaEvent_t a = nullptr;
  SpanGuard(pp_plan* p, int k) : pl(p), kind(k) {
    if (pl->timing) { a = get_event(pl); cudaEventRecord(a, pl->stream); }
  }
  ~SpanGuard() {
    if (pl->timing) {
      cudaEvent_t b = get_event(pl);
      cudaEventRecord(b, pl->stream);
      pl->spans.push_back({kind, a, b});
    }
  }
};

static void stats_begin(pp_plan* pl) {
  memset(&pl->stats, 0, sizeof pl->stats);
  pl->stats.timing_enabled = pl->timing ? 1 : 0;
  pl->ev_used = 0;
  pl->spans.clear();
}

static void stats_end(pp_plan* pl) {
  if (!pl->timing) return;
  for (auto& sp : pl->spans) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, sp.a, sp.b);
    switch (sp.kind) {
      case SP_SPECTRA: pl->stats.ms_spectra += ms; break;
      case SP_GUESS: pl->stats.ms_guess += ms; break;
      case SP_PASS: pl->stats.ms_pass += ms; break;
      case SP_UPDATE: pl->stats.ms_update += ms; break;
      case SP_COARSE: pl->stats.ms_coarse += ms; break;
      case SP_TOTAL: pl->stats.ms_total += ms; break;
    }
  }
}

// ----------------------------------------------------------------------------
// pointer staging: returns a device pointer for host-or-device input
// ----------------------------------------------------------------------------
enum MemKind { kMemPageable, kMemPinned, kMemDevice };
static MemKind mem_kind(const void* p) {
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) { cudaGetLastError(); return kMemPageable; }
  if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) return kMemDevice;
  return at.type == cudaMemoryTypeHost ? kMemPinned : kMemPageable;
}
static bool is_device_ptr(const void* p) { return mem_kind(p) == kMemDevice; }

static cudaError_t h2d_any(pp_plan* pl, void* dst, const void* src, size_t bytes, bool src_pinned, cudaStream_t st, bool narrow);

template <typename T>
static int stage_in(pp_plan* pl, DBuf& buf, const T* src, size_t n, const T** out) {
  if (!src) { *out = nullptr; return 0; }
  const MemKind kind = mem_kind(src);
  if (kind == kMemDevice) { *out = src; return 0; }
  CK(buf.need(n * sizeof(T)));
  const size_t bytes = n * sizeof(T);
  CK(h2d_any(pl, buf.p, src, bytes, bytes < (8u << 20) || kind == kMemPinned, pl->stream, false));
  *out = buf.as<T>();
  return 0;
}

template <typename T>
static int copy_out_at(cudaStream_t st, T* dst, const T* dev, size_t off, size_t n) {
  if (!dst || n == 0) return 0;
  CK(cudaMemcpyAsync(dst + off, dev + off, n * sizeof(T),
                     is_device_ptr(dst) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  return 0;
}

// ----------------------------------------------------------------------------
// dispatch on N = nbin/2
// ----------------------------------------------------------------------------
template <int N, typename T> static size_t fft_smem_bytes() {
  return (size_t)(N + N / 2 + 2 + RowGeom<N>::kRows * 2 * N) * sizeof(cx<T>);
}
// CTAs of a row kernel (RowGeom<N>::kRows rows each) for nrows rows
template <int N> static unsigned row_ctas(long nrows) { return (unsigned)((nrows + RowGeom<N>::kRows - 1) / RowGeom<N>::kRows); }

#define DISPATCH_N(Nval, ...)                                   \
  switch (Nval) {                                               \
    case 32: { constexpr int NN = 32; __VA_ARGS__; } break;     \
    case 64: { constexpr int NN = 64; __VA_ARGS__; } break;     \
    case 128: { constexpr int NN = 128; __VA_ARGS__; } break;   \
    case 256: { constexpr int NN = 256; __VA_ARGS__; } break;   \
    case 512: { constexpr int NN = 512; __VA_ARGS__; } break;   \
    case 1024: { constexpr int NN = 1024; __VA_ARGS__; } break; \
    case 2048: { constexpr int NN = 2048; __VA_ARGS__; } break; \
    default: return fail(-1, "unsupported nbin %d", 2 * (Nval)); \
  }

template <int N> static size_t spectra_smem_bytes() { return spectra_smem_bytes_of<N>(); }
// row slots per k_spectra CTA for this nbin
static int spectra_slots(int N) {
  DISPATCH_N(N, return SpecPlan<NN>::kSlots);
  return 0;
}

template <int N> static void build_tw8(std::vector<double2>& out) { TwBuilder<SpecPlan<N>>::build(out); }

// k_spectra16 (nbin = 2048): one instantiation per (16-bit samples, FFTFIT guess, kept data spectra)
static void (*const kSpectra16[8])(SpectraArgs) = {
    k_spectra16<false, false, false>, k_spectra16<false, false, true>, k_spectra16<false, true, false>, k_spectra16<false, true, true>,
    k_spectra16<true, false, false>, k_spectra16<true, false, true>, k_spectra16<true, true, false>, k_spectra16<true, true, true>};
static cudaError_t spectra16_attrs() {
  for (auto k : kSpectra16) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)spectra_smem_bytes_of<1024, SpecPlan16>());
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
static void launch_spectra16(bool i16, bool guess, bool keepd, dim3 grid, cudaStream_t st, const SpectraArgs& a) {
  kSpectra16[4 * i16 + 2 * guess + keepd]<<<grid, 64, spectra_smem_bytes_of<1024, SpecPlan16>(), st>>>(a);
}
// the generic kernel on the other power-of-two nbin (N = 1024 is launch_spectra16's)
template <int N> static void launch_spectra(bool i16, dim3 grid, cudaStream_t st, const SpectraArgs& a) {
  if constexpr (N != 1024) {
    if (i16) k_spectra<N, SpecPlan<N>, true><<<grid, SpecPlan<N>::kThreads, spectra_smem_bytes<N>(), st>>>(a);
    else k_spectra<N><<<grid, SpecPlan<N>::kThreads, spectra_smem_bytes<N>(), st>>>(a);
  }
}

// ---- arbitrary nbin: Bluestein row transforms (bluestein.cuh) ----------------------------------------------
#define DISPATCH_M(Mval, ...)                                   \
  switch (Mval) {                                               \
    case 64: { constexpr int MM = 64; __VA_ARGS__; } break;     \
    case 128: { constexpr int MM = 128; __VA_ARGS__; } break;   \
    case 256: { constexpr int MM = 256; __VA_ARGS__; } break;   \
    case 512: { constexpr int MM = 512; __VA_ARGS__; } break;   \
    case 1024: { constexpr int MM = 1024; __VA_ARGS__; } break; \
    case 2048: { constexpr int MM = 2048; __VA_ARGS__; } break; \
    case 4096: { constexpr int MM = 4096; __VA_ARGS__; } break; \
    default: return fail(-1, "unsupported Bluestein length %d", (Mval)); \
  }
static int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }
template <int M> static cudaError_t any_attrs() {
  const int bytes = 2 * M * (int)sizeof(cx<double>);
  cudaError_t e;
#define A_(fn) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); if (e != cudaSuccess) return e;
  A_((k_fwd_any<M, false>)) A_((k_fwd_any<M, true>)) A_((k_inv_any<M, float>)) A_((k_inv_any<M, double>)) A_((k_cfft_row<M>))
#undef A_
  return cudaSuccess;
}
template <int N> static cudaError_t setup_attrs() {
  const int b32 = (int)fft_smem_bytes<N, float>(), b64 = (int)fft_smem_bytes<N, double>();
  cudaError_t e;
#define SET_(fn, bytes) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); if (e != cudaSuccess) return e;
  if constexpr (N != 1024) {   // nbin 2048 rows go to k_spectra16 (spectra16_attrs)
    SET_((k_spectra<N>), (int)spectra_smem_bytes<N>())
    SET_((k_spectra<N, SpecPlan<N>, true>), (int)spectra_smem_bytes<N>())
  }
  SET_((k_model<N>), b64)
  SET_((k_pass5<N>), (int)Pass5Ring<N>::kBytes)
  SET_((k_pass2<N>), (int)Pass2Ring<N>::kBytes)
  SET_((k_rfft_rows<N, float>), b32)
  SET_((k_rfft_rows<N, double>), b64)
  SET_((k_align_accum<N>), b64)
  SET_((k_align_finish<N>), b64)
  SET_((k_rotate<N, float>), b32)
  SET_((k_rotate<N, double>), b64)
  SET_((k_simulate<N>), b64)
#undef SET_
  return cudaFuncSetAttribute(k_guess, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double2) * 2048));
}

// ----------------------------------------------------------------------------
// plan
// ----------------------------------------------------------------------------
extern "C" int pp_plan_create(int32_t nchan, int32_t nbin, int32_t device, pp_plan_t** out) {
  if (!out) return fail(-1, "plan_out is NULL");
  *out = nullptr;
  if (nchan < 1) return fail(-1, "nchan must be >= 1 (got %d)", nchan);
  if (nbin < 64 || nbin > 4096 || (nbin & 1)) return fail(-1, "nbin must be even and in [64,4096] (got %d)", nbin);
  const bool pow2 = (nbin & (nbin - 1)) == 0;
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(-1, "device %d not available (%d devices)", device, ndev);
  CK(cudaSetDevice(device));
  std::unique_ptr<pp_plan> pl(new pp_plan());   // freed with all it holds when a step below fails
  pl->nchan = nchan; pl->nbin = nbin; pl->N = nbin / 2; pl->device = device;
  if (!pow2) {   // any other even nbin: Npad slots per spectrum row, Bluestein transforms of length M (bluestein.cuh)
    pl->anyn = true;
    pl->L = nbin / 2;
    pl->N = next_pow2(pl->L + 1);
    pl->M = next_pow2(2 * pl->L - 1);
  }
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  pl->l2_bytes = prop.l2CacheSize;
  pl->sm_count = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&pl->own_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&pl->copy_stream, cudaStreamNonBlocking));
  pl->stream = pl->own_stream;
  for (int i = 0; i < 2; ++i) {
    CK(cudaEventCreateWithFlags(&pl->ev_copy[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&pl->ev_free[i], cudaEventDisableTiming));
  }
  // twiddle tables in double, rounded once
  const int N = pl->N;
  std::vector<float2> t1(N), t2(N / 2 + 1);
  std::vector<double2> u1(N), u2(N / 2 + 1);
  for (int j = 0; j < N; ++j) {
    // octant-reduced so that the table has the exact symmetries of the roots of unity
    const double a = -2.0 * M_PI * (double)j / (double)N;
    u1[j] = make_double2(cos(a), sin(a));
    if (4 * j == N) u1[j] = make_double2(0.0, -1.0);
    if (2 * j == N) u1[j] = make_double2(-1.0, 0.0);
    if (4 * j == 3 * N) u1[j] = make_double2(0.0, 1.0);
    t1[j] = make_float2((float)u1[j].x, (float)u1[j].y);
  }
  for (int k = 0; k <= N / 2; ++k) {
    const double a = -2.0 * M_PI * (double)k / (double)(2 * N);
    u2[k] = make_double2(cos(a), sin(a));
    if (2 * k == N) u2[k] = make_double2(0.0, -1.0);
    t2[k] = make_float2((float)u2[k].x, (float)u2[k].y);
  }
  CK(pl->twN32.need(t1.size() * sizeof(float2)));
  CK(pl->tw2N32.need(t2.size() * sizeof(float2)));
  CK(pl->twN64.need(u1.size() * sizeof(double2)));
  CK(pl->tw2N64.need(u2.size() * sizeof(double2)));
  CK(cudaMemcpy(pl->twN32.p, t1.data(), t1.size() * sizeof(float2), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->tw2N32.p, t2.data(), t2.size() * sizeof(float2), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->twN64.p, u1.data(), u1.size() * sizeof(double2), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->tw2N64.p, u2.data(), u2.size() * sizeof(double2), cudaMemcpyHostToDevice));
  {
    cudaError_t e = cudaSuccess;
    DISPATCH_N(N, e = setup_attrs<NN>());
    CK(e);
    if (N == 1024) CK(spectra16_attrs());
    if (pl->anyn) {
      const int L = pl->L, M = pl->M;
      DISPATCH_M(M, e = any_attrs<MM>());
      CK(e);
      std::vector<double2> chirp(L), b(M, make_double2(0.0, 0.0)), twM(M), tw2n(L / 2 + 1);
      for (int j = 0; j < L; ++j) {                      // c_j = e^{-pi i j^2 / L}, the angle reduced in integers
        const long r = ((long)j * j) % (2L * L);
        const double ang = -M_PI * (double)r / (double)L;
        chirp[j] = make_double2(cos(ang), sin(ang));
      }
      b[0] = make_double2(1.0, 0.0);
      for (int m = 1; m < L; ++m) b[m] = b[M - m] = make_double2(chirp[m].x, -chirp[m].y);
      for (int j = 0; j < M; ++j) twM[j] = unit_root(j, M);
      for (int k = 0; k <= L / 2; ++k) tw2n[k] = unit_root(k, 2L * L);
      CK(pl->any_chirp.need(sizeof(double2) * L));
      CK(pl->any_B.need(sizeof(double2) * M));
      CK(pl->any_twM.need(sizeof(double2) * M));
      CK(pl->any_tw2n.need(sizeof(double2) * (L / 2 + 1)));
      {   // L = 2^a 3^b 5^c: radices of the direct transform (no radices: Bluestein)
        int rest = L;
        std::vector<int> rad;
        while (rest % 5 == 0) { rad.push_back(5); rest /= 5; }
        while (rest % 3 == 0) { rad.push_back(3); rest /= 3; }
        while (rest % 4 == 0) { rad.push_back(4); rest /= 4; }
        if (rest % 2 == 0) { rad.push_back(2); rest /= 2; }
        if (rest == 1 && rad.size() <= 12 && !getenv("PP_FORCE_BLUESTEIN")) pl->any_rad = rad;
        std::vector<double2> twL(L);
        for (int j = 0; j < L; ++j) twL[j] = unit_root(j, L);
        CK(pl->any_twL.need(sizeof(double2) * L));
        CK(cudaMemcpy(pl->any_twL.p, twL.data(), sizeof(double2) * L, cudaMemcpyHostToDevice));
      }
      CK(cudaMemcpy(pl->any_chirp.p, chirp.data(), sizeof(double2) * L, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(pl->any_B.p, b.data(), sizeof(double2) * M, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(pl->any_twM.p, twM.data(), sizeof(double2) * M, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(pl->any_tw2n.p, tw2n.data(), sizeof(double2) * (L / 2 + 1), cudaMemcpyHostToDevice));
      // the chirp filter's transform, divided by M (the inverse transform of the convolution)
      DISPATCH_M(M, (k_cfft_row<MM><<<1, 256, 2 * MM * sizeof(cx<double>), pl->stream>>>(
                        pl->any_B.as<cx<double>>(), pl->any_twM.as<cx<double>>(), 1.0 / (double)MM)));
      CK(cudaGetLastError());
      CK(cudaStreamSynchronize(pl->stream));
    }
    std::vector<double2> t8;
    DISPATCH_N(N, build_tw8<NN>(t8));
    CK(pl->tw8.need(t8.size() * sizeof(double2)));
    CK(cudaMemcpy(pl->tw8.p, t8.data(), t8.size() * sizeof(double2), cudaMemcpyHostToDevice));
  }
  *out = pl.release();
  return 0;
}

extern "C" void pp_plan_destroy(pp_plan_t* pl) {
  if (!pl) return;
  cudaSetDevice(pl->device);
  cudaStreamSynchronize(pl->stream);   // nothing is freed under the plan's queued work
  delete pl;
}

extern "C" int pp_plan_set_stream(pp_plan_t* pl, void* s) {
  if (!pl) return fail(-1, "plan is NULL");
  pl->stream = s ? reinterpret_cast<cudaStream_t>(s) : pl->own_stream;
  return 0;
}

extern "C" int pp_plan_set_chunk(pp_plan_t* pl, int32_t n) {
  if (!pl) return fail(-1, "plan is NULL");
  if (n < 0) return fail(-1, "chunk must be >= 0");
  pl->chunk_req = n;
  return 0;
}

extern "C" int pp_plan_enable_timing(pp_plan_t* pl, int32_t on) {
  if (!pl) return fail(-1, "plan is NULL");
  pl->timing = on != 0;
  return 0;
}

extern "C" int pp_get_stats(pp_plan_t* pl, pp_stats_t* st) {
  if (!pl || !st) return fail(-1, "NULL argument");
  *st = pl->stats;
  st->x_keep_frac = pl->x_keep;
  return 0;
}

static int grid_table(pp_plan* pl, int Ns, const double2** out) {
  for (auto& gt : pl->grid_tables)
    if (gt.first == Ns) { *out = gt.second.as<double2>(); return 0; }
  const int M = Ns - 1;
  std::vector<double2> t(M);
  for (int m = 0; m < M; ++m) {
    // e^{2 pi i m/M} with exact quadrant symmetry handled by cos/sin of a reduced angle
    const double a = 2.0 * M_PI * (double)m / (double)M;
    t[m] = make_double2(cos(a), sin(a));
  }
  pl->grid_tables.emplace_back(Ns, DBuf());
  DBuf& b = pl->grid_tables.back().second;
  CK(b.need(sizeof(double2) * M));
  CK(cudaMemcpyAsync(b.p, t.data(), sizeof(double2) * M, cudaMemcpyHostToDevice, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));  // t goes out of scope
  *out = b.as<double2>();
  return 0;
}

// general grid np.mgrid[lo:hi:Ns j] = lo + arange(Ns) * (hi - lo)/(Ns - 1): e^{2 pi i phi_j}, j < Ns
static int grid_table_general(pp_plan* pl, int Ns, double lo, double hi, const double2** out) {
  const double step = (hi - lo) / (double)(Ns - 1);
  std::vector<double2> t(Ns);
  for (int j = 0; j < Ns; ++j) {
    double phi = lo + (double)j * step;
    phi -= nearbyint(phi);
    t[j] = make_double2(cos(2.0 * M_PI * phi), sin(2.0 * M_PI * phi));
  }
  CK(pl->grid_general.need(sizeof(double2) * Ns));
  CK(cudaMemcpyAsync(pl->grid_general.p, t.data(), sizeof(double2) * Ns, cudaMemcpyHostToDevice, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));  // t goes out of scope
  *out = pl->grid_general.as<double2>();
  return 0;
}

// ----------------------------------------------------------------------------
// model
// ----------------------------------------------------------------------------
static AnyPlan any_dev(pp_plan* pl) {
  AnyPlan p;
  p.chirp = pl->any_chirp.as<cx<double>>(); p.Bspec = pl->any_B.as<cx<double>>(); p.twM = pl->any_twM.as<cx<double>>();
  p.tw2n = pl->any_tw2n.as<cx<double>>(); p.L = pl->L; p.Npad = pl->N;
  p.twL = pl->any_twL.as<cx<double>>();
  p.nrad = (int)pl->any_rad.size();
  for (int i = 0; i < 12; ++i) p.rad[i] = i < p.nrad ? pl->any_rad[i] : 1;
  return p;
}
static int launch_fwd_any(pp_plan* pl, const void* in, bool i16, const float* scl, const float* offs, long nrows,
                          cx<double>* spec, double* dc, const double* in64 = nullptr) {
  FwdAnyArgs a;
  a.in = in; a.in64 = in64; a.dat_scl = scl; a.dat_offs = offs; a.spec = spec; a.dc = dc; a.p = any_dev(pl); a.nrows = nrows;
  const unsigned grid = (unsigned)std::min<long>(nrows, 148L * 64);
  // (the direct mixed-radix transform works on 2 L points, the Bluestein convolution on 2 M)
  const size_t sm = 2 * sizeof(cx<double>) * (pl->any_rad.empty() ? (size_t)pl->M : (size_t)pl->L);
  if (i16) { DISPATCH_M(pl->M, (k_fwd_any<MM, true><<<grid, 256, sm, pl->stream>>>(a))); }
  else { DISPATCH_M(pl->M, (k_fwd_any<MM, false><<<grid, 256, sm, pl->stream>>>(a))); }
  pl->stats.launches++;
  return 0;
}
static int launch_inv_any(pp_plan* pl, const cx<double>* spec, const double* dc, void* out, long nrows, bool out_double) {
  InvAnyArgs a;
  a.spec = spec; a.dc = dc; a.out = out; a.p = any_dev(pl); a.nrows = nrows;
  const unsigned grid = (unsigned)std::min<long>(nrows, 148L * 64);
  const size_t sm = 2 * sizeof(cx<double>) * (pl->any_rad.empty() ? (size_t)pl->M : (size_t)pl->L);
  if (out_double) { DISPATCH_M(pl->M, (k_inv_any<MM, double><<<grid, 256, sm, pl->stream>>>(a))); }
  else { DISPATCH_M(pl->M, (k_inv_any<MM, float><<<grid, 256, sm, pl->stream>>>(a))); }
  pl->stats.launches++;
  return 0;
}
// (nbin not a power of two) the rotated / multiplied spectra of the a.nsub * a.nchan rows into any_spec2 / any_dc2
static int rotate_spectra_any(pp_plan* pl, const RotateArgs& a) {
  const int N = pl->N;
  const long nrows = (long)a.nsub * a.nchan;
  CK(pl->any_spec2.need(sizeof(double2) * (size_t)nrows * N));
  CK(pl->any_dc2.need(sizeof(double) * (size_t)nrows));
  if (launch_fwd_any(pl, a.in, false, nullptr, nullptr, nrows, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>())) return -2;
  k_rot_mul<<<(unsigned)nrows, 256, 0, pl->stream>>>(a, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>(), N, pl->L);
  pl->stats.launches++;
  return 0;
}

// rfft -> multiply (rotation / scattering kernel / response) -> irfft of nrows = a.nsub * a.nchan rows: one
// fused kernel for nbin = 2^m, transform / multiply / transform through the spectrum scratch otherwise
static int rotate_rows(pp_plan* pl, RotateArgs a, bool fp64) {
  const int N = pl->N;
  const long nrows = (long)a.nsub * a.nchan;
  if (pl->anyn) {
    if (rotate_spectra_any(pl, a)) return -2;
    return launch_inv_any(pl, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>(), a.out, nrows, false);
  }
  if (fp64) {
    a.twN = pl->twN64.p; a.tw2N = pl->tw2N64.p;
    DISPATCH_N(N, (k_rotate<NN, double><<<row_ctas<NN>(nrows), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(a)));
  } else {
    a.twN = pl->twN32.p; a.tw2N = pl->tw2N32.p;
    DISPATCH_N(N, (k_rotate<NN, float><<<row_ctas<NN>(nrows), 256, fft_smem_bytes<NN, float>(), pl->stream>>>(a)));
  }
  pl->stats.launches++;
  return 0;
}

// the frequency tables of models 0 .. ntab - 1 ([ntab, nchan]; pp_set_freqs: model 0's)
static int set_freqs_impl(pp_plan* pl, const double* freqs, int ntab = 1) {
  const int nchan = pl->nchan * ntab;   // rows
  std::vector<double> hf(nchan), hn2(nchan), hlg(nchan);
  if (is_device_ptr(freqs)) CK(cudaMemcpy(hf.data(), freqs, sizeof(double) * nchan, cudaMemcpyDeviceToHost));
  else memcpy(hf.data(), freqs, sizeof(double) * nchan);
  for (int n = 0; n < nchan; ++n) {
    if (!(hf[n] > 0.0)) {
      if (ntab == 1) return fail(-1, "freqs[%d] = %g is not positive", n, hf[n]);
      return fail(-1, "freqs[%d, %d] = %g is not positive", n / pl->nchan, n % pl->nchan, hf[n]);
    }
    hn2[n] = 1.0 / (hf[n] * hf[n]);
    hlg[n] = log2(hf[n]);
  }
  CK(pl->freqs.need(sizeof(double) * nchan));
  CK(pl->nu2.need(sizeof(double) * nchan));
  CK(cudaMemcpyAsync(pl->freqs.p, hf.data(), sizeof(double) * nchan, cudaMemcpyHostToDevice, pl->stream));
  CK(cudaMemcpyAsync(pl->nu2.p, hn2.data(), sizeof(double) * nchan, cudaMemcpyHostToDevice, pl->stream));
  CK(pl->lgf.need(sizeof(double) * nchan));
  CK(cudaMemcpyAsync(pl->lgf.p, hlg.data(), sizeof(double) * nchan, cudaMemcpyHostToDevice, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));  // hf/hn2 are stack-owned
  pl->freqs_set = true;
  return 0;
}

extern "C" int pp_set_freqs(pp_plan_t* pl, const double* freqs) {
  if (!pl || !freqs) return fail(-1, "NULL argument");
  CK(cudaSetDevice(pl->device));
  return set_freqs_impl(pl, freqs);
}

extern "C" int pp_plan_set_model_steps(pp_plan_t* pl, int32_t steps) {
  if (!pl) return fail(-1, "NULL plan");
  if (steps < 0 || steps > 64) return fail(-1, "model steps must be 0 (default) .. 64");
  pl->model_steps = steps == 0 ? 8 : steps;
  return 0;
}

// The coarse objective of the general solver: the leading groups of 16 harmonics that hold `frac` of the
// (scattered) model's phase information; 0 = no coarse stage (it would not be at most half of the harmonics).
static int choose_coarse(const double* info, double frac, int N) {
  const int NJ = N / 16;
  if (!(frac > 0.0) || NJ < 8) return 0;
  double tot = 0.0;
  for (int j = 0; j < NJ; ++j) tot += info[j];
  if (!(tot > 0.0) || !(tot < INFINITY)) return 0;
  double cum = 0.0;
  int nj = NJ;
  for (int j = 0; j < NJ; ++j) { cum += info[j]; if (cum >= frac * tot) { nj = j + 1; break; } }
  nj = std::max(nj, 4);   // the groups that carry float32 residuals (LoK = 64 harmonics) are always summed
  return 2 * nj <= NJ ? nj : 0;
}

// the cut-offs of every channel of every model; x_keep over all of them, kmax_used per model
static int model_cutoffs(pp_plan* pl) {
  const int N = pl->N, nchan = pl->nchan, NJ = N / 16, KJ = (N < 64 ? N : 64) / 16;
  const int nrows = pl->nmodel * nchan;
  CK(pl->njn.need(sizeof(int) * nrows));
  k_model_cutoff<<<nrows, 256, 0, pl->stream>>>(pl->mpow.as<double>(), pl->njn.as<int>(), N, KJ, pl->cutoff_eps2);
  pl->stats.launches++;
  std::vector<int> h(nrows);
  CK(cudaMemcpyAsync(h.data(), pl->njn.p, sizeof(int) * nrows, cudaMemcpyDeviceToHost, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));
  double keep = 0.0;
  pl->kmax_used.assign(pl->nmodel, 0);
  for (int r = 0; r < nrows; ++r) {
    keep += h[r];
    int& vmax = pl->kmax_used[r / nchan];
    vmax = std::max(vmax, 16 * h[r]);
  }
  pl->x_keep = keep / ((double)nrows * NJ);
  // (a pageable source: the copy has read it when the call returns)
  CK(pl->kmax_dev.need(sizeof(int) * pl->nmodel));
  CK(cudaMemcpyAsync(pl->kmax_dev.p, pl->kmax_used.data(), sizeof(int) * pl->nmodel, cudaMemcpyHostToDevice, pl->stream));
  return 0;
}

extern "C" int pp_plan_set_model_cutoff(pp_plan_t* pl, double eps) {
  if (!pl) return fail(-1, "NULL plan");
  if (!(eps >= 0.0 && eps < 1e-3)) return fail(-1, "model cut-off must be in [0, 1e-3): 0 keeps every harmonic");
  CK(cudaSetDevice(pl->device));
  pl->cutoff_eps2 = eps * eps;
  if (pl->model_set && model_cutoffs(pl)) return -2;
  return 0;
}

extern "C" int pp_plan_set_coarse(pp_plan_t* pl, double frac) {
  if (!pl) return fail(-1, "NULL plan");
  if (!(frac >= 0.0 && frac < 1.0)) return fail(-1, "coarse fraction must be in [0, 1): 0 disables the coarse stage");
  pl->coarse_frac = frac;
  return 0;
}

extern "C" int pp_plan_set_fft_precision(pp_plan_t* pl, int32_t bits) {
  if (!pl) return fail(-1, "plan is NULL");
  if (bits != 0 && bits != 32 && bits != 64) return fail(-1, "fft precision must be 0 (auto), 32 or 64");
  pl->fft_precision = bits;
  return 0;
}

// float64 -> float32 (cvt.rn) of n2 pairs of samples on st
static void cvt_f64_f32(const void* src, void* dst, size_t n2, cudaStream_t st) {
  k_cvt_f64_f32<<<(unsigned)std::min<size_t>((n2 + 255) / 256, 148 * 32), 256, 0, st>>>(
      static_cast<const double2*>(src), static_cast<float2*>(dst), n2);
}

static int set_model_impl(pp_plan* pl, int nmodel, const float* model, const double* model64, const double* freqs) {
  if (nmodel < 1) return fail(-1, "nmodel must be >= 1 (got %d)", nmodel);
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int N = pl->N, nchan = nmodel * pl->nchan;   // the model rows of all models: one transform
  const float* dmodel = nullptr;
  const double* dmodel64 = nullptr;
  const size_t nsamp = (size_t)nchan * pl->nbin;
  if (model64) {
    if (stage_in(pl, pl->model_stage64, model64, nsamp, &dmodel64)) return -2;
    if (pl->anyn) {   // the arbitrary-nbin rows take float32 input: round on the device
      CK(pl->model_stage.need(sizeof(float) * nsamp));
      cvt_f64_f32(dmodel64, pl->model_stage.p, nsamp / 2, pl->stream);
      dmodel = pl->model_stage.as<float>();
      dmodel64 = nullptr;
    }
  } else if (stage_in(pl, pl->model_stage, model, nsamp, &dmodel)) return -2;
  if (set_freqs_impl(pl, freqs, nmodel)) return -2;
  pl->model_set = false;
  pl->nmodel = nmodel;
  CK(pl->mconj32.need(sizeof(float2) * (size_t)nchan * N));
  CK(pl->mconj64.need(sizeof(double2) * (size_t)nchan * N));
  CK(pl->mpow.need(sizeof(double) * (size_t)nchan * N));
  CK(pl->pn.need(sizeof(double) * nchan));
  CK(pl->mmean.need(sizeof(float2) * (size_t)nmodel * N));
  ModelArgs a;
  a.model = dmodel; a.model64 = dmodel64; a.mconj32 = pl->mconj32.as<cx<float>>(); a.mconj64 = pl->mconj64.as<cx<double>>();
  a.mpow = pl->mpow.as<double>(); a.pn = pl->pn.as<double>();
  a.twN = pl->twN64.as<cx<double>>(); a.tw2N = pl->tw2N64.as<cx<double>>(); a.spec = nullptr; a.nchan = nchan;
  if (pl->anyn) {
    CK(pl->any_spec2.need(sizeof(double2) * (size_t)nchan * N));
    if (launch_fwd_any(pl, dmodel, false, nullptr, nullptr, nchan, pl->any_spec2.as<cx<double>>(), nullptr)) return -2;
    k_model_from_spec<<<nchan, 256, 0, pl->stream>>>(pl->any_spec2.as<cx<double>>(), a.mconj32, a.mconj64, a.mpow, a.pn, N);
  } else {
    DISPATCH_N(N, (k_model<NN><<<row_ctas<NN>(nchan), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(a)));
  }
  k_model_mean<<<dim3((N + 127) / 128, nmodel), 128, 0, pl->stream>>>(pl->mconj64.as<cx<double>>(), pl->mmean.as<float2>(),
                                                                      pl->nchan, N);
  pl->stats.launches += 2;
  CK(cudaGetLastError());
  if (model_cutoffs(pl)) return -2;
  pl->model_set = true;
  return 0;
}

extern "C" int pp_set_models(pp_plan_t* pl, int32_t nmodel, const float* models, const double* freqs) {
  if (!pl || !models || !freqs) return fail(-1, "NULL argument");
  return set_model_impl(pl, nmodel, models, nullptr, freqs);
}

extern "C" int pp_set_models_f64(pp_plan_t* pl, int32_t nmodel, const double* models, const double* freqs) {
  if (!pl || !models || !freqs) return fail(-1, "NULL argument");
  return set_model_impl(pl, nmodel, nullptr, models, freqs);
}

extern "C" int pp_set_model(pp_plan_t* pl, const float* model, const double* freqs) {
  return pp_set_models(pl, 1, model, freqs);
}

extern "C" int pp_set_model_f64(pp_plan_t* pl, const double* model, const double* freqs) {
  return pp_set_models_f64(pl, 1, model, freqs);
}

// ----------------------------------------------------------------------------
// fit
// ----------------------------------------------------------------------------
// run(o, m) on elements [o, o + m) of [0, n) from nthreads host threads, in pieces of a multiple of `align` (a power of two)
template <typename F> static void parallel_pieces(size_t n, size_t align, int nthreads, F run) {
  std::vector<std::thread> th;
  const size_t per = ((n / nthreads) + align - 1) & ~(align - 1);
  for (int i = 1; i < nthreads; ++i) {
    const size_t o = (size_t)i * per;
    if (o >= n) break;
    th.emplace_back([=]() { run(o, std::min(per, n - o)); });
  }
  run(0, std::min(per, n));
  for (auto& t : th) t.join();
}

static void parallel_memcpy(void* dst, const void* src, size_t n, int nthreads) {
  if (nthreads <= 1 || n < (4u << 20)) { memcpy(dst, src, n); return; }
  parallel_pieces(n, 4096, nthreads, [=](size_t o, size_t m) { memcpy((char*)dst + o, (const char*)src + o, m); });
}

// float64 -> float32 (round to nearest even, as the device's cvt.rn.f32.f64) while staging pageable rows
static void parallel_narrow(float* dst, const double* src, size_t n, int nthreads) {
  auto run = [=](size_t o, size_t m) { for (size_t i = o; i < o + m; ++i) dst[i] = (float)src[i]; };
  if (nthreads <= 1 || n < (1u << 20)) { run(0, n); return; }
  parallel_pieces(n, 1024, nthreads, run);
}

static bool h2d_stages(size_t bytes, bool src_pinned) { return !src_pinned && bytes >= (8u << 20); }

// host -> device on `st`: straight from page-locked memory, through the plan's page-locked ring otherwise.
// narrow: src holds float64 samples and dst receives them as float32 (only when the copy is staged: h2d_stages());
// `bytes` counts source bytes.
static cudaError_t h2d_any(pp_plan* pl, void* dst, const void* src, size_t bytes, bool src_pinned, cudaStream_t st,
                           bool narrow) {
  if (!h2d_stages(bytes, src_pinned)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
  static const int nthreads = std::max(1, std::min(8, (int)std::thread::hardware_concurrency() / 2));
  // pieces of kPinPiece bytes as they are sent: counted in source elements (float64 when narrowing, else bytes)
  const size_t src_size = narrow ? sizeof(double) : 1, dst_size = narrow ? sizeof(float) : 1;
  const size_t n = bytes / src_size, per = pp_plan::kPinPiece / dst_size;
  for (size_t off = 0; off < n; off += per) {
    const size_t len = std::min(per, n - off);
    const int slot = (int)(pl->pin_count++ % pp_plan::kPinSlots);
    cudaError_t e;
    if (!pl->pin_ring[slot]) {
      e = cudaHostAlloc(&pl->pin_ring[slot], pp_plan::kPinPiece, cudaHostAllocDefault);
      if (e != cudaSuccess) return e;
      e = cudaEventCreateWithFlags(&pl->pin_ev[slot], cudaEventDisableTiming);
      if (e != cudaSuccess) return e;
    } else {
      e = cudaEventSynchronize(pl->pin_ev[slot]);      // the copy that last used this slot has left it
      if (e != cudaSuccess) return e;
    }
    if (narrow) parallel_narrow(static_cast<float*>(pl->pin_ring[slot]), static_cast<const double*>(src) + off, len, nthreads);
    else parallel_memcpy(pl->pin_ring[slot], (const char*)src + off, len, nthreads);
    e = cudaMemcpyAsync((char*)dst + off * dst_size, pl->pin_ring[slot], len * dst_size, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    e = cudaEventRecord(pl->pin_ev[slot], st);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

static const int kMaxChunk = 32768;   // the chunk index is gridDim.y of the row kernels (<= 65535)
static int pick_chunk(pp_plan* pl, int nsub, bool data_on_host, double bytes_per_sample = 4.0) {
  if (pl->chunk_req > 0) return std::min(std::min(pl->chunk_req, kMaxChunk), nsub);
  if (data_on_host) {
    // Host data arrive over PCIe (~50 GB/s), ten times slower than the kernels consume them: small
    // chunks so that the copy of chunk c+1 runs under the kernels of chunk c from early on (the
    // kernels' per-chunk overheads stay hidden behind the copies).  ~16 chunks, 64..512 subints.
    const double per_in = bytes_per_sample * pl->nbin * (double)pl->nchan;
    long c = std::max(64L, std::min(512L, (long)nsub / 16));
    c = std::min(c, std::max(1L, (long)floor(2.0 * 1073741824.0 / per_in)));   // staging <= 2 GiB each
    return (int)std::min<long>(c, nsub);
  }
  // Streaming mode: chunks large enough that every launch fills the GPU many
  // times over (launch latency and the serial FFTFIT-guess tail amortised);
  // the cross-spectrum scratch (8 N nchan bytes per subint) is capped at 8 GiB.
  const double per = 8.0 * pl->N * (double)pl->nchan;
  long c = (long)floor(8.0 * 1073741824.0 / per);
  c = std::min<long>(std::max(c, 64L), kMaxChunk);
  return (int)std::min<long>(c, nsub);
}

constexpr int kSpectraGMax = 32;   // most channel rows per spectra CTA
// nbin 2048 has one row slot per CTA, so its G never exceeds kSpectraGMax: k_spectra16 takes every such launch
static_assert(SpecPlan<1024>::kSlots == 1 && kSpectraGMax <= kSpec16MaxRows, "nbin 2048: G <= kSpec16MaxRows");

static int rows_per_cta(pp_plan* pl) {
  // Channel rows handled by one k_spectra CTA.  It fixes how the partial profile spectra of
  // the FFTFIT guess are grouped, so it must NOT depend on the batch or chunk size (results
  // are bit-identical for any chunking): a function of nchan only, ~16 CTAs per subint.
  const int rows_conc = spectra_slots(pl->N);
  int g = std::max(rows_conc, std::min(kSpectraGMax, pl->nchan / (512 / kSpectraGMax)));
  g = ((g + rows_conc - 1) / rows_conc) * rows_conc;
  // k_spectra finalises one row per thread of a row slot: rows per slot <= N/8 (32 <= 128 here)
  return g;
}

// One pp_fit_batch call: the validated flags, the staged inputs, the chunk geometry and the kernel arguments.  The
// pass and update arguments are built once per call: each chunk sets s0, the coarse stage its own fields.
struct FitCall {
  const pp_fit_args_t* args;
  const pp_fit_out_t* out;
  std::chrono::steady_clock::time_point tr0;
  bool general, want_guess, want_align, i16, f64, data_on_device, data_pinned;
  int nsub, Ns, max_iter, n_launch_iter;
  double tol;
  // device copies of the inputs (or the caller's device pointers)
  const double *dP, *derrs, *dw, *dinit, *ddmg, *dsnrs, *dnufits, *dnuouts, *dscat;
  const uint8_t* dmask;
  const float *dscl = nullptr, *doffs = nullptr;
  const double2* table = nullptr;   // FFTFIT grid
  const int* dmidx = nullptr;       // the model of each subint on the device (null: the plan's one model)
  std::vector<int> hmidx;           // ... and on the host
  std::vector<int> cfirst, cnjm;    // coarse stage with several models: the models' first subints, their levels' groups
  const char* data;                 // the caller's rows
  size_t sub_bytes, src_bytes;      // one subint as the kernels read it, and as the caller stores it
  int chunk, G, gx, nparts, align_nsplit = 1;
  std::vector<int> cstart;          // chunk c is subints cstart[c] .. cstart[c + 1] - 1
  SolverState st;
  Box box;
  PassArgs pa; UpdateArgs ua; Pass5Args p5; Update5Args u5;
  // chunk loop
  int coarse_nj = 0;                // harmonic groups of this chunk's coarse objective (0: no coarse stage)
  int pending_out = -1;             // chunk whose result copies still have to be queued
  bool expect_third = false;        // the previous chunk still had unfinished subints after two passes
};

// PP_TRACE=1: host-side wall-clock marks of the call on stderr (where a step's time goes outside the kernels)
static void mark(const FitCall& f, const char* fmt, ...) {
  static const bool trace = getenv("PP_TRACE") != nullptr;
  if (!trace) return;
  char what[128];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(what, sizeof what, fmt, ap);
  va_end(ap);
  fprintf(stderr, "[pp_fit_batch] %-22s %8.3f ms\n", what,
          std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - f.tr0).count());
}

static int fit_stage_inputs(pp_plan* pl, FitCall& f) {
  const pp_fit_args_t* args = f.args;
  const int nsub = f.nsub;
  const size_t nsc = (size_t)nsub * pl->nchan;
  if (stage_in(pl, pl->in_P, args->P, (size_t)nsub, &f.dP)) return -2;
  if (stage_in(pl, pl->in_errs, args->errs, nsc, &f.derrs)) return -2;
  if (stage_in(pl, pl->in_mask, args->chan_mask, nsc, &f.dmask)) return -2;
  if (stage_in(pl, pl->in_w, args->weights, nsc, &f.dw)) return -2;
  if (stage_in(pl, pl->in_init, args->init, (size_t)nsub * 5, &f.dinit)) return -2;
  if (stage_in(pl, pl->in_dmg, args->DM_guess, (size_t)nsub, &f.ddmg)) return -2;
  if (stage_in(pl, pl->in_snrs, args->snrs, nsc, &f.dsnrs)) return -2;
  if (stage_in(pl, pl->in_nufits, args->nu_fits, (size_t)nsub * 3, &f.dnufits)) return -2;
  if (stage_in(pl, pl->in_nuouts, args->nu_outs, (size_t)nsub * 3, &f.dnuouts)) return -2;
  if (stage_in(pl, pl->in_scat, args->scat_guess, (size_t)nsub * 2, &f.dscat)) return -2;
  f.want_guess = (args->init == nullptr);
  Box& box = f.box;
  box.on = 0;
  for (int i = 0; i < 5; ++i) { box.lo[i] = -INFINITY; box.hi[i] = INFINITY; }
  if (args->bounds) {
    if (is_device_ptr(args->bounds)) return fail(-1, "bounds must be a host pointer");
    for (int i = 0; i < 5; ++i) {
      const double lo = args->bounds[2 * i], hi = args->bounds[2 * i + 1];
      if (lo == lo && lo > -INFINITY) { box.lo[i] = lo; box.on = 1; }
      if (hi == hi && hi < INFINITY) { box.hi[i] = hi; box.on = 1; }
      if (box.lo[i] > box.hi[i]) return fail(-1, "bounds[%d]: lower %g > upper %g", i, lo, hi);
    }
  }
  return 0;
}

// per-subint and per-channel workspace; chunk size, spectra grid, the chunk-sized buffers and the chunk boundaries
static int fit_workspace(pp_plan* pl, FitCall& f) {
  const pp_fit_args_t* args = f.args;
  const int nsub = f.nsub, nchan = pl->nchan, N = pl->N;
  const size_t nsc = (size_t)nsub * nchan;
  CK(pl->nu_fit.need(sizeof(double) * nsub * 3));
  CK(pl->nu_mean.need(sizeof(double) * nsub));
  CK(pl->wsum.need(sizeof(double) * nsub));
  CK(pl->nok.need(sizeof(int) * nsub));
  CK(pl->sigma.need(sizeof(double) * nsc));
  CK(pl->Ssn.need(sizeof(double) * nsc));
  CK(pl->Sdn.need(sizeof(double) * nsc));
  CK(pl->csum.need(sizeof(double) * nsc * kNCsum));
  // k_pass2 writes slots 0-4 only: the (phi, DM) layout returns slots 5-8 as 0, not what an earlier call left there
  if (!f.general && f.out->chan_sums) CK(cudaMemsetAsync(pl->csum.p, 0, sizeof(double) * nsc * kNCsum, pl->stream));
  CK(pl->st_x.need(sizeof(double) * nsub * 5));
  CK(pl->st_xprev.need(sizeof(double) * nsub * 5));
  CK(pl->st_step.need(sizeof(double) * nsub * 5));
  CK(pl->st_fprev.need(sizeof(double) * nsub));
  CK(pl->st_lam.need(sizeof(double) * nsub));
  CK(pl->st_iter.need(sizeof(int) * nsub));
  CK(pl->st_iterc.need(sizeof(int) * nsub));
  CK(pl->st_done.need(sizeof(int) * nsub));
  CK(pl->o_params.need(sizeof(double) * nsub * 5));
  CK(pl->o_perrs.need(sizeof(double) * nsub * 5));
  CK(pl->o_nuout.need(sizeof(double) * nsub * 3));
  CK(pl->o_cov.need(sizeof(double) * nsub * 25));
  CK(pl->o_chi2.need(sizeof(double) * nsub));
  CK(pl->o_rchi2.need(sizeof(double) * nsub));
  CK(pl->o_snr.need(sizeof(double) * nsub));
  CK(pl->o_nfev.need(sizeof(int) * nsub));
  CK(pl->o_rc.need(sizeof(int) * nsub));
  CK(pl->o_scales.need(sizeof(double) * nsc));
  CK(pl->o_serrs.need(sizeof(double) * nsc));
  CK(pl->o_csnr.need(sizeof(double) * nsc));
  CK(pl->o_lag.need(sizeof(int) * nsub));
  CK(pl->o_phig.need(sizeof(double) * nsub));
  CK(pl->running.need(sizeof(int)));
  mark(f, "inputs staged");

  const MemKind data_kind = mem_kind(args->data);
  f.data_on_device = data_kind == kMemDevice;
  f.data_pinned = data_kind == kMemPinned;
  const int chunk = f.chunk = pick_chunk(pl, nsub, !f.data_on_device, f.f64 ? 8.0 : 4.0);
  f.G = rows_per_cta(pl);
  f.gx = (nchan + f.G - 1) / f.G;
  f.nparts = f.gx * spectra_slots(N);
  pl->stats.chunk = chunk;
  CK(pl->X.need(sizeof(float2) * (size_t)chunk * nchan * N));
  // fused ppalign accumulation (ppalign.py:197-213): keep the data spectra of the chunk
  f.want_align = f.out->align_sum != nullptr;
  if (f.want_align) {
    if (!f.out->align_wsum) return fail(-1, "align_sum needs align_wsum");
    CK(pl->Dspec.need(sizeof(float2) * (size_t)chunk * nchan * N));
    CK(pl->Ddc.need(sizeof(double) * (size_t)chunk * nchan));
    // partial sums per k_align_spec grid slice (each slice is owned by one CTA: no atomics, so the
    // result is reproducible); the slice count depends on nchan only
    const int nsplit = f.align_nsplit = std::max(1, (8 * 148 * 8) / std::max(1, nchan));   // ~8 CTAs per SM
    CK(pl->al_acc.need(sizeof(double2) * (size_t)nsplit * nchan * N));
    CK(pl->al_wparts.need(sizeof(double) * (size_t)nsplit * nchan));
    CK(pl->al_wsum.need(sizeof(double) * nchan));
    CK(pl->al_out.need(sizeof(double) * (size_t)nchan * pl->nbin));
    CK(cudaMemsetAsync(pl->al_acc.p, 0, sizeof(double2) * (size_t)nsplit * nchan * N, pl->stream));
    CK(cudaMemsetAsync(pl->al_wparts.p, 0, sizeof(double) * (size_t)nsplit * nchan, pl->stream));
  }
  CK(pl->Xlo.need(sizeof(float2) * (size_t)chunk * nchan * std::min(N, 64)));
  if (f.want_guess) CK(pl->partial.need(sizeof(float2) * (size_t)chunk * f.nparts * N));
  if (f.data_on_device && !pl->anyn && (reinterpret_cast<uintptr_t>(args->data) & 15))
    return fail(-1, "device data pointer must be 16-byte aligned");
  f.sub_bytes = (size_t)nchan * pl->nbin * (f.i16 ? sizeof(int16_t) : sizeof(float));
  f.src_bytes = f.f64 ? (size_t)nchan * pl->nbin * sizeof(double) : f.sub_bytes;
  f.data = reinterpret_cast<const char*>(args->data);
  if (!f.data_on_device || f.f64)
    for (int i = 0; i < 2; ++i) CK(pl->data_stage[i].need((size_t)chunk * f.sub_bytes));
  if (f.f64 && !f.data_on_device)
    for (int i = 0; i < 2; ++i) CK(pl->data_stage64[i].need((size_t)chunk * f.src_bytes));
  if (f.i16) {
    if (stage_in(pl, pl->in_scl, args->dat_scl, (size_t)nsub * nchan, &f.dscl)) return -2;
    if (stage_in(pl, pl->in_offs, args->dat_offs, (size_t)nsub * nchan, &f.doffs)) return -2;
  }
  // chunk boundaries; with several chunks the last one is kept short (<= 256 subints) because its
  // result copy is the only one that cannot hide under a following chunk's kernels
  for (int s0 = 0; s0 < nsub; s0 += chunk) f.cstart.push_back(s0);
  if (f.cstart.size() >= 2) {
    const int tail = 256, last0 = f.cstart.back();
    if (nsub - last0 > tail) f.cstart.push_back(nsub - tail);
  }
  f.cstart.push_back(nsub);
  return 0;
}

// the solver state and the pass / update kernel arguments of the call (s0 is set per chunk)
static void fit_kernel_args(pp_plan* pl, FitCall& f) {
  const pp_fit_args_t* args = f.args;
  const uint8_t* ff = args->fit_flags;
  const int nchan = pl->nchan, N = pl->N;
  SolverState& st = f.st;
  st.x = pl->st_x.as<double>(); st.xprev = pl->st_xprev.as<double>(); st.step = pl->st_step.as<double>();
  st.fprev = pl->st_fprev.as<double>(); st.lam = pl->st_lam.as<double>(); st.iter = pl->st_iter.as<int>(); st.iterc = pl->st_iterc.as<int>();
  st.done = pl->st_done.as<int>();
  PassArgs& pa = f.pa;
  pa.X = pl->X.as<float2>(); pa.Xlo = pl->Xlo.as<float2>(); pa.nu2 = pl->nu2.as<double>(); pa.P = f.dP; pa.nu_fit = pl->nu_fit.as<double>();
  pa.Ssn = pl->Ssn.as<double>(); pa.sigma = pl->sigma.as<double>(); pa.csum = pl->csum.as<double>(); pa.st = st;
  pa.s0 = 0; pa.nchan = nchan; pa.N = N; pa.nhalf = pl->anyn ? pl->L : 0; pa.njn = pl->njn.as<int>();
  const ModelRows mr{f.dmidx, nchan};
  pa.mr = mr;
  UpdateArgs& ua = f.ua;
  memset(&ua, 0, sizeof ua);
  ua.csum = pl->csum.as<double>(); ua.Ssn = pl->Ssn.as<double>(); ua.Sdn = pl->Sdn.as<double>(); ua.nu2 = pl->nu2.as<double>();
  ua.freqs = pl->freqs.as<double>(); ua.P = f.dP; ua.nu_fit = pl->nu_fit.as<double>(); ua.nu_outs = f.dnuouts;
  ua.nok = pl->nok.as<int>(); ua.st = st;
  ua.params = pl->o_params.as<double>(); ua.param_errs = pl->o_perrs.as<double>(); ua.nu_out = pl->o_nuout.as<double>();
  ua.cov = pl->o_cov.as<double>(); ua.chi2 = pl->o_chi2.as<double>(); ua.red_chi2 = pl->o_rchi2.as<double>();
  ua.snr = pl->o_snr.as<double>(); ua.nfeval = pl->o_nfev.as<int>(); ua.rc = pl->o_rc.as<int>();
  ua.scales = pl->o_scales.as<double>(); ua.scale_errs = pl->o_serrs.as<double>(); ua.channel_snrs = pl->o_csnr.as<double>();
  ua.s0 = 0; ua.nchan = nchan; ua.nbin = pl->nbin; ua.max_iter = f.max_iter; ua.semantics = args->semantics;
  ua.fit_phi = ff[0] ? 1 : 0; ua.fit_dm = ff[1] ? 1 : 0; ua.is_toa = args->is_toa; ua.tol = f.tol; ua.box = f.box;
  ua.model_steps = pl->model_steps; ua.tol_model = (args->tol > 0 && args->tol < 1e-4) ? args->tol : 1e-4;
  ua.mr = mr;
  if (!f.general) return;
  Pass5Args& p5 = f.p5;
  p5.X = pl->X.as<float2>(); p5.Xlo = pl->Xlo.as<float2>(); p5.mpow = pl->mpow.as<double>(); p5.nu2 = pl->nu2.as<double>(); p5.lgf = pl->lgf.as<double>();
  p5.freqs = pl->freqs.as<double>(); p5.P = f.dP; p5.nu_fit = pl->nu_fit.as<double>(); p5.Ssn = pl->Ssn.as<double>();
  p5.sigma = pl->sigma.as<double>(); p5.csum = pl->csum.as<double>(); p5.st = st; p5.s0 = 0; p5.nchan = nchan;
  p5.log10_tau = args->log10_tau; p5.nhalf = pl->anyn ? pl->L : 0; p5.nj = N / 16; p5.cstride = 1; p5.njn = pl->njn.as<int>();
  p5.mr = mr; p5.njm = nullptr;
  Update5Args& u5 = f.u5;
  memset(&u5, 0, sizeof u5);
  u5.csum = pl->csum.as<double>(); u5.Sdn = pl->Sdn.as<double>(); u5.nu2 = pl->nu2.as<double>(); u5.lgf = pl->lgf.as<double>();
  u5.freqs = pl->freqs.as<double>(); u5.P = f.dP; u5.nu_fit = pl->nu_fit.as<double>(); u5.nu_outs = f.dnuouts;
  u5.nok = pl->nok.as<int>(); u5.st = st;
  u5.params = ua.params; u5.param_errs = ua.param_errs; u5.nu_out = ua.nu_out; u5.cov = ua.cov; u5.chi2 = ua.chi2;
  u5.red_chi2 = ua.red_chi2; u5.snr = ua.snr; u5.nfeval = ua.nfeval; u5.rc = ua.rc; u5.scales = ua.scales;
  u5.scale_errs = ua.scale_errs; u5.channel_snrs = ua.channel_snrs;
  u5.s0 = 0; u5.nchan = nchan; u5.nbin = pl->nbin; u5.max_iter = f.max_iter; u5.log10_tau = args->log10_tau;
  u5.option = args->option; u5.is_toa = args->is_toa; u5.tol = f.tol; u5.box = f.box;
  u5.taylor_finish = pl->model_steps != 1;
  for (int i = 0; i < 5; ++i) u5.flags[i] = ff[i] ? 1 : 0;
  u5.coarse = 0; u5.ctol = 0.0; u5.cstride = 1;
  u5.mr = mr;
}

// per-subint scalars, the start state of fits from caller-supplied values, the FFTFIT grid
static int fit_prep(pp_plan* pl, FitCall& f) {
  const int nsub = f.nsub;
  PrepArgs p;
  p.freqs = pl->freqs.as<double>(); p.mask = f.dmask; p.weights = f.dw; p.snrs = f.dsnrs; p.nu_fits_in = f.dnufits;
  p.nu_fit = pl->nu_fit.as<double>(); p.nu_mean = pl->nu_mean.as<double>(); p.wsum = pl->wsum.as<double>();
  p.nok = pl->nok.as<int>(); p.nsub = nsub; p.nchan = pl->nchan; p.nu_fit_mode = f.args->nu_fit_mode;
  p.mr = ModelRows{f.dmidx, pl->nchan};
  k_prep<<<(nsub + 3) / 4, 128, 0, pl->stream>>>(p);
  pl->stats.launches++;
  if (!f.want_guess) {
    k_init_state<<<(nsub + 127) / 128, 128, 0, pl->stream>>>(f.st, f.dinit, 0, nsub);
    if (f.box.on) k_clamp_state<<<(nsub + 127) / 128, 128, 0, pl->stream>>>(f.st, f.box, 0, nsub);
    pl->stats.launches++;
    CK(cudaMemsetAsync(pl->o_lag.p, 0xff, sizeof(int) * nsub, pl->stream));
  }
  if (f.want_guess && grid_table(pl, f.Ns, &f.table)) return -2;
  return 0;
}

// host data: chunk c's rows into staging buffer c & 1 on the copy stream, once the kernels that read it last are done
static cudaError_t issue_copy(pp_plan* pl, const FitCall& f, int c) {
  const int b = c & 1;
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0;
  cudaError_t e = cudaStreamWaitEvent(pl->copy_stream, pl->ev_free[b], 0);
  if (e != cudaSuccess) return e;
  // float64 rows from pageable memory are rounded to float32 by the host threads that stage them anyway (half
  // the bytes over PCIe); from page-locked memory they cross as they are and a kernel on the copy stream rounds
  const bool narrow = f.f64 && h2d_stages((size_t)ns * f.src_bytes, f.data_pinned);
  void* dst = (f.f64 && !narrow) ? pl->data_stage64[b].p : pl->data_stage[b].p;
  e = h2d_any(pl, dst, f.data + (size_t)s0 * f.src_bytes, (size_t)ns * f.src_bytes, f.data_pinned, pl->copy_stream, narrow);
  if (e != cudaSuccess) return e;
  if (f.f64 && !narrow) {
    cvt_f64_f32(dst, pl->data_stage[b].p, (size_t)ns * pl->nchan * (pl->nbin / 2), pl->copy_stream);
    pl->stats.launches++;
  }
  return cudaEventRecord(pl->ev_copy[b], pl->copy_stream);
}

// chunk c's spectra from the caller's device rows or from the staging buffer the copy stream fills (the next chunk's
// copy is issued first)
static int fit_spectra(pp_plan* pl, const FitCall& f, int c) {
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0, nchan = pl->nchan, N = pl->N, nchunks = (int)f.cstart.size() - 1;
  const char* dchunk = f.data;
  if (f.data_on_device && f.f64) {   // round the chunk to float32 next to the kernels that read it
    cvt_f64_f32(f.data + (size_t)s0 * f.src_bytes, pl->data_stage[c & 1].p, (size_t)ns * pl->nchan * (pl->nbin / 2), pl->stream);
    pl->stats.launches++;
  }
  if (!f.data_on_device) {
    if (c + 1 < nchunks) CK(issue_copy(pl, f, c + 1));
    CK(cudaStreamWaitEvent(pl->stream, pl->ev_copy[c & 1], 0));
  }
  // kernels index data with the global subint number: bias the base pointer of the staged chunk
  if (!f.data_on_device || f.f64) dchunk = pl->data_stage[c & 1].as<char>() - (size_t)s0 * f.sub_bytes;
  SpanGuard g(pl, SP_SPECTRA);
  SpectraArgs a;
  a.data = dchunk; a.dat_scl = f.dscl; a.dat_offs = f.doffs;
  a.mconj64 = pl->mconj64.as<cx<double>>(); a.mconj32 = pl->mconj32.as<cx<float>>();
  a.pn = pl->pn.as<double>(); a.nu2 = pl->nu2.as<double>();
  a.errs = f.derrs; a.mask = f.dmask; a.weights = f.dw; a.P = f.dP; a.DMg = f.ddmg; a.nu_mean = pl->nu_mean.as<double>();
  a.X = pl->X.as<float2>(); a.Xlo = pl->Xlo.as<float2>(); a.partial = f.want_guess ? pl->partial.as<float2>() : nullptr;
  a.D = f.want_align ? pl->Dspec.as<float2>() : nullptr; a.Ddc = f.want_align ? pl->Ddc.as<double>() : nullptr;
  a.sigma = pl->sigma.as<double>(); a.Ssn = pl->Ssn.as<double>(); a.Sdn = pl->Sdn.as<double>();
  a.tw8 = pl->tw8.as<cx<double>>();
  a.s0 = s0; a.nchan = nchan; a.G = f.G; a.nparts = f.nparts;
  a.dspec = nullptr; a.ddc = nullptr; a.nhalf = 0; a.kc_true = 0; a.njn = pl->njn.as<int>();
  a.mr = ModelRows{f.dmidx, nchan};
  if (pl->anyn) {   // rows transformed by Bluestein into the spectrum scratch, then the same emit code
    if (c == 0) {
      CK(pl->any_spec.need(sizeof(double2) * (size_t)f.chunk * nchan * N));
      CK(pl->any_dc.need(sizeof(double) * (size_t)f.chunk * nchan));
    }
    if (launch_fwd_any(pl, dchunk + (size_t)s0 * f.sub_bytes, f.i16, f.i16 ? f.dscl + (size_t)s0 * nchan : nullptr,
                       f.i16 ? f.doffs + (size_t)s0 * nchan : nullptr, (long)ns * nchan, pl->any_spec.as<cx<double>>(),
                       pl->any_dc.as<double>())) return -2;
    a.dspec = pl->any_spec.as<cx<double>>(); a.ddc = pl->any_dc.as<double>();
    a.nhalf = pl->L; a.kc_true = (3 * (pl->L + 1)) / 4;
    DISPATCH_N(N, (k_spectra<NN, SpecPlan<NN>, false, true><<<dim3(f.gx, ns), SpecPlan<NN>::kThreads, 0, pl->stream>>>(a)));
  } else if (N == 1024) {
    launch_spectra16(f.i16, f.want_guess, f.want_align, dim3(f.gx, ns), pl->stream, a);
  } else {
    DISPATCH_N(N, launch_spectra<NN>(f.i16, dim3(f.gx, ns), pl->stream, a));
  }
  pl->stats.launches++;
  return 0;
}

static int fit_guess(pp_plan* pl, const FitCall& f, int c) {
  if (!f.want_guess) return 0;
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0, N = pl->N;
  SpanGuard g(pl, SP_GUESS);
  GuessArgs ga;
  memset(&ga, 0, sizeof ga);
  ga.partial = pl->partial.as<float2>(); ga.mconj = pl->mmean.as<float2>(); ga.nparts = f.nparts; ga.nmodel = 1;
  if (f.dmidx) {   // each subint's own model: its mean spectrum and its cut-off
    ga.model = f.dmidx; ga.nused_of = pl->kmax_dev.as<int>(); ga.tmpl_by_model = 1;
  }
  if (f.dmask) {   // the guess template is the mean model over the subint's usable channels (pptoas.py:446, 454)
    CK(pl->mmean_sub.need(sizeof(float2) * (size_t)f.chunk * N));
    k_model_mean_masked<<<dim3((N + 127) / 128, ns), 128, 0, pl->stream>>>(
        pl->mconj64.as<cx<double>>(), f.dmask, pl->mmean.as<float2>(), pl->mmean_sub.as<float2>(), s0, pl->nchan, N,
        ModelRows{f.dmidx, pl->nchan});
    pl->stats.launches++;
    ga.mconj = pl->mmean_sub.as<float2>();
    ga.nmodel = ns;  // one template per subint of the chunk
    ga.tmpl_by_model = 0;
  }
  ga.N = N; ga.Ns = f.Ns; ga.wsum = pl->wsum.as<double>(); ga.noise = nullptr; ga.table = f.table; ga.s0 = s0;
  ga.nhalf = pl->anyn ? pl->L : 0;
  ga.nused = pl->kmax_used[0];   // the mean model has no power beyond the largest channel cut-off
  ga.phase = pl->o_phig.as<double>(); ga.lag = pl->o_lag.as<int>();
  ga.x = f.st.x; ga.DMg = f.ddmg; ga.P = f.dP; ga.nu_mean = pl->nu_mean.as<double>(); ga.nu_fit = pl->nu_fit.as<double>();
  ga.polish_tol = 1e-6;   // a start value (the last step is still applied): the Newton solver refines it
  ga.init = nullptr; ga.scat = f.dscat; ga.log10_tau = f.args->log10_tau; ga.fit_scat = f.args->fit_flags[3] ? 1 : 0;
  k_guess<<<ns, 256, sizeof(double2) * N, pl->stream>>>(ga);
  k_reset_state<<<(ns + 127) / 128, 128, 0, pl->stream>>>(f.st, s0, ns);
  pl->stats.launches += 2;
  if (f.box.on) { k_clamp_state<<<(ns + 127) / 128, 128, 0, pl->stream>>>(f.st, f.box, s0, ns); pl->stats.launches++; }
  return 0;
}

static void launch_update5(pp_plan* pl, const FitCall& f, int ns) {   // many channels: more threads per subint for the per-channel chain rule
  if (pl->nchan >= 1024) k_update5<256><<<ns, 256, 0, pl->stream>>>(f.u5);
  else k_update5<128><<<ns, 128, 0, pl->stream>>>(f.u5);
}

// the count of the chunk's subints that `count` finds still running, read back on the host
static int poll_running(pp_plan* pl, void (*count)(SolverState, int, int, int*), const FitCall& f, int s0, int ns,
                        int* running) {
  count<<<1, 256, 0, pl->stream>>>(f.st, s0, ns, pl->running.as<int>());
  pl->stats.launches++;
  *running = 0;
  CK(cudaMemcpyAsync(running, pl->running.p, sizeof(int), cudaMemcpyDeviceToHost, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

// Coarse stage of the general solver: Newton iterations on the objective of the low harmonics only (those
// that hold coarse_frac of the model's phase information: a fraction of a pass each) carry the start values
// to within a fraction of a sigma of the optimum; the full-resolution iterations then need two passes.
// With several models the levels are chosen per model present in the chunk, from that model's first subint of
// the chunk: a subint gets the levels a call with its model alone would give it, and sits out the others.
static int fit_coarse(pp_plan* pl, FitCall& f, int c) {
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0, nchan = pl->nchan, N = pl->N, NJ = N / 16;
  const pp_fit_args_t* args = f.args;
  f.coarse_nj = 0;
  if (!(f.general && f.max_iter > 0 && pl->coarse_frac > 0.0 && pl->model_steps != 1 && N >= 128)) return 0;
  // where the information sits, with the scattering of the (model's) first subint at its start values
  const uint8_t* ff = args->fit_flags;
  const bool scat = ff[3] || ff[4] || f.dscat || f.dinit;
  std::vector<int> models;   // the chunk's models, in order of first appearance (f.cfirst: their first subints)
  f.cfirst.clear();
  if (f.dmidx) {
    std::vector<char> seen(pl->nmodel, 0);
    for (int s = s0; s < s0 + ns; ++s) {
      const int m = f.hmidx[s];
      if (!seen[m]) { seen[m] = 1; models.push_back(m); f.cfirst.push_back(s); }
    }
  }
  const int nm = f.dmidx ? (int)models.size() : 1;
  CK(pl->minfo.need(sizeof(double) * NJ * nm));
  pl->model_info.assign((size_t)NJ * nm, 0.0);
  if (f.dmidx) {
    CK(pl->coarse_first.need(sizeof(int) * nm));
    CK(cudaMemcpyAsync(pl->coarse_first.p, f.cfirst.data(), sizeof(int) * nm, cudaMemcpyHostToDevice, pl->stream));
    k_model_info<<<dim3(NJ, nm), 256, 0, pl->stream>>>(pl->mpow.as<double>(), pl->lgf.as<double>(), scat ? f.st.x : nullptr,
                                                        pl->nu_fit.as<double>(), args->log10_tau, pl->minfo.as<double>(),
                                                        nchan, N, ModelRows{f.dmidx, nchan}, pl->coarse_first.as<int>());
  } else {
    k_model_info<<<NJ, 256, 0, pl->stream>>>(pl->mpow.as<double>(), pl->lgf.as<double>(), scat ? f.st.x + (size_t)s0 * 5 : nullptr,
                                             pl->nu_fit.as<double>() + (size_t)s0 * 3, args->log10_tau,
                                             pl->minfo.as<double>(), nchan, N, ModelRows{nullptr, nchan}, nullptr);
  }
  pl->stats.launches++;
  CK(cudaMemcpyAsync(pl->model_info.data(), pl->minfo.p, sizeof(double) * NJ * nm, cudaMemcpyDeviceToHost, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));
  // Two levels: most of the iterations run on a cheaper objective still -- the harmonics that hold coarse_frac0
  // of the information (when that is clearly fewer) of every cstride-th channel -- the second level then needs
  // one or two.  A level is left once its Newton step is below ctol sigma (the step is still taken): the next
  // level, or the full-resolution iterations, start next to that level's optimum either way.
  // Per model: the groups of level A (0: no such level) and of level B (0: no coarse stage).
  const int cst = nchan >= 2048 ? 8 : (nchan >= 512 ? 4 : (nchan >= 128 ? 2 : 1));
  std::vector<int> njA(nm, 0), njB(nm, 0);
  bool anyA = false;
  for (int i = 0; i < nm; ++i) {
    const double* info = pl->model_info.data() + (size_t)i * NJ;
    const int coarse_nj = choose_coarse(info, pl->coarse_frac, N);
    if (coarse_nj == 0) continue;
    f.coarse_nj = std::max(f.coarse_nj, coarse_nj);
    int nj0 = choose_coarse(info, std::min(0.65, pl->coarse_frac), N);
    if (!(nj0 > 0 && 3 * nj0 <= 2 * coarse_nj)) nj0 = coarse_nj;
    if (nj0 < coarse_nj || cst > 1) { njA[i] = nj0; anyA = true; }
    njB[i] = coarse_nj;
  }
  if (f.coarse_nj == 0) return 0;
  struct { int cstride; double ctol; const std::vector<int>* nj; } levels[2];
  int nlev = 0;
  if (anyA) levels[nlev++] = {cst, 2.0, &njA};
  levels[nlev++] = {1, 1.0, &njB};
  if (f.dmidx) {   // the levels' groups by model number, read by k_pass5 through the subint's model
    f.cnjm.assign((size_t)2 * pl->nmodel, 0);
    for (int lv = 0; lv < nlev; ++lv)
      for (int i = 0; i < nm; ++i) f.cnjm[(size_t)lv * pl->nmodel + models[i]] = (*levels[lv].nj)[i];
    CK(pl->coarse_njm.need(sizeof(int) * 2 * pl->nmodel));
    CK(cudaMemcpyAsync(pl->coarse_njm.p, f.cnjm.data(), sizeof(int) * 2 * pl->nmodel, cudaMemcpyHostToDevice, pl->stream));
  }
  Pass5Args& p5 = f.p5;
  Update5Args& u5 = f.u5;
  u5.coarse = 1;
  for (int lv = 0; lv < nlev; ++lv) {
    const int max_coarse = std::min(f.max_iter, 12);
    const std::vector<int>& nj = *levels[lv].nj;
    const bool sitout = std::find(nj.begin(), nj.end(), 0) != nj.end();   // some model has no such level
    if (f.dmidx) { p5.nj = 0; p5.njm = pl->coarse_njm.as<int>() + (size_t)lv * pl->nmodel; }
    else p5.nj = nj[0];
    p5.cstride = u5.cstride = levels[lv].cstride; u5.ctol = levels[lv].ctol;
    const int gx5 = ((nchan + p5.cstride - 1) / p5.cstride + 31) / 32;
    if (sitout) {
      k_coarse_sitout<<<(ns + 127) / 128, 128, 0, pl->stream>>>(f.st, p5.mr, p5.njm, s0, ns, 1);
      pl->stats.launches++;
    }
    mark(f, "coarse level: %d of %d harmonic groups, every %d-th channel", *std::max_element(nj.begin(), nj.end()), NJ, p5.cstride);
    for (int it = 0; it < max_coarse; ++it) {
      {
        SpanGuard g(pl, SP_COARSE);
        DISPATCH_N(N, k_pass5<NN><<<dim3(gx5, ns), 256, Pass5Ring<NN>::kBytes, pl->stream>>>(p5));
        launch_update5(pl, f, ns);
      }
      pl->stats.launches += 2;
      pl->stats.coarse_launches++;
      // the first level starts far from its optimum (three iterations before asking), the second next to it
      if (it >= (lv == 0 ? 2 : 0) && it + 1 < max_coarse) {
        int running;
        if (poll_running(pl, k_count_coarse, f, s0, ns, &running)) return -2;
        if (running == 0) break;
      }
    }
    k_coarse_end<<<(ns + 127) / 128, 128, 0, pl->stream>>>(f.st, s0, ns);
    pl->stats.launches++;
    if (sitout) {
      k_coarse_sitout<<<(ns + 127) / 128, 128, 0, pl->stream>>>(f.st, p5.mr, p5.njm, s0, ns, 0);
      pl->stats.launches++;
    }
  }
  // (k_update5 reads ctol only in the coarse stage)
  p5.nj = NJ; p5.njm = nullptr; p5.cstride = u5.cstride = 1; u5.coarse = 0; u5.ctol = 0.0;
  return 0;
}

// queue the device-to-host copies of the results of chunk f.pending_out (if any) on the copy stream
static int enqueue_results(pp_plan* pl, FitCall& f) {
  const int c = f.pending_out;
  if (c < 0) return 0;
  f.pending_out = -1;
  const pp_fit_out_t* out = f.out;
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0, nchan = pl->nchan;
  CK(cudaStreamWaitEvent(pl->copy_stream, pl->ev_chunk[c], 0));
  cudaStream_t cs = pl->copy_stream;
  const size_t o1 = (size_t)s0, n1 = (size_t)ns, oc = (size_t)s0 * nchan, ncn = (size_t)ns * nchan;
  if (copy_out_at(cs, out->params, pl->o_params.as<double>(), o1 * 5, n1 * 5)) return -2;
  if (copy_out_at(cs, out->param_errs, pl->o_perrs.as<double>(), o1 * 5, n1 * 5)) return -2;
  if (copy_out_at(cs, out->nu_out, pl->o_nuout.as<double>(), o1 * 3, n1 * 3)) return -2;
  if (copy_out_at(cs, out->cov, pl->o_cov.as<double>(), o1 * 25, n1 * 25)) return -2;
  if (copy_out_at(cs, out->chi2, pl->o_chi2.as<double>(), o1, n1)) return -2;
  if (copy_out_at(cs, out->red_chi2, pl->o_rchi2.as<double>(), o1, n1)) return -2;
  if (copy_out_at(cs, out->snr, pl->o_snr.as<double>(), o1, n1)) return -2;
  if (copy_out_at(cs, out->nfeval, pl->o_nfev.as<int>(), o1, n1)) return -2;
  if (copy_out_at(cs, out->return_code, pl->o_rc.as<int>(), o1, n1)) return -2;
  if (copy_out_at(cs, out->scales, pl->o_scales.as<double>(), oc, ncn)) return -2;
  if (copy_out_at(cs, out->scale_errs, pl->o_serrs.as<double>(), oc, ncn)) return -2;
  if (copy_out_at(cs, out->channel_snrs, pl->o_csnr.as<double>(), oc, ncn)) return -2;
  if (copy_out_at(cs, out->noise, pl->sigma.as<double>(), oc, ncn)) return -2;
  if (copy_out_at(cs, out->lag_index, pl->o_lag.as<int>(), o1, n1)) return -2;
  if (f.want_guess && copy_out_at(cs, out->phi_guess, pl->o_phig.as<double>(), o1, n1)) return -2;
  if (copy_out_at(cs, out->chan_sums, pl->csum.as<double>(), oc * kNCsum, ncn * kNCsum)) return -2;
  return 0;
}

// the full-resolution passes of chunk c, launched while some subint is still running (polled)
static int fit_passes(pp_plan* pl, FitCall& f, int c) {
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0, nchan = pl->nchan, N = pl->N;
  for (int it = 0; it < f.n_launch_iter; ++it) {
    {
      SpanGuard g(pl, SP_PASS);
      if (f.general) { DISPATCH_N(N, k_pass5<NN><<<dim3((nchan + 31) / 32, ns), 256, Pass5Ring<NN>::kBytes, pl->stream>>>(f.p5)); }
      else { DISPATCH_N(N, k_pass2<NN><<<dim3((nchan + 31) / 32, ns), 256, Pass2Ring<NN>::kBytes, pl->stream>>>(f.pa)); }
    }
    {
      SpanGuard g(pl, SP_UPDATE);
      if (f.general) launch_update5(pl, f, ns);
      else k_update2<<<ns, 128, 0, pl->stream>>>(f.ua);
    }
    pl->stats.launches += 2;
    pl->stats.pass_launches++;
    // data-dependent number of passes: poll the count of unfinished subints (an empty
    // launch of the full grid costs ~80 us, the poll ~20 us)
    // (when the previous chunk needed a third pass this one most likely does too: launch it
    // without asking first)
    const bool poll = f.general ? (it >= (f.coarse_nj > 0 ? 1 : 3)) : (it >= 2 || (it == 1 && !f.expect_third));
    // this chunk's first passes are queued: now the previous chunk's copies
    if (it == 1 && enqueue_results(pl, f)) return -2;
    if (poll && it + 1 < f.n_launch_iter) {
      int running;
      if (poll_running(pl, k_count_running, f, s0, ns, &running)) return -2;
      if (!f.general && it == 1) f.expect_third = running > 0;
      if (!f.general && it == 2 && running == 0) f.expect_third = true;   // needed exactly three
      if (running == 0) break;
    }
  }
  return enqueue_results(pl, f);   // (single-pass calls never reach it == 1)
}

// sum_s w_sn rotate(d_sn) with the fitted phi, DM of chunk c (ppalign.py:197-208)
static int fit_align_chunk(pp_plan* pl, const FitCall& f, int c) {
  if (!f.want_align) return 0;
  const int s0 = f.cstart[c], ns = f.cstart[c + 1] - s0, nchan = pl->nchan;
  AlignSpecArgs aa;
  aa.D = pl->Dspec.as<float2>(); aa.Ddc = pl->Ddc.as<double>(); aa.params = pl->o_params.as<double>();
  aa.nu_out = pl->o_nuout.as<double>(); aa.P = f.dP; aa.scales = pl->o_scales.as<double>(); aa.sigma = pl->sigma.as<double>();
  aa.rc = pl->o_rc.as<int>(); aa.nu2 = pl->nu2.as<double>(); aa.acc = pl->al_acc.as<double2>();
  aa.wsum = pl->al_wparts.as<double>(); aa.s0 = s0; aa.ns = ns; aa.nchan = nchan;
  DISPATCH_N(pl->N, k_align_spec<NN><<<dim3(nchan, f.align_nsplit), NN / 8, 0, pl->stream>>>(aa));
  pl->stats.launches++;
  return 0;
}

// the aligned portrait from the chunks' partial sums, and its copies to the caller
static int fit_align_finish(pp_plan* pl, const FitCall& f) {
  if (!f.want_align) return 0;
  const int nchan = pl->nchan, N = pl->N;
  AlignFinishArgs fa;
  fa.acc = pl->al_acc.as<double2>(); fa.wsum_parts = pl->al_wparts.as<double>(); fa.aligned = pl->al_out.as<double>();
  fa.wsum = pl->al_wsum.as<double>(); fa.twN = pl->twN64.p; fa.tw2N = pl->tw2N64.p;
  fa.nchan = nchan; fa.nsplit = f.align_nsplit;
  if (pl->anyn) {
    CK(pl->any_spec2.need(sizeof(double2) * (size_t)nchan * N));
    CK(pl->any_dc2.need(sizeof(double) * (size_t)nchan));
    k_align_reduce_any<<<nchan, 256, 0, pl->stream>>>(fa.acc, fa.wsum_parts, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>(),
                                                      fa.wsum, nchan, N, f.align_nsplit);
    if (launch_inv_any(pl, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>(), fa.aligned, nchan, true)) return -2;
  } else {
    DISPATCH_N(N, (k_align_finish<NN><<<row_ctas<NN>(nchan), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(fa)));
  }
  pl->stats.launches++;
  if (copy_out_at(pl->stream, f.out->align_sum, pl->al_out.as<double>(), 0, (size_t)nchan * pl->nbin)) return -2;
  if (copy_out_at(pl->stream, f.out->align_wsum, pl->al_wsum.as<double>(), 0, (size_t)nchan)) return -2;
  return 0;
}

// the model of each subint, checked on the host before any kernel reads it (a device index costs one small copy)
static int fit_model_index(pp_plan* pl, FitCall& f, const int32_t* model_index) {
  if (!model_index) {
    if (pl->nmodel > 1) return fail(-1, "model_index is required: the plan holds %d models", pl->nmodel);
    return 0;
  }
  const int nsub = f.nsub;
  f.hmidx.resize(nsub);
  const bool dev = is_device_ptr(model_index);
  if (dev) {
    CK(cudaMemcpyAsync(f.hmidx.data(), model_index, sizeof(int) * nsub, cudaMemcpyDeviceToHost, pl->stream));
    CK(cudaStreamSynchronize(pl->stream));
  } else {
    memcpy(f.hmidx.data(), model_index, sizeof(int) * nsub);
  }
  for (int s = 0; s < nsub; ++s)
    if (f.hmidx[s] < 0 || f.hmidx[s] >= pl->nmodel)
      return fail(-1, "model_index[%d] = %d is outside [0, %d)", s, f.hmidx[s], pl->nmodel);
  if (dev) f.dmidx = model_index;
  else {
    CK(pl->in_models.need(sizeof(int) * nsub));
    CK(cudaMemcpyAsync(pl->in_models.p, f.hmidx.data(), sizeof(int) * nsub, cudaMemcpyHostToDevice, pl->stream));
    f.dmidx = pl->in_models.as<int>();
  }
  return 0;
}

extern "C" int pp_fit_batch(pp_plan_t* pl, const pp_fit_args_t* args, const pp_fit_out_t* out) {
  return pp_fit_batch_models(pl, args, nullptr, out);
}

extern "C" int pp_fit_batch_models(pp_plan_t* pl, const pp_fit_args_t* args, const int32_t* model_index,
                                   const pp_fit_out_t* out) {
  if (!pl || !args || !out) return fail(-1, "NULL argument");
  if (!pl->model_set) return fail(-1, "pp_set_model must be called before pp_fit_batch");
  if (!args->data || !args->P) return fail(-1, "data and P are required");
  const bool i16 = args->data_type == PP_DATA_I16, f64 = args->data_type == PP_DATA_F64;
  if (args->data_type != PP_DATA_F32 && !i16 && !f64) return fail(-1, "unknown data_type %d", args->data_type);
  if (i16 && (!args->dat_scl || !args->dat_offs)) return fail(-1, "int16 data need dat_scl and dat_offs");
  if (args->nsub < 1) return fail(-1, "nsub must be >= 1");
  const uint8_t* ff = args->fit_flags;
  if (!ff[0] && !ff[1] && !ff[2] && !ff[3] && !ff[4]) return fail(-1, "nothing to fit");
  // The (phi, DM) kernels apply when GM, tau, alpha are neither fit nor non-zero.
  bool general = ff[2] || ff[3] || ff[4] || args->log10_tau;
  if (!general && args->init) {
    if (is_device_ptr(args->init)) general = true;   // cannot inspect cheaply: take the general path
    else
      for (int i = 0; i < args->nsub && !general; ++i)
        if (args->init[(size_t)i * 5 + 2] != 0.0 || args->init[(size_t)i * 5 + 3] != 0.0) general = true;
  }
  if (!general && args->scat_guess) general = true;
  if (general && args->semantics == PP_SEM_FIT_PORTRAIT)
    return fail(-1, "PP_SEM_FIT_PORTRAIT is defined for the (phi, DM) fit only");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  FitCall f;
  f.tr0 = std::chrono::steady_clock::now();
  f.args = args; f.out = out; f.general = general; f.i16 = i16; f.f64 = f64; f.nsub = args->nsub;
  f.Ns = args->Ns > 0 ? args->Ns : 100;
  if (f.Ns < 2) return fail(-1, "Ns must be >= 2");
  if (out->align_sum && pl->nmodel > 1) return fail(-1, "align_sum needs one model (the plan holds %d)", pl->nmodel);
  if (int rc = fit_model_index(pl, f, model_index)) return rc;
  // passes are launched only while some subint is still running (polled), so a generous limit costs
  // nothing for batches started from the FFTFIT guess (1-2 passes) and lets caller-supplied start
  // values far from the optimum converge (10-14 passes from 0.05-0.08 turn away, tools/far_start_probe.py)
  const int dflt_iter = 40;
  f.max_iter = args->max_iter > 0 ? args->max_iter : (args->max_iter < 0 ? -1 : dflt_iter);
  f.n_launch_iter = f.max_iter < 0 ? 1 : (general ? f.max_iter + 1 : f.max_iter);
  // (phi, DM): the epilogue applies the last Newton step through a second-order Taylor update of
  // the per-channel sums, so stopping at 1e-2 sigma leaves < 2e-5 sigma (measured, tools/gpu_tol.py);
  // the general solver re-evaluates at the final point instead and keeps 1e-3.
  f.tol = args->tol > 0 ? args->tol : (general ? 1e-3 : 1e-2);

  if (int rc = fit_stage_inputs(pl, f)) return rc;
  if (int rc = fit_workspace(pl, f)) return rc;
  fit_kernel_args(pl, f);
  cudaEvent_t ev_t0 = nullptr;
  if (pl->timing) { ev_t0 = get_event(pl); CK(cudaEventRecord(ev_t0, pl->stream)); }
  if (int rc = fit_prep(pl, f)) return rc;
  if (!f.data_on_device) {   // host data: the first chunk's copy starts right away
    // the staging buffers are free at the start
    CK(cudaEventRecord(pl->ev_free[0], pl->stream));
    CK(cudaEventRecord(pl->ev_free[1], pl->stream));
    CK(issue_copy(pl, f, 0));
  }

  mark(f, "before chunk loop");
  const int nchunks = (int)f.cstart.size() - 1;
  for (int c = 0; c < nchunks; ++c) {
    mark(f, "chunk %d (%d subints)", c, f.cstart[c + 1] - f.cstart[c]);
    if (int rc = fit_spectra(pl, f, c)) return rc;
    if (!f.data_on_device) CK(cudaEventRecord(pl->ev_free[c & 1], pl->stream));
    if (int rc = fit_guess(pl, f, c)) return rc;
    f.pa.s0 = f.ua.s0 = f.p5.s0 = f.u5.s0 = f.cstart[c];
    if (int rc = fit_coarse(pl, f, c)) return rc;
    if (int rc = fit_passes(pl, f, c)) return rc;
    if (int rc = fit_align_chunk(pl, f, c)) return rc;
    // the chunk is done at this point of the stream; its results go back on the copy stream
    // while the next chunk computes.  The (host-side) enqueue of those copies is deferred until
    // the next chunk's first kernels are in the queue, so that the device does not idle over it.
    while ((int)pl->ev_chunk.size() <= c) {
      cudaEvent_t e;
      CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      pl->ev_chunk.push_back(e);
    }
    CK(cudaEventRecord(pl->ev_chunk[c], pl->stream));
    f.pending_out = c;
  }
  if (enqueue_results(pl, f)) return -2;
  mark(f, "all chunks queued");
  CK(cudaGetLastError());
  if (pl->timing) {
    cudaEvent_t ev_t1 = get_event(pl);
    CK(cudaEventRecord(ev_t1, pl->stream));
    pl->spans.push_back({SP_TOTAL, ev_t0, ev_t1});
  }
  if (int rc = fit_align_finish(pl, f)) return rc;
  // ---- results (per-chunk copies were queued on the copy stream) -------------------------
  if (!f.want_guess && out->phi_guess && f.dinit) {
    // phi_guess = init[:,0]
    CK(cudaMemcpy2DAsync(out->phi_guess, sizeof(double), f.dinit, 5 * sizeof(double), sizeof(double), f.nsub,
                         is_device_ptr(out->phi_guess) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, pl->stream));
  }
  CK(cudaStreamSynchronize(pl->copy_stream));
  mark(f, "copy stream drained");
  CK(cudaStreamSynchronize(pl->stream));
  mark(f, "done");
  CK(cudaGetLastError());
  stats_end(pl);
  return 0;
}

// ----------------------------------------------------------------------------
// batched 1-D FFTFIT, rotation, noise
// ----------------------------------------------------------------------------
template <typename T> static const void* tw1(pp_plan* pl) { return sizeof(T) == 8 ? pl->twN64.p : pl->twN32.p; }
template <typename T> static const void* tw2(pp_plan* pl) { return sizeof(T) == 8 ? pl->tw2N64.p : pl->tw2N32.p; }

static int launch_rfft_rows(pp_plan* pl, const float* in, int nrows, float2* spec, int conj, double* noise, int bits,
                            int kc = -1, double2* spec64 = nullptr, double* dc64 = nullptr) {
  const int N = pl->N;
  if (pl->anyn) {   // Bluestein rows into the spectrum scratch, then float spectra / noise from it
    const int L = pl->L;
    CK(pl->any_spec2.need(sizeof(double2) * (size_t)nrows * N));
    CK(pl->any_dc2.need(sizeof(double) * (size_t)nrows));
    if (launch_fwd_any(pl, in, false, nullptr, nullptr, nrows, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>())) return -2;
    k_rows_from_spec<<<nrows, 256, 0, pl->stream>>>(pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>(), spec, noise, N, L,
                                                    kc >= 0 ? kc : (3 * (L + 1)) / 4, conj);
    pl->stats.launches++;
    return 0;
  }
  RowsArgs a;
  a.in = in; a.spec = spec; a.noise = noise; a.nrows = nrows; a.conj = conj;
  a.kc = kc >= 0 ? kc : (3 * (N + 1)) / 4;
  a.spec64 = spec64; a.dc64 = dc64;
  if (bits == 64) {
    a.twN = tw1<double>(pl); a.tw2N = tw2<double>(pl);
    DISPATCH_N(N, (k_rfft_rows<NN, double><<<row_ctas<NN>(nrows), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(a)));
  } else {
    a.twN = tw1<float>(pl); a.tw2N = tw2<float>(pl);
    DISPATCH_N(N, (k_rfft_rows<NN, float><<<row_ctas<NN>(nrows), 256, fft_smem_bytes<NN, float>(), pl->stream>>>(a)));
  }
  pl->stats.launches++;
  return 0;
}

static int pshift_impl(pp_plan_t* pl, const float* profiles, int32_t n, const float* models, int32_t nmodel,
                       const double* noise, int32_t Ns, bool general, double phi_lo, double phi_hi,
                       const pp_pshift_out_t* out) {
  if (!pl || !profiles || !models || !out) return fail(-1, "NULL argument");
  if (n < 1) return fail(-1, "n must be >= 1");
  if (nmodel < 1 || n % nmodel) return fail(-1, "nmodel must divide n (profile i is fit against model i mod nmodel)");
  if (Ns <= 0) Ns = 100;
  if (Ns < 2) return fail(-1, "Ns must be >= 2");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int N = pl->N;
  const float *dprof, *dmod;
  const double* dnoise;
  if (stage_in(pl, pl->rot_in, profiles, (size_t)n * pl->nbin, &dprof)) return -2;
  if (stage_in(pl, pl->model_stage, models, (size_t)nmodel * pl->nbin, &dmod)) return -2;
  if (stage_in(pl, pl->in_noise, noise, (size_t)n, &dnoise)) return -2;
  CK(pl->ps_spec.need(sizeof(float2) * (size_t)n * N));
  CK(pl->ps_mspec.need(sizeof(float2) * (size_t)nmodel * N));
  CK(pl->ps_phase.need(sizeof(double) * n)); CK(pl->ps_perr.need(sizeof(double) * n));
  CK(pl->ps_scale.need(sizeof(double) * n)); CK(pl->ps_serr.need(sizeof(double) * n));
  CK(pl->ps_snr.need(sizeof(double) * n)); CK(pl->ps_rchi2.need(sizeof(double) * n));
  CK(pl->ps_lag.need(sizeof(int) * n));
  const int bits = pl->fft_precision ? pl->fft_precision : 64;
  if (launch_rfft_rows(pl, dprof, n, pl->ps_spec.as<float2>(), 0, nullptr, bits)) return -2;
  if (launch_rfft_rows(pl, dmod, nmodel, pl->ps_mspec.as<float2>(), 1, nullptr, 64)) return -2;
  const double2* table = nullptr;
  if (general) { if (grid_table_general(pl, Ns, phi_lo, phi_hi, &table)) return -2; }
  else if (grid_table(pl, Ns, &table)) return -2;
  GuessArgs ga;
  memset(&ga, 0, sizeof ga);
  ga.grid_general = general ? 1 : 0; ga.phi_lo = phi_lo; ga.phi_step = (phi_hi - phi_lo) / (double)(Ns - 1);
  ga.partial = pl->ps_spec.as<float2>(); ga.mconj = pl->ps_mspec.as<float2>(); ga.nparts = 1; ga.nmodel = nmodel;
  ga.N = N; ga.Ns = Ns; ga.wsum = nullptr; ga.noise = dnoise; ga.table = table; ga.s0 = 0; ga.polish_tol = 1e-14;
  ga.nhalf = pl->anyn ? pl->L : 0;
  ga.phase = pl->ps_phase.as<double>(); ga.phase_err = pl->ps_perr.as<double>(); ga.scale = pl->ps_scale.as<double>();
  ga.scale_err = pl->ps_serr.as<double>(); ga.snr = pl->ps_snr.as<double>(); ga.red_chi2 = pl->ps_rchi2.as<double>();
  ga.lag = pl->ps_lag.as<int>();
  k_guess<<<n, 256, sizeof(double2) * N, pl->stream>>>(ga);
  pl->stats.launches++;
  CK(cudaGetLastError());
  if (copy_out_at(pl->stream, out->phase, pl->ps_phase.as<double>(), 0, (size_t)n)) return -2;
  if (copy_out_at(pl->stream, out->phase_err, pl->ps_perr.as<double>(), 0, (size_t)n)) return -2;
  if (copy_out_at(pl->stream, out->scale, pl->ps_scale.as<double>(), 0, (size_t)n)) return -2;
  if (copy_out_at(pl->stream, out->scale_err, pl->ps_serr.as<double>(), 0, (size_t)n)) return -2;
  if (copy_out_at(pl->stream, out->snr, pl->ps_snr.as<double>(), 0, (size_t)n)) return -2;
  if (copy_out_at(pl->stream, out->red_chi2, pl->ps_rchi2.as<double>(), 0, (size_t)n)) return -2;
  if (copy_out_at(pl->stream, out->lag_index, pl->ps_lag.as<int>(), 0, (size_t)n)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_fit_phase_shift_batch(pp_plan_t* pl, const float* profiles, int32_t n, const float* models, int32_t nmodel,
                                        const double* noise, int32_t Ns, const pp_pshift_out_t* out) {
  return pshift_impl(pl, profiles, n, models, nmodel, noise, Ns, false, -0.5, 0.5, out);
}

extern "C" int pp_fit_phase_shift_batch_bounds(pp_plan_t* pl, const float* profiles, int32_t n, const float* models,
                                               int32_t nmodel, const double* noise, int32_t Ns, double phi_lo,
                                               double phi_hi, const pp_pshift_out_t* out) {
  if (!(phi_hi > phi_lo)) return fail(-1, "bounds: need phi_lo < phi_hi");
  const bool dflt = phi_lo == -0.5 && phi_hi == 0.5;
  return pshift_impl(pl, profiles, n, models, nmodel, noise, Ns, !dflt, phi_lo, phi_hi, out);
}

// where an entry point writes its n results: the caller's array when it is device memory, else `stage`;
// finish_out copies staged results back to the caller
template <typename T> static int stage_out(DBuf& stage, T* dst, size_t n, T** dev) {
  *dev = dst;
  if (is_device_ptr(dst)) return 0;
  CK(stage.need(sizeof(T) * n));
  *dev = stage.as<T>();
  return 0;
}
template <typename T> static int finish_out(pp_plan* pl, T* dst, const T* dev, size_t n) {
  if (dev != dst) CK(cudaMemcpyAsync(dst, dev, sizeof(T) * n, cudaMemcpyDeviceToHost, pl->stream));
  return 0;
}

// device scalars 0.0 (gm_zero) and 1.0 (gm_one): phase, DM and P, nu_ref of a rotation by nothing
static int unit_scalars(pp_plan* pl) {
  if (pl->gm_zero.p) return 0;
  const double z = 0.0, o = 1.0;
  CK(pl->gm_zero.need(sizeof(double)));
  CK(pl->gm_one.need(sizeof(double)));
  CK(cudaMemcpyAsync(pl->gm_zero.p, &z, sizeof(double), cudaMemcpyHostToDevice, pl->stream));
  CK(cudaMemcpyAsync(pl->gm_one.p, &o, sizeof(double), cudaMemcpyHostToDevice, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_rotate_full_batch(pp_plan_t* pl, const float* in, float* outp, int32_t nsub, const double* phase,
                                    const double* DM, const double* GM, const double* P, const double* nu_ref,
                                    const double* nu_GM) {
  if (!pl || !in || !outp || !phase || !DM || !P || !nu_ref) return fail(-1, "NULL argument");
  if ((GM == nullptr) != (nu_GM == nullptr)) return fail(-1, "GM and nu_GM must be given together");
  if (nsub < 1) return fail(-1, "nsub must be >= 1");
  if (!pl->freqs_set) return fail(-1, "pp_set_model or pp_set_freqs must be called before pp_rotate_batch");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int nchan = pl->nchan;
  const size_t tot = (size_t)nsub * nchan * pl->nbin;
  const float* din;
  if (stage_in(pl, pl->rot_in, in, tot, &din)) return -2;
  float* dout;
  if (stage_out(pl->rot_out, outp, tot, &dout)) return -2;
  const double *dph, *ddm, *dP, *dnr, *dgm, *dng;
  if (stage_in(pl, pl->rot_phase, phase, (size_t)nsub, &dph)) return -2;
  if (stage_in(pl, pl->rot_dm, DM, (size_t)nsub, &ddm)) return -2;
  if (stage_in(pl, pl->rot_P, P, (size_t)nsub, &dP)) return -2;
  if (stage_in(pl, pl->rot_nuref, nu_ref, (size_t)nsub, &dnr)) return -2;
  if (stage_in(pl, pl->rot_gm, GM, (size_t)nsub, &dgm)) return -2;
  if (stage_in(pl, pl->rot_nugm, nu_GM, (size_t)nsub, &dng)) return -2;
  RotateArgs a;
  a.in = din; a.out = dout; a.phase = dph; a.DM = ddm; a.P = dP; a.nu_ref = dnr; a.GM = dgm; a.nu_GM = dng;
  a.nu2 = pl->nu2.as<double>(); a.taus = nullptr; a.resp = nullptr; a.nsub = nsub; a.nchan = nchan;
  if (rotate_rows(pl, a, pl->fft_precision == 64)) return -2;
  CK(cudaGetLastError());
  if (finish_out(pl, outp, dout, tot)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_rotate_batch(pp_plan_t* pl, const float* in, float* outp, int32_t nsub, const double* phase, const double* DM,
                               const double* P, const double* nu_ref) {
  return pp_rotate_full_batch(pl, in, outp, nsub, phase, DM, nullptr, P, nu_ref, nullptr);
}

extern "C" int pp_apply_response_batch(pp_plan_t* pl, const float* in, float* outp, int32_t nsub, const double* resp) {
  if (!pl || !in || !outp || !resp) return fail(-1, "NULL argument");
  if (nsub < 1) return fail(-1, "nsub must be >= 1");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int nchan = pl->nchan;
  const size_t tot = (size_t)nsub * nchan * pl->nbin;
  const float* din;
  if (stage_in(pl, pl->rot_in, in, tot, &din)) return -2;
  float* dout;
  if (stage_out(pl->rot_out, outp, tot, &dout)) return -2;
  const double* dresp;
  if (stage_in(pl, pl->resp, resp, (size_t)nchan * (pl->nbin / 2 + 1), &dresp)) return -2;
  if (unit_scalars(pl)) return -2;
  // zero rotation for every subint: phase, DM from a zero-filled array
  CK(pl->rot_phase.need(sizeof(double) * nsub));
  CK(pl->rot_P.need(sizeof(double) * nsub));
  CK(cudaMemsetAsync(pl->rot_phase.p, 0, sizeof(double) * nsub, pl->stream));
  {
    std::vector<double> ones((size_t)nsub, 1.0);
    CK(cudaMemcpyAsync(pl->rot_P.p, ones.data(), sizeof(double) * nsub, cudaMemcpyHostToDevice, pl->stream));
    CK(cudaStreamSynchronize(pl->stream));
  }
  RotateArgs a;
  a.in = din; a.out = dout; a.phase = pl->rot_phase.as<double>(); a.DM = pl->rot_phase.as<double>();
  a.P = pl->rot_P.as<double>(); a.nu_ref = pl->rot_P.as<double>(); a.GM = nullptr; a.nu_GM = nullptr;
  a.nu2 = pl->nu2.as<double>(); a.taus = nullptr; a.resp = dresp; a.nsub = nsub; a.nchan = nchan;
  if (!pl->nu2.p) { CK(pl->nu2.need(sizeof(double) * nchan)); CK(cudaMemsetAsync(pl->nu2.p, 0, sizeof(double) * nchan, pl->stream)); a.nu2 = pl->nu2.as<double>(); }
  if (rotate_rows(pl, a, true)) return -2;
  CK(cudaGetLastError());
  if (finish_out(pl, outp, dout, tot)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_align_accumulate(pp_plan_t* pl, const float* data, int32_t nsub, const double* phase, const double* DM,
                                   const double* P, const double* nu_ref, const double* weights, double* aligned,
                                   double* wsum) {
  if (!pl || !data || !phase || !DM || !P || !nu_ref || !weights || !aligned || !wsum) return fail(-1, "NULL argument");
  if (nsub < 1) return fail(-1, "nsub must be >= 1");
  if (!pl->freqs_set) return fail(-1, "pp_set_model or pp_set_freqs must be called first");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int N = pl->N, nchan = pl->nchan;
  const float* din;
  if (stage_in(pl, pl->rot_in, data, (size_t)nsub * nchan * pl->nbin, &din)) return -2;
  const double *dph, *ddm, *dP, *dnr, *dw;
  if (stage_in(pl, pl->rot_phase, phase, (size_t)nsub, &dph)) return -2;
  if (stage_in(pl, pl->rot_dm, DM, (size_t)nsub, &ddm)) return -2;
  if (stage_in(pl, pl->rot_P, P, (size_t)nsub, &dP)) return -2;
  if (stage_in(pl, pl->rot_nuref, nu_ref, (size_t)nsub, &dnr)) return -2;
  if (stage_in(pl, pl->al_w, weights, (size_t)nsub * nchan, &dw)) return -2;
  CK(pl->al_out.need(sizeof(double) * (size_t)nchan * pl->nbin));
  CK(pl->al_wsum.need(sizeof(double) * nchan));
  if (pl->anyn) {   // rotate blocks of subints in the Fourier domain, add their spectra up in double, transform once
    const int blk = 64;
    CK(pl->al_acc.need(sizeof(double2) * (size_t)nchan * N));
    CK(pl->al_dc.need(sizeof(double) * nchan));
    for (int s0 = 0; s0 < nsub; s0 += blk) {
      const int ns = std::min(blk, nsub - s0);
      RotateArgs r;
      r.in = din + (size_t)s0 * nchan * pl->nbin; r.out = nullptr; r.phase = dph + s0; r.DM = ddm + s0;
      r.P = dP + s0; r.nu_ref = dnr + s0; r.GM = nullptr; r.nu_GM = nullptr; r.nu2 = pl->nu2.as<double>(); r.taus = nullptr;
      r.resp = nullptr; r.nsub = ns; r.nchan = nchan;
      if (rotate_spectra_any(pl, r)) return -2;
      k_wsum_spec<<<nchan, 256, 0, pl->stream>>>(pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>(), dw + (size_t)s0 * nchan,
                                                 pl->al_acc.as<cx<double>>(), pl->al_dc.as<double>(), pl->al_wsum.as<double>(),
                                                 ns, nchan, N, s0 == 0);
      pl->stats.launches++;
    }
    if (launch_inv_any(pl, pl->al_acc.as<cx<double>>(), pl->al_dc.as<double>(), pl->al_out.as<double>(), nchan, true)) return -2;
  } else {
    AlignArgs a;
    a.r.in = din; a.r.out = nullptr; a.r.phase = dph; a.r.DM = ddm; a.r.P = dP; a.r.nu_ref = dnr; a.r.GM = nullptr;
    a.r.nu_GM = nullptr; a.r.taus = nullptr; a.r.resp = nullptr; a.r.nu2 = pl->nu2.as<double>(); a.r.twN = pl->twN64.p; a.r.tw2N = pl->tw2N64.p;
    a.r.nsub = nsub; a.r.nchan = nchan;
    a.weights = dw; a.aligned = pl->al_out.as<double>(); a.wsum = pl->al_wsum.as<double>();
    DISPATCH_N(N, (k_align_accum<NN><<<row_ctas<NN>(nchan), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(a)));
    pl->stats.launches++;
  }
  CK(cudaGetLastError());
  if (copy_out_at(pl->stream, aligned, pl->al_out.as<double>(), 0, (size_t)nchan * pl->nbin)) return -2;
  if (copy_out_at(pl->stream, wsum, pl->al_wsum.as<double>(), 0, (size_t)nchan)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

static int gen_gaussian_impl(pp_plan* pl, const char* model_code, const double* params, int32_t ngauss,
                             double scattering_index, double nu_ref, float* outp, double* outp64) {
  if (!pl || !model_code || !params || !(outp || outp64)) return fail(-1, "NULL argument");
  if (ngauss < 0 || ngauss > kMaxGauss) return fail(-1, "ngauss must be in [0, %d]", kMaxGauss);
  if (strlen(model_code) < 3) return fail(-1, "model_code needs three characters (loc, wid, amp)");
  for (int i = 0; i < 3; ++i)
    if (model_code[i] != '0' && model_code[i] != '1') return fail(-1, "model_code digit %d must be '0' or '1'", i);
  if (!(nu_ref > 0.0)) return fail(-1, "nu_ref must be positive");
  if (!pl->freqs_set) return fail(-1, "pp_set_freqs must be called before pp_gen_gaussian_portrait");
  if (is_device_ptr(params)) return fail(-1, "params must be a host array");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int nchan = pl->nchan;
  const size_t np = 2 + 6 * (size_t)ngauss, tot = (size_t)nchan * pl->nbin;
  CK(pl->gm_params.need(sizeof(double) * np));
  CK(pl->gm_taus.need(sizeof(double) * nchan));
  CK(cudaMemcpyAsync(pl->gm_params.p, params, sizeof(double) * np, cudaMemcpyHostToDevice, pl->stream));
  const bool scat = params[1] != 0.0;          // the scattering multiply works on float32 rows
  const bool want64 = outp64 != nullptr;
  float* dout = nullptr;
  double* dout64 = nullptr;
  if (want64) {
    if (stage_out(pl->model_stage64, outp64, tot, &dout64)) return -2;
    if (scat) { CK(pl->rot_out.need(sizeof(float) * tot)); dout = pl->rot_out.as<float>(); }
  } else if (stage_out(pl->rot_out, outp, tot, &dout)) return -2;
  GaussModelArgs g;
  g.params = pl->gm_params.as<double>(); g.freqs = pl->freqs.as<double>(); g.taus = pl->gm_taus.as<double>();
  g.out = dout; g.out64 = (want64 && !scat) ? dout64 : nullptr;
  g.nu_ref = nu_ref; g.alpha = scattering_index; g.ngauss = ngauss; g.nchan = nchan; g.nbin = pl->nbin;
  g.code_loc = model_code[0] - '0'; g.code_wid = model_code[1] - '0'; g.code_amp = model_code[2] - '0';
  k_gauss_model<<<nchan, 256, 0, pl->stream>>>(g);
  pl->stats.launches++;
  if (scat) {   // scattering: rfft, times 1/(1 + 2 pi i k tau_n), irfft (pplib.py:921-927), in place
    if (unit_scalars(pl)) return -2;
    RotateArgs a;
    a.in = dout; a.out = dout; a.phase = pl->gm_zero.as<double>(); a.DM = pl->gm_zero.as<double>();
    a.P = pl->gm_one.as<double>(); a.nu_ref = pl->gm_one.as<double>(); a.GM = nullptr; a.nu_GM = nullptr;
    a.nu2 = pl->nu2.as<double>(); a.taus = pl->gm_taus.as<double>(); a.resp = nullptr; a.nsub = 1; a.nchan = nchan;
    if (rotate_rows(pl, a, true)) return -2;
    if (want64) {
      k_cvt_f32_f64<<<(unsigned)std::min<size_t>((tot + 255) / 256, 148 * 32), 256, 0, pl->stream>>>(dout, dout64, tot);
      pl->stats.launches++;
    }
  }
  CK(cudaGetLastError());
  if (want64 ? finish_out(pl, outp64, dout64, tot) : finish_out(pl, outp, dout, tot)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_gen_gaussian_portrait(pp_plan_t* pl, const char* model_code, const double* params, int32_t ngauss,
                                        double scattering_index, double nu_ref, float* outp) {
  return gen_gaussian_impl(pl, model_code, params, ngauss, scattering_index, nu_ref, outp, nullptr);
}

extern "C" int pp_gen_gaussian_portrait_f64(pp_plan_t* pl, const char* model_code, const double* params, int32_t ngauss,
                                            double scattering_index, double nu_ref, double* outp) {
  return gen_gaussian_impl(pl, model_code, params, ngauss, scattering_index, nu_ref, nullptr, outp);
}

extern "C" int pp_gen_spline_portrait(pp_plan_t* pl, const double* mean_prof, const double* eigvec, int32_t ncomp,
                                      const double* knots, int32_t nknots, const double* coefs, int32_t degree,
                                      float* outp) {
  if (!pl || !mean_prof || !outp) return fail(-1, "NULL argument");
  if (ncomp < 0 || ncomp > kMaxSplineComp) return fail(-1, "ncomp must be in [0, %d]", kMaxSplineComp);
  if (ncomp > 0) {
    if (!eigvec || !knots || !coefs) return fail(-1, "NULL spline argument");
    if (degree < 1 || degree > 5) return fail(-1, "spline degree must be in [1, 5]");
    if (nknots < 2 * (degree + 1)) return fail(-1, "need at least 2 (degree + 1) knots");
  }
  if (!pl->freqs_set) return fail(-1, "pp_set_freqs must be called before pp_gen_spline_portrait");
  if (is_device_ptr(mean_prof) || (ncomp > 0 && (is_device_ptr(eigvec) || is_device_ptr(knots) || is_device_ptr(coefs))))
    return fail(-1, "the spline model arrays must be host arrays");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int nchan = pl->nchan, nbin = pl->nbin;
  const int ncoef = ncomp > 0 ? nknots - degree - 1 : 0;
  const size_t n_mean = nbin, n_eig = (size_t)nbin * ncomp, n_kn = ncomp > 0 ? nknots : 0, n_co = (size_t)ncomp * ncoef;
  const size_t total = n_mean + n_eig + n_kn + n_co;
  CK(pl->gm_params.need(sizeof(double) * total));
  double* base = pl->gm_params.as<double>();
  CK(cudaMemcpyAsync(base, mean_prof, sizeof(double) * n_mean, cudaMemcpyHostToDevice, pl->stream));
  if (ncomp > 0) {
    CK(cudaMemcpyAsync(base + n_mean, eigvec, sizeof(double) * n_eig, cudaMemcpyHostToDevice, pl->stream));
    CK(cudaMemcpyAsync(base + n_mean + n_eig, knots, sizeof(double) * n_kn, cudaMemcpyHostToDevice, pl->stream));
    CK(cudaMemcpyAsync(base + n_mean + n_eig + n_kn, coefs, sizeof(double) * n_co, cudaMemcpyHostToDevice, pl->stream));
  }
  const size_t tot = (size_t)nchan * nbin;
  float* dout;
  if (stage_out(pl->rot_out, outp, tot, &dout)) return -2;
  SplineModelArgs g;
  g.mean_prof = base; g.eigvec = base + n_mean; g.knots = base + n_mean + n_eig; g.coefs = base + n_mean + n_eig + n_kn;
  g.freqs = pl->freqs.as<double>(); g.out = dout; g.ncomp = ncomp; g.nknots = nknots; g.degree = degree;
  g.nchan = nchan; g.nbin = nbin;
  k_spline_model<<<nchan, 256, 0, pl->stream>>>(g);
  pl->stats.launches++;
  CK(cudaGetLastError());
  if (finish_out(pl, outp, dout, tot)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_get_noise_fit_batch(pp_plan_t* pl, const float* data, int32_t nsub, double fact, double* noise_out) {
  if (!pl || !data || !noise_out) return fail(-1, "NULL argument");
  if (nsub < 1) return fail(-1, "nsub must be >= 1");
  if (!(fact > 0.0)) return fail(-1, "fact must be positive");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int N = pl->N, nchan = pl->nchan, L = pl->nbin / 2;
  const long nrows = (long)nsub * nchan;
  const float* din;
  if (stage_in(pl, pl->rot_in, data, (size_t)nrows * pl->nbin, &din)) return -2;
  CK(pl->ps_noise.need(sizeof(double) * nrows));
  CK(pl->any_spec2.need(sizeof(double2) * (size_t)nrows * N));
  CK(pl->any_dc2.need(sizeof(double) * (size_t)nrows));
  if (pl->anyn) {
    if (launch_fwd_any(pl, din, false, nullptr, nullptr, nrows, pl->any_spec2.as<cx<double>>(), pl->any_dc2.as<double>())) return -2;
  } else {
    if (launch_rfft_rows(pl, din, (int)nrows, nullptr, 0, nullptr, 64, -1, pl->any_spec2.as<double2>(), pl->any_dc2.as<double>())) return -2;
  }
  const size_t smem = sizeof(double) * 3 * (size_t)(L + 1);
  CK(cudaFuncSetAttribute(k_noise_fit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_noise_fit<<<(unsigned)nrows, 256, smem, pl->stream>>>(pl->any_spec2.as<double2>(), pl->any_dc2.as<double>(), pl->ps_noise.as<double>(),
                                                          N, L, pl->anyn ? L : 0, fact);
  pl->stats.launches++;
  CK(cudaGetLastError());
  if (copy_out_at(pl->stream, noise_out, pl->ps_noise.as<double>(), 0, (size_t)nrows)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_measure_fp64(pp_plan_t* pl, double* dfma_per_second) {
  if (!pl || !dfma_per_second) return fail(-1, "NULL argument");
  CK(cudaSetDevice(pl->device));
  const int ctas = pl->sm_count * 4, iters = 2048;
  CK(pl->ps_noise.need(sizeof(double) * (size_t)ctas * 256));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {
    CK(cudaEventRecord(e0, pl->stream));
    k_fp64_peak<<<ctas, 256, 0, pl->stream>>>(pl->ps_noise.as<double>(), iters, 1.0000001, 1e-9);
    CK(cudaEventRecord(e1, pl->stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  CK(cudaGetLastError());
  *dfma_per_second = (double)ctas * 256.0 * (double)iters * 64.0 / ((double)best * 1e-3);
  return 0;
}

extern "C" int pp_get_noise_batch(pp_plan_t* pl, const float* data, int32_t nsub, double* noise_out) {
  return pp_get_noise_cut_batch(pl, data, nsub, -1, noise_out);
}

extern "C" int pp_get_noise_cut_batch(pp_plan_t* pl, const float* data, int32_t nsub, int32_t kc, double* noise_out) {
  if (!pl || !data || !noise_out) return fail(-1, "NULL argument");
  if (nsub < 1) return fail(-1, "nsub must be >= 1");
  if (kc > pl->nbin / 2) return fail(-1, "kc must be <= nbin/2 (got %d)", kc);
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const long nrows = (long)nsub * pl->nchan;
  const float* din;
  if (stage_in(pl, pl->rot_in, data, (size_t)nrows * pl->nbin, &din)) return -2;
  CK(pl->ps_noise.need(sizeof(double) * nrows));
  const int bits = pl->fft_precision ? pl->fft_precision : 64;
  if (launch_rfft_rows(pl, din, (int)nrows, nullptr, 0, pl->ps_noise.as<double>(), bits, kc)) return -2;
  CK(cudaGetLastError());
  if (copy_out_at(pl->stream, noise_out, pl->ps_noise.as<double>(), 0, (size_t)nrows)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

// ----------------------------------------------------------------------------
// evolving-Gaussian portrait fit (gaussfit.cuh)
// ----------------------------------------------------------------------------
// Device scratch of one call: the per-CTA slabs, nslab x (L + 1) x (nbin/2 + 1) x 16 bytes with nslab =
// (resident CTAs of k_gfit_pass), and per chunk of portraits the channel records (nchan x S doubles),
// the staged data, the state and the outputs (~ 3 P^2 + nchan nbin doubles) of each portrait.  The
// chunk is sized so that this per-chunk part stays under kGfitChunkBytes (at least one portrait, at most
// 65535), or is pp_plan_set_chunk's count: the scratch does not grow with nport.
static const size_t kGfitChunkBytes = 256u << 20;

template <int N> static int gfit_slabs(pp_plan* pl, int* nslab) {
  const size_t smem = fft_smem_bytes<N, double>();
  CK(cudaFuncSetAttribute(k_gfit_pass<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gfit_pass<N>, 256, smem));
  *nslab = std::max(1, per_sm) * pl->sm_count;
  return 0;
}

template <int N> static int gfit_pass(pp_plan* pl, const GfitArgs& a, int nslab) {
  const long units = (long)a.nc * a.nchan;
  const unsigned grid = (unsigned)std::min<long>(units, nslab);
  k_gfit_pass<N><<<grid, 256, fft_smem_bytes<N, double>(), pl->stream>>>(a);
  pl->stats.launches++;
  pl->stats.pass_launches++;
  CK(cudaGetLastError());
  return 0;
}

extern "C" int pp_fit_gaussian_portraits(pp_plan_t* pl, const pp_gfit_args_t* args, const pp_gfit_out_t* out) {
  if (!pl || !args || !out) return fail(-1, "NULL argument");
  const pp_gfit_args_t& A = *args;
  if (A.nport < 1) return fail(-1, "nport must be >= 1");
  if (!A.data || !A.errs || !A.init || !A.model_code || !A.fit_flags) return fail(-1, "NULL input array");
  if (A.ngauss < 1 || A.ngauss > kGfitMaxGauss) return fail(-1, "ngauss must be in [1, %d] (got %d)", kGfitMaxGauss, A.ngauss);
  if (strlen(A.model_code) < 3) return fail(-1, "model_code needs three characters (loc, wid, amp)");
  for (int i = 0; i < 3; ++i)
    if (A.model_code[i] != '0' && A.model_code[i] != '1') return fail(-1, "model_code digit %d must be '0' or '1'", i);
  if (!(A.nu_ref > 0.0)) return fail(-1, "nu_ref must be positive");
  if (pl->anyn) return fail(-1, "the Gaussian portrait fit needs nbin a power of two in [64, 4096] (got %d)", pl->nbin);
  if (!pl->freqs_set) return fail(-1, "pp_set_freqs must be called before pp_fit_gaussian_portraits");
  if (is_device_ptr(A.fit_flags) || (A.bounds && is_device_ptr(A.bounds))) return fail(-1, "fit_flags and bounds must be host arrays");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int N = pl->N, nbin = pl->nbin, nchan = pl->nchan, ng = A.ngauss;
  const int P = 3 + 6 * ng, L = 2 + 3 * ng, S = (L + 1) * (L + 2) / 2 + P;
  const int nport = A.nport;
  // host checks of sigma (a device array is read back once)
  {
    std::vector<double> e((size_t)nport * nchan);
    CK(cudaMemcpy(e.data(), A.errs, sizeof(double) * e.size(), cudaMemcpyDefault));
    for (size_t i = 0; i < e.size(); ++i)
      if (!(e[i] > 0.0) || !std::isfinite(e[i]))
        return fail(-1, "errs must be positive and finite (portrait %d, channel %d: %g)", (int)(i / nchan), (int)(i % nchan), e[i]);
  }
  std::vector<uint8_t> fr(P);
  std::vector<double> lo(P, -INFINITY), hi(P, INFINITY);
  int nfree = 0;
  for (int i = 0; i < P; ++i) { fr[i] = A.fit_flags[i] ? 1 : 0; nfree += fr[i]; }
  if (A.bounds)
    for (int i = 0; i < P; ++i) {
      if (!std::isnan(A.bounds[2 * i])) lo[i] = A.bounds[2 * i];
      if (!std::isnan(A.bounds[2 * i + 1])) hi[i] = A.bounds[2 * i + 1];
      if (lo[i] > hi[i]) return fail(-1, "bounds of parameter %d: lower > upper", i);
    }
  const int max_iter = A.max_iter == 0 ? 200 : A.max_iter;
  const double tol = A.tol > 0.0 ? A.tol : 1e-4;
  // chunk of portraits
  const size_t per_port = sizeof(double) * ((size_t)nchan * S + (size_t)nchan * nbin * (out->model ? 2 : 1) + 4 * (size_t)P * P + 8 * P + 16);
  size_t want = pl->chunk_req > 0 ? (size_t)pl->chunk_req : std::max<size_t>(1, kGfitChunkBytes / per_port);
  // the chunk's portraits are gridDim.y of k_gfit_reduce (<= 65535)
  const int chunk = (int)std::min<size_t>(std::min<size_t>(want, 65535), (size_t)nport);
  int nslab = 0;
  DISPATCH_N(N, if (gfit_slabs<NN>(pl, &nslab)) return -2);
  nslab = (int)std::min<long>(nslab, (long)chunk * nchan);
  CK(pl->gf_slab.need(sizeof(double2) * (size_t)nslab * (L + 1) * (N + 1)));
  CK(pl->gf_rec.need(sizeof(double) * (size_t)chunk * nchan * S));
  CK(pl->gf_data.need(sizeof(double) * (size_t)chunk * nchan * nbin));
  CK(pl->gf_errs.need(sizeof(double) * (size_t)chunk * nchan));
  if (out->model) CK(pl->gf_model.need(sizeof(double) * (size_t)chunk * nchan * nbin));
  // parameter tables: free flags (as bytes after lo, hi)
  CK(pl->gf_par.need(sizeof(double) * 2 * P + P));
  {
    std::vector<unsigned char> h(sizeof(double) * 2 * P + P);
    memcpy(h.data(), lo.data(), sizeof(double) * P);
    memcpy(h.data() + sizeof(double) * P, hi.data(), sizeof(double) * P);
    memcpy(h.data() + sizeof(double) * 2 * P, fr.data(), P);
    CK(cudaMemcpyAsync(pl->gf_par.p, h.data(), h.size(), cudaMemcpyHostToDevice, pl->stream));
    CK(cudaStreamSynchronize(pl->stream));
  }
  const double* d_lo = pl->gf_par.as<double>();
  const double* d_hi = d_lo + P;
  const uint8_t* d_free = reinterpret_cast<const uint8_t*>(d_lo + 2 * P);
  // chunk state
  const size_t PP = (size_t)P * P;
  const size_t n_state = (size_t)chunk * (4 * P + 2 * PP + 3);
  CK(pl->gf_state.need(sizeof(double) * n_state + sizeof(int) * (2 * (size_t)chunk + 1)));
  GfitState st;
  {
    double* b = pl->gf_state.as<double>();
    st.x = b; b += (size_t)chunk * P;
    st.xt = b; b += (size_t)chunk * P;
    st.jtj_t = b; b += chunk * PP;
    st.jtj = b; b += chunk * PP;
    st.jtr_t = b; b += (size_t)chunk * P;
    st.jtr = b; b += (size_t)chunk * P;
    st.chi2_t = b; b += chunk;
    st.chi2 = b; b += chunk;
    st.lam = b; b += chunk;
    int* ib = reinterpret_cast<int*>(b);
    st.nfev = ib; ib += chunk;
    st.done = ib; ib += chunk;
  }
  int* d_running = reinterpret_cast<int*>(st.done + chunk);
  // chunk outputs: params, errs, cov, chi2, red_chi2, jtr, jtj (doubles), nfeval, rc (ints)
  const size_t n_out = (size_t)chunk * (2 * P + 2 * PP + 2 + P);
  CK(pl->gf_out.need(sizeof(double) * n_out + sizeof(int) * 2 * (size_t)chunk));
  GfitUpdateArgs u;
  {
    double* b = pl->gf_out.as<double>();
    u.params = b; b += (size_t)chunk * P;
    u.errs = b; b += (size_t)chunk * P;
    u.cov = b; b += chunk * PP;
    u.jtj = b; b += chunk * PP;
    u.jtr = b; b += (size_t)chunk * P;
    u.chi2 = b; b += chunk;
    u.red_chi2 = b; b += chunk;
    u.nfeval = reinterpret_cast<int*>(b);
    u.rc = u.nfeval + chunk;
  }
  u.free_ = d_free; u.lo = d_lo; u.hi = d_hi; u.P = P; u.max_iter = max_iter; u.tol = tol;
  u.ndata = (double)nchan * (double)nbin; u.running = d_running;
  const size_t usmem = sizeof(double) * 2 * PP;
  CK(cudaFuncSetAttribute(k_gfit_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)usmem));
  GfitArgs g;
  g.freqs = pl->freqs.as<double>(); g.rec = pl->gf_rec.as<double>(); g.slab = pl->gf_slab.as<double2>();
  g.twN = pl->twN64.p; g.tw2N = pl->tw2N64.p; g.nu_ref = A.nu_ref; g.nchan = nchan; g.ngauss = ng;
  g.P = P; g.L = L; g.S = S;
  for (int i = 0; i < 3; ++i) g.code[i] = A.model_code[i] - '0';
  const int npair_all = P * (P + 1) / 2 + P + 1;
  std::vector<double> x0((size_t)chunk * P);
  for (int s0 = 0; s0 < nport; s0 += chunk) {
    const int nc = std::min(chunk, nport - s0);
    const size_t rows = (size_t)nc * nchan;
    CK(cudaMemcpyAsync(pl->gf_data.p, A.data + (size_t)s0 * nchan * nbin, sizeof(double) * rows * nbin,
                       cudaMemcpyDefault, pl->stream));
    CK(cudaMemcpyAsync(pl->gf_errs.p, A.errs + (size_t)s0 * nchan, sizeof(double) * rows, cudaMemcpyDefault, pl->stream));
    // start values moved into the box
    CK(cudaMemcpyAsync(x0.data(), A.init + (size_t)s0 * P, sizeof(double) * nc * P, cudaMemcpyDefault, pl->stream));
    CK(cudaStreamSynchronize(pl->stream));
    for (int s = 0; s < nc; ++s)
      for (int i = 0; i < P; ++i) x0[(size_t)s * P + i] = std::min(std::max(x0[(size_t)s * P + i], lo[i]), hi[i]);
    CK(cudaMemcpyAsync(st.xt, x0.data(), sizeof(double) * nc * P, cudaMemcpyHostToDevice, pl->stream));
    {
      std::vector<double> lam(nc, kGfitLam0);
      CK(cudaMemcpyAsync(st.lam, lam.data(), sizeof(double) * nc, cudaMemcpyHostToDevice, pl->stream));
      CK(cudaMemsetAsync(st.nfev, 0, sizeof(int) * 2 * chunk, pl->stream));   // nfev and done
      CK(cudaStreamSynchronize(pl->stream));
    }
    g.data = pl->gf_data.as<double>(); g.errs = pl->gf_errs.as<double>(); g.nc = nc;
    // passes are launched while some portrait of the chunk is still running
    for (;;) {
      g.xt = st.xt; g.done = st.done; g.model = nullptr;
      DISPATCH_N(N, if (gfit_pass<NN>(pl, g, nslab)) return -2);
      k_gfit_reduce<<<dim3((npair_all + 255) / 256, nc), 256, 0, pl->stream>>>(g, st, d_free);
      CK(cudaMemsetAsync(d_running, 0, sizeof(int), pl->stream));
      k_gfit_update<<<nc, 256, usmem, pl->stream>>>(st, u);
      pl->stats.launches += 2;
      CK(cudaGetLastError());
      int running = 0;
      CK(cudaMemcpyAsync(&running, d_running, sizeof(int), cudaMemcpyDeviceToHost, pl->stream));
      CK(cudaStreamSynchronize(pl->stream));
      if (running == 0) break;
    }
    if (out->model) {   // the fitted portraits, evaluated at the final point of each
      g.xt = st.x; g.done = nullptr; g.model = pl->gf_model.as<double>();
      DISPATCH_N(N, if (gfit_pass<NN>(pl, g, nslab)) return -2);
      if (copy_out_at(pl->stream, out->model + (size_t)s0 * nchan * nbin, pl->gf_model.as<double>(), 0, rows * nbin)) return -2;
    }
    const cudaStream_t sm = pl->stream;
    if (copy_out_at(sm, out->params + (out->params ? (size_t)s0 * P : 0), u.params, 0, (size_t)nc * P)) return -2;
    if (copy_out_at(sm, out->param_errs + (out->param_errs ? (size_t)s0 * P : 0), u.errs, 0, (size_t)nc * P)) return -2;
    if (copy_out_at(sm, out->cov + (out->cov ? (size_t)s0 * PP : 0), u.cov, 0, (size_t)nc * PP)) return -2;
    if (copy_out_at(sm, out->jtj + (out->jtj ? (size_t)s0 * PP : 0), u.jtj, 0, (size_t)nc * PP)) return -2;
    if (copy_out_at(sm, out->jtr + (out->jtr ? (size_t)s0 * P : 0), u.jtr, 0, (size_t)nc * P)) return -2;
    if (copy_out_at(sm, out->chi2 + (out->chi2 ? s0 : 0), u.chi2, 0, (size_t)nc)) return -2;
    if (copy_out_at(sm, out->red_chi2 + (out->red_chi2 ? s0 : 0), u.red_chi2, 0, (size_t)nc)) return -2;
    if (copy_out_at(sm, out->nfeval + (out->nfeval ? s0 : 0), u.nfeval, 0, (size_t)nc)) return -2;
    if (copy_out_at(sm, out->return_code + (out->return_code ? s0 : 0), u.rc, 0, (size_t)nc)) return -2;
    CK(cudaStreamSynchronize(pl->stream));
  }
  CK(cudaGetLastError());
  return 0;
}

// ----------------------------------------------------------------------------
// simulated archives (kernels.cuh k_simulate / k_sim_mul / k_sim_store)
// ----------------------------------------------------------------------------
// a page-locked piece of the plan's ring for a device -> host copy (the copy that last used it has finished)
static int pin_piece(pp_plan* pl, void** buf) {
  const int slot = (int)(pl->pin_count++ % pp_plan::kPinSlots);
  if (!pl->pin_ring[slot]) {
    CK(cudaHostAlloc(&pl->pin_ring[slot], pp_plan::kPinPiece, cudaHostAllocDefault));
    CK(cudaEventCreateWithFlags(&pl->pin_ev[slot], cudaEventDisableTiming));
  } else {
    CK(cudaEventSynchronize(pl->pin_ev[slot]));
  }
  *buf = pl->pin_ring[slot];
  return 0;
}

// index of the first of n values (host or device) for which bad(v) holds, or n; device values are read back
// in pieces through the page-locked ring
template <typename T, typename Bad> static int find_bad(pp_plan* pl, const T* p, size_t n, Bad bad, size_t* at) {
  *at = n;
  if (!is_device_ptr(p)) {
    for (size_t i = 0; i < n; ++i) if (bad(p[i])) { *at = i; return 0; }
    return 0;
  }
  const size_t per = pp_plan::kPinPiece / sizeof(T);
  for (size_t off = 0; off < n; off += per) {
    const size_t len = std::min(per, n - off);
    void* buf;
    if (pin_piece(pl, &buf)) return -2;
    CK(cudaMemcpyAsync(buf, p + off, len * sizeof(T), cudaMemcpyDeviceToHost, pl->stream));
    CK(cudaStreamSynchronize(pl->stream));
    const T* h = static_cast<const T*>(buf);
    for (size_t i = 0; i < len; ++i) if (bad(h[i])) { *at = off + i; return 0; }
  }
  return 0;
}

// device -> caller's host memory through the plan's page-locked ring (page-locked destinations directly)
static int d2h_staged(pp_plan* pl, void* dst, const void* src, size_t bytes) {
  if (mem_kind(dst) == kMemPinned) {
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, pl->stream));
    return 0;
  }
  static const int nthreads = std::max(1, std::min(8, (int)std::thread::hardware_concurrency() / 2));
  for (size_t off = 0; off < bytes; off += pp_plan::kPinPiece) {
    const size_t len = std::min(pp_plan::kPinPiece, bytes - off);
    void* buf;
    if (pin_piece(pl, &buf)) return -2;
    CK(cudaMemcpyAsync(buf, (const char*)src + off, len, cudaMemcpyDeviceToHost, pl->stream));
    CK(cudaStreamSynchronize(pl->stream));
    parallel_memcpy((char*)dst + off, buf, len, nthreads);
  }
  return 0;
}

// elements [off, off + n) of an input for one chunk: a device array in place, a host one copied into buf
template <typename T> static int chunk_in(pp_plan* pl, DBuf& buf, const T* src, bool dev, size_t off, size_t n, const T** out) {
  if (!src) { *out = nullptr; return 0; }
  if (dev) { *out = src + off; return 0; }
  CK(buf.need(sizeof(T) * n));
  CK(cudaMemcpyAsync(buf.p, src + off, sizeof(T) * n, cudaMemcpyHostToDevice, pl->stream));
  *out = buf.as<T>();
  return 0;
}

static const size_t kSimChunkBytes = 256u << 20;   // device scratch of one chunk of a simulate call

extern "C" int pp_simulate_batch(pp_plan_t* pl, const pp_sim_args_t* args, const pp_sim_out_t* out) {
  if (!pl || !args || !out) return fail(-1, "NULL argument");
  const pp_sim_args_t& A = *args;
  if (A.nsub < 0) return fail(-1, "nsub must be >= 0 (got %d)", A.nsub);
  if (A.nsub == 0) return 0;
  if (A.nmodel < 1) return fail(-1, "nmodel must be >= 1 (got %d)", A.nmodel);
  if (!A.models || !A.freqs || !A.phase || !A.DM || !A.P || !A.nu_DM) return fail(-1, "NULL input array");
  if ((A.GM == nullptr) != (A.nu_GM == nullptr)) return fail(-1, "GM and nu_GM must be given together");
  if (!((A.tau && A.alpha && A.nu_tau) || (!A.tau && !A.alpha && !A.nu_tau)))
    return fail(-1, "tau, alpha and nu_tau must be given together");
  if (!out->data && !out->raw) return fail(-1, "no output: data or raw must be given");
  if (out->raw && (!out->dat_scl || !out->dat_offs)) return fail(-1, "raw output needs dat_scl and dat_offs");
  CK(cudaSetDevice(pl->device));
  const int nsub = A.nsub, nchan = pl->nchan, nbin = pl->nbin, nmodel = A.nmodel;
  const size_t nsc = (size_t)nsub * nchan, nfreq = (size_t)nmodel * nchan;
  // ---- validation (device inputs are read back in pieces): nothing runs before it passes
  std::vector<double> hf(nfreq), hn2(nfreq);
  if (is_device_ptr(A.freqs)) CK(cudaMemcpy(hf.data(), A.freqs, sizeof(double) * nfreq, cudaMemcpyDeviceToHost));
  else memcpy(hf.data(), A.freqs, sizeof(double) * nfreq);
  for (size_t i = 0; i < nfreq; ++i) {
    if (!(hf[i] > 0.0)) return fail(-1, "freqs[%d, %d] = %g is not positive", (int)(i / nchan), (int)(i % nchan), hf[i]);
    hn2[i] = 1.0 / (hf[i] * hf[i]);
  }
  size_t at;
  if (A.model_index) {
    if (find_bad(pl, A.model_index, (size_t)nsub, [nmodel](int32_t v) { return v < 0 || v >= nmodel; }, &at)) return -2;
    if (at < (size_t)nsub) return fail(-1, "model_index[%d] is out of range [0, %d)", (int)at, nmodel);
  }
  struct PosCheck { const double* p; const char* name; };
  for (const PosCheck& c : {PosCheck{A.P, "P"}, PosCheck{A.nu_DM, "nu_DM"}, PosCheck{A.nu_GM, "nu_GM"}, PosCheck{A.nu_tau, "nu_tau"}}) {
    if (!c.p) continue;
    if (find_bad(pl, c.p, (size_t)nsub, [](double v) { return !(v > 0.0); }, &at)) return -2;
    if (at < (size_t)nsub) return fail(-1, "%s[%d] is not positive", c.name, (int)at);
  }
  if (A.noise_std) {
    if (find_bad(pl, A.noise_std, nsc, [](double v) { return !(v >= 0.0); }, &at)) return -2;
    if (at < nsc) return fail(-1, "noise_std[%d, %d] is negative", (int)(at / nchan), (int)(at % nchan));
  }
  stats_begin(pl);
  // ---- the call's model spectra and frequency tables (own buffers: the fit's model set stays as it is)
  const int N = pl->N, L = nbin / 2;
  const int sstride = pl->anyn ? N : N + 1;
  const double* dmodels;
  if (stage_in(pl, pl->sim_models, A.models, nfreq * nbin, &dmodels)) return -2;
  CK(pl->sim_freqs.need(sizeof(double) * nfreq));
  CK(pl->sim_nu2.need(sizeof(double) * nfreq));
  CK(cudaMemcpyAsync(pl->sim_freqs.p, hf.data(), sizeof(double) * nfreq, cudaMemcpyHostToDevice, pl->stream));
  CK(cudaMemcpyAsync(pl->sim_nu2.p, hn2.data(), sizeof(double) * nfreq, cudaMemcpyHostToDevice, pl->stream));
  CK(pl->sim_mspec.need(sizeof(double2) * nfreq * sstride));
  if (pl->anyn) {
    CK(pl->sim_mdc.need(sizeof(double) * nfreq));
    if (launch_fwd_any(pl, nullptr, false, nullptr, nullptr, (long)nfreq, pl->sim_mspec.as<cx<double>>(),
                       pl->sim_mdc.as<double>(), dmodels)) return -2;
  } else {
    ModelArgs m;
    memset(&m, 0, sizeof m);
    m.model64 = dmodels; m.spec = pl->sim_mspec.as<cx<double>>(); m.nchan = (int)nfreq;
    m.twN = pl->twN64.as<cx<double>>(); m.tw2N = pl->tw2N64.as<cx<double>>();
    DISPATCH_N(N, (k_model<NN><<<row_ctas<NN>((long)nfreq), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(m)));
    pl->stats.launches++;
  }
  CK(cudaGetLastError());
  // ---- per-subint inputs and outputs: device arrays are used in place, host ones go through chunk-sized buffers,
  // so that the device scratch does not grow with nsub; each pointer is taken for what it is
  const double* src[9] = {A.phase, A.DM, A.P, A.nu_DM, A.GM, A.nu_GM, A.tau, A.alpha, A.nu_tau};
  bool src_dev[9];
  for (int i = 0; i < 9; ++i) src_dev[i] = src[i] && is_device_ptr(src[i]);
  const bool idx_dev = A.model_index && is_device_ptr(A.model_index);
  const bool scales_dev = A.scales && is_device_ptr(A.scales), sigma_dev = A.noise_std && is_device_ptr(A.noise_std);
  const bool data_dev = out->data && is_device_ptr(out->data), raw_dev = out->raw && is_device_ptr(out->raw);
  const bool scl_dev = out->raw && is_device_ptr(out->dat_scl), offs_dev = out->raw && is_device_ptr(out->dat_offs);
  size_t per_sub = sizeof(double) * 9 + sizeof(int);   // scratch bytes per subint (upper bound)
  if (A.scales && !scales_dev) per_sub += (size_t)nchan * sizeof(double);
  if (A.noise_std && !sigma_dev) per_sub += (size_t)nchan * sizeof(double);
  if (out->data && !data_dev) per_sub += (size_t)nchan * nbin * sizeof(float);
  if (out->raw && !raw_dev) per_sub += (size_t)nchan * nbin * sizeof(int16_t);
  if (out->raw && !scl_dev) per_sub += (size_t)nchan * sizeof(float);
  if (out->raw && !offs_dev) per_sub += (size_t)nchan * sizeof(float);
  if (pl->anyn) per_sub += (size_t)nchan * (sizeof(double2) * N + sizeof(double) + sizeof(double) * nbin);
  int chunk = pl->chunk_req > 0 ? std::min(pl->chunk_req, nsub)
                                : (int)std::max<size_t>(1, std::min<size_t>((size_t)nsub, kSimChunkBytes / per_sub));
  // (one CTA per row for the other-nbin kernels: gridDim.x <= 2^31 - 1 rows)
  chunk = (int)std::min<long>(chunk, std::max(1L, 2000000000L / nchan));
  if (out->data && !data_dev) CK(pl->sim_out.need((size_t)chunk * nchan * nbin * sizeof(float)));
  if (out->raw && !raw_dev) CK(pl->sim_raw.need((size_t)chunk * nchan * nbin * sizeof(int16_t)));
  if (out->raw && !scl_dev) CK(pl->sim_scl.need((size_t)chunk * nchan * sizeof(float)));
  if (out->raw && !offs_dev) CK(pl->sim_offs.need((size_t)chunk * nchan * sizeof(float)));
  if (pl->anyn) {
    CK(pl->sim_spec.need(sizeof(double2) * (size_t)chunk * nchan * N));
    CK(pl->sim_dc.need(sizeof(double) * (size_t)chunk * nchan));
    CK(pl->sim_rows.need(sizeof(double) * (size_t)chunk * nchan * nbin));
  }
  SimArgs a;
  memset(&a, 0, sizeof a);
  a.r.nu2 = pl->sim_nu2.as<double>(); a.r.nchan = nchan;
  a.r.twN = pl->twN64.p; a.r.tw2N = pl->tw2N64.p;
  a.mspec = pl->sim_mspec.as<cx<double>>(); a.mdc = pl->anyn ? pl->sim_mdc.as<double>() : nullptr;
  a.freqs = pl->sim_freqs.as<double>();
  a.key0 = (unsigned)A.seed; a.key1 = (unsigned)(A.seed >> 32);
  a.nchan = nchan; a.nbin = nbin; a.sstride = sstride;
  {
    SpanGuard sg(pl, SP_TOTAL);
    for (int s0 = 0; s0 < nsub; s0 += chunk) {
      const int ns = std::min(chunk, nsub - s0);
      const size_t r0 = (size_t)s0 * nchan, rows = (size_t)ns * nchan;
      const double* par[9];
      for (int i = 0; i < 9; ++i)
        if (chunk_in(pl, pl->sim_par[i], src[i], src_dev[i], (size_t)s0, (size_t)ns, &par[i])) return -2;
      a.r.phase = par[0]; a.r.DM = par[1]; a.r.P = par[2]; a.r.nu_ref = par[3]; a.r.GM = par[4]; a.r.nu_GM = par[5];
      a.tau = par[6]; a.alpha = par[7]; a.nu_tau = par[8];
      const int32_t* idx;
      if (chunk_in(pl, pl->sim_index, A.model_index, idx_dev, (size_t)s0, (size_t)ns, &idx)) return -2;
      a.index = idx;
      if (chunk_in(pl, pl->sim_scales, A.scales, scales_dev, r0, rows, &a.scales)) return -2;
      if (chunk_in(pl, pl->sim_sigma, A.noise_std, sigma_dev, r0, rows, &a.sigma)) return -2;
      a.s_first = (long long)A.first_subint + s0;
      a.out = !out->data ? nullptr : data_dev ? out->data + r0 * nbin : pl->sim_out.as<float>();
      a.raw = !out->raw ? nullptr : raw_dev ? out->raw + r0 * nbin : pl->sim_raw.as<int16_t>();
      a.dat_scl = !out->raw ? nullptr : scl_dev ? out->dat_scl + r0 : pl->sim_scl.as<float>();
      a.dat_offs = !out->raw ? nullptr : offs_dev ? out->dat_offs + r0 : pl->sim_offs.as<float>();
      if (pl->anyn) {
        k_sim_mul<<<(unsigned)rows, 256, 0, pl->stream>>>(a, pl->sim_spec.as<cx<double>>(), pl->sim_dc.as<double>(), N, L);
        if (launch_inv_any(pl, pl->sim_spec.as<cx<double>>(), pl->sim_dc.as<double>(), pl->sim_rows.p, (long)rows, true)) return -2;
        k_sim_store<<<(unsigned)rows, 256, 0, pl->stream>>>(a, pl->sim_rows.as<double>());
        pl->stats.launches += 2;
      } else {
        DISPATCH_N(N, (k_simulate<NN><<<row_ctas<NN>((long)rows), 256, fft_smem_bytes<NN, double>(), pl->stream>>>(a, ns)));
        pl->stats.launches++;
      }
      CK(cudaGetLastError());
      if (out->data && !data_dev && d2h_staged(pl, out->data + r0 * nbin, a.out, rows * nbin * sizeof(float))) return -2;
      if (out->raw && !raw_dev && d2h_staged(pl, out->raw + r0 * nbin, a.raw, rows * nbin * sizeof(int16_t))) return -2;
      if (out->raw && !scl_dev && d2h_staged(pl, out->dat_scl + r0, a.dat_scl, rows * sizeof(float))) return -2;
      if (out->raw && !offs_dev && d2h_staged(pl, out->dat_offs + r0, a.dat_offs, rows * sizeof(float))) return -2;
    }
  }
  CK(cudaStreamSynchronize(pl->stream));
  stats_end(pl);
  return 0;
}

// ----------------------------------------------------------------------------
// PCA / B-spline model building (pca.cuh)
// ----------------------------------------------------------------------------
static int pca_tile(pp_plan* pl, const PcaTileArgs& t) {
  const dim3 grid((unsigned)((t.J + kPcaTile - 1) / kPcaTile), (unsigned)((t.I + kPcaTile - 1) / kPcaTile));
  k_pca_tile<<<grid, 256, 0, pl->stream>>>(t);
  pl->stats.launches++;
  CK(cudaGetLastError());
  return 0;
}

static PcaOp pca_op(const double* p, const double* mean, const double* rw, int ld, int trans) {
  PcaOp o;
  o.p = p; o.mean = mean; o.rw = rw; o.ld = ld; o.trans = trans;
  return o;
}

extern "C" int pp_pca_moments(pp_plan_t* pl, const double* port, const double* weights, int32_t gram, double* mean_out,
                              double* moment_out) {
  if (!pl || !port || !weights || !mean_out || !moment_out) return fail(-1, "NULL argument");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int nchan = pl->nchan, nbin = pl->nbin;
  const double *dx, *dw;
  if (stage_in(pl, pl->pca_x, port, (size_t)nchan * nbin, &dx)) return -2;
  if (stage_in(pl, pl->pca_w, weights, (size_t)nchan, &dw)) return -2;
  CK(pl->pca_mu.need(sizeof(double) * nbin));
  CK(pl->pca_rw.need(sizeof(double) * nchan));
  CK(pl->pca_wsum.need(sizeof(double)));
  const int dim = gram ? nchan : nbin;
  CK(pl->pca_out.need(sizeof(double) * (size_t)dim * dim));
  double* mu = pl->pca_mu.as<double>();
  double* rw = pl->pca_rw.as<double>();
  double* W = pl->pca_wsum.as<double>();
  k_pca_mean<<<(unsigned)((std::max(nbin, nchan) + 255) / 256), 256, 0, pl->stream>>>(dx, dw, mu, rw, W, nchan, nbin);
  pl->stats.launches++;
  CK(cudaGetLastError());
  double wsum = 0.0;
  CK(cudaMemcpyAsync(&wsum, W, sizeof(double), cudaMemcpyDeviceToHost, pl->stream));
  CK(cudaStreamSynchronize(pl->stream));
  if (!(wsum > 0.0) || !std::isfinite(wsum)) return fail(-1, "the weights must sum to a positive finite value (got %g)", wsum);
  PcaTileArgs t;
  const PcaOp D = pca_op(dx, mu, rw, nbin, 0);
  t.a = D; t.b = D;
  t.a.trans = gram ? 0 : 1;   // covariance: a(i, k) = d_k[i]; Gram: a(i, k) = d_i[k]
  t.b.trans = gram ? 1 : 0;
  t.out = pl->pca_out.as<double>(); t.div = W;
  t.I = t.J = dim; t.K = gram ? nbin : nchan; t.sym = 1;
  if (pca_tile(pl, t)) return -2;
  if (copy_out_at(pl->stream, mean_out, mu, 0, (size_t)nbin)) return -2;
  if (copy_out_at(pl->stream, moment_out, t.out, 0, (size_t)dim * dim)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

extern "C" int pp_pca_project(pp_plan_t* pl, const double* port, const double* weights, const double* mean,
                              const double* vecs, int32_t m, int32_t back, double* out) {
  if (!pl || !port || !mean || !vecs || !out || (back && !weights)) return fail(-1, "NULL argument");
  const int nchan = pl->nchan, nbin = pl->nbin;
  const int rows_in = back ? nchan : nbin;   // rows of vecs
  if (m < 1 || m > rows_in) return fail(-1, "m must be in [1, %d] (got %d)", rows_in, m);
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const double *dx, *dmu, *dv, *dw = nullptr;
  if (stage_in(pl, pl->pca_x, port, (size_t)nchan * nbin, &dx)) return -2;
  if (stage_in(pl, pl->pca_mu, mean, (size_t)nbin, &dmu)) return -2;
  if (stage_in(pl, pl->pca_vecs, vecs, (size_t)rows_in * m, &dv)) return -2;
  const int rows_out = back ? nbin : nchan;
  CK(pl->pca_out.need(sizeof(double) * (size_t)rows_out * m));
  PcaTileArgs t;
  if (back) {
    if (stage_in(pl, pl->pca_w, weights, (size_t)nchan, &dw)) return -2;
    CK(pl->pca_rw.need(sizeof(double) * nchan));
    k_pca_mean<<<(unsigned)((nchan + 255) / 256), 256, 0, pl->stream>>>(dx, dw, nullptr, pl->pca_rw.as<double>(), nullptr,
                                                                        nchan, nbin);   // rw only
    pl->stats.launches++;
    CK(cudaGetLastError());
    t.a = pca_op(dx, dmu, pl->pca_rw.as<double>(), nbin, 1);   // a(b, n) = d_n[b]
  } else {
    t.a = pca_op(dx, dmu, nullptr, nbin, 0);                   // a(n, b) = x_n[b] - mean[b]
  }
  t.b = pca_op(dv, nullptr, nullptr, m, 0);
  t.out = pl->pca_out.as<double>(); t.div = nullptr;
  t.I = rows_out; t.J = m; t.K = rows_in; t.sym = 0;
  if (pca_tile(pl, t)) return -2;
  if (back) {
    k_pca_unit<<<(unsigned)m, 256, 0, pl->stream>>>(t.out, nbin, m);
    pl->stats.launches++;
    CK(cudaGetLastError());
  }
  if (copy_out_at(pl->stream, out, t.out, 0, (size_t)rows_out * m)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}

template <int N> static cudaError_t launch_lowpass(pp_plan* pl, const LowpassArgs& a, int nrows) {
  const cudaError_t e = cudaFuncSetAttribute(k_lowpass<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lowpass_smem_bytes<N>());
  if (e != cudaSuccess) return e;
  k_lowpass<N><<<(unsigned)nrows, 256, lowpass_smem_bytes<N>(), pl->stream>>>(a);
  return cudaGetLastError();
}

extern "C" int pp_lowpass_rows(pp_plan_t* pl, const double* rows, int32_t nrows, double* out, int32_t* kc_out) {
  if (!pl || !rows || !out || !kc_out) return fail(-1, "NULL argument");
  if (nrows < 1) return fail(-1, "nrows must be >= 1");
  CK(cudaSetDevice(pl->device));
  stats_begin(pl);
  const int nbin = pl->nbin;
  const double* din;
  if (stage_in(pl, pl->lp_in, rows, (size_t)nrows * nbin, &din)) return -2;
  CK(pl->lp_out.need(sizeof(double) * (size_t)nrows * nbin));
  CK(pl->lp_kc.need(sizeof(int) * (size_t)nrows));
  double* dout = pl->lp_out.as<double>();
  int* dkc = pl->lp_kc.as<int>();
  if (pl->anyn) {
    const int N = pl->N, L = pl->L;
    CK(pl->any_spec2.need(sizeof(double2) * (size_t)nrows * N));
    CK(pl->any_dc2.need(sizeof(double) * (size_t)nrows));
    cx<double>* spec = pl->any_spec2.as<cx<double>>();
    double* dc = pl->any_dc2.as<double>();
    if (launch_fwd_any(pl, nullptr, false, nullptr, nullptr, nrows, spec, dc, din)) return -2;
    const size_t smem = sizeof(double) * 2 * (size_t)(L + 1);
    CK(cudaFuncSetAttribute(k_lowpass_spec, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_lowpass_spec<<<(unsigned)nrows, 256, smem, pl->stream>>>(spec, dc, dkc, N, L);
    pl->stats.launches++;
    CK(cudaGetLastError());
    if (launch_inv_any(pl, spec, dc, dout, nrows, true)) return -2;
  } else {
    LowpassArgs a;
    a.in = din; a.out = dout; a.kc = dkc; a.twN = pl->twN64.p; a.tw2N = pl->tw2N64.p;
    cudaError_t e = cudaSuccess;
    DISPATCH_N(pl->N, e = launch_lowpass<NN>(pl, a, nrows));
    CK(e);
    pl->stats.launches++;
  }
  CK(cudaGetLastError());
  if (copy_out_at(pl->stream, out, dout, 0, (size_t)nrows * nbin)) return -2;
  if (copy_out_at(pl->stream, kc_out, (int32_t*)dkc, 0, (size_t)nrows)) return -2;
  CK(cudaStreamSynchronize(pl->stream));
  return 0;
}
