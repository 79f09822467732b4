/*
 * ppb200.h -- C ABI of the B200-native wideband-TOA engine.
 *
 * This is the drop-in boundary for ONE hot path of pennucci/PulsePortraiture:
 * the extended-FFTFIT fit.  Plain pointers and sizes only; no torch / numpy
 * types.  Every entry point cites the reference interface it replaces
 * (file:line into the reference tree).  The Python facade in
 * pulseportraiture_b200/ binds these symbols with ctypes (see INTEGRATION.md
 * for the stub a reference maintainer would add).
 *
 * Conventions
 *   - All array arguments may be HOST or DEVICE pointers (detected with
 *     cudaPointerGetAttributes); outputs are written where they point.
 *   - Row-major, C-contiguous.  data/model are float32 (the device storage
 *     type); every scalar/vector parameter is float64.
 *   - A plan is bound to one device and one stream; calls are synchronous
 *     with respect to the caller (they return after results are complete)
 *     unless stated otherwise.  One plan per (device, host thread).
 *   - DEVICE inputs are read on the plan's stream: work queued on another
 *     stream that produces them must be complete (or pp_plan_set_stream must
 *     name that stream) before the call.  The Python wrapper synchronises the
 *     caller's current torch stream for CUDA tensors.
 *   - Return value 0 = success, negative = error (see pp_last_error()).
 *   - nbin: any even number, 64 <= nbin <= 4096 (the reference's np.fft.rfft takes any length,
 *     pplib.py:2127).  Powers of two run the tuned row kernels; other lengths run the same DFT as a
 *     chirp-z (Bluestein) transform on top of them (csrc/bluestein.cuh): same results, not tuned.
 *   - The DC harmonic is ignored (reference F0_fact = 0, pplib.py:66) and
 *     Dconst = 1/0.000241 (pplib.py:48-51).
 */
#ifndef PPB200_H
#define PPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPB200_ABI_VERSION 6

typedef struct pp_plan pp_plan_t;

/* ---- plan ---------------------------------------------------------------
 * Replaces the implicit per-call setup of pplib.fit_portrait
 * (pplib.py:2127-2138) / pptoaslib.fit_portrait_full (pptoaslib.py:972-989):
 * FFT twiddles, device scratch, the model-side spectra. */
int pp_plan_create(int32_t nchan, int32_t nbin, int32_t device,
                   pp_plan_t** plan_out);
void pp_plan_destroy(pp_plan_t* plan);

/* Use an externally created cudaStream_t (e.g. a torch stream) for all work
 * of this plan.  NULL restores the plan's own stream. */
int pp_plan_set_stream(pp_plan_t* plan, void* cuda_stream);

/* Number of subints processed per pipeline chunk (0 = automatic: sized so a
 * chunk's cross-spectra stay L2-resident). */
int pp_plan_set_chunk(pp_plan_t* plan, int32_t subints_per_chunk);

/* FFT arithmetic of the auxiliary row transforms (pp_fit_phase_shift_batch
 * profiles, pp_get_noise_batch; pp_rotate_batch uses double only with 64):
 * 0 = automatic (double), 32, 64.  pp_fit_batch always transforms the data
 * rows in double (chi^2 to 1e-8 needs it, DESIGN.md section 4). */
int pp_plan_set_fft_precision(pp_plan_t* plan, int32_t bits);

/* (phi, DM) solver: Newton steps taken per pass on the local model built from
 * the per-channel theta-derivatives up to the fourth order (0 = default 8).
 * 1 = one Newton step per pass over the cross-spectrum, i.e. every step is
 * evaluated on the data (more passes, same optimum; used by the tests to
 * check the model-based steps). */
int pp_plan_set_model_steps(pp_plan_t* plan, int32_t steps);

/* General (GM / tau / alpha) solver, coarse-to-fine start.  Its first Newton iterations run on cheaper objectives:
 * the low harmonics only -- the leading groups of 16 harmonics that hold `frac` (default 0.99) of the phase
 * information sum_n sum_k k^2 |m_nk|^2 |B_nk|^2 of the model scattered with the start values -- preceded, where
 * that pays, by a level with fewer harmonics still (0.65 of the information) of every 2nd / 4th / 8th channel.
 * Each costs a fraction of a pass over the cross-spectrum and brings the start values to within a fraction of a
 * sigma of the optimum; the full-resolution iterations that follow decide convergence exactly as without it
 * (same optimum and errors, two full passes instead of five to nine).  frac = 0 disables the coarse levels, as do
 * pp_plan_set_model_steps(plan, 1) and a model whose information is spread over more than half of the harmonics.
 * nfeval counts coarse and full evaluations alike; pp_stats_t tells them apart. */
int pp_plan_set_coarse(pp_plan_t* plan, double frac);

/* Harmonic cut-off from the model.  The objective sees the data only through X_nk = d_nk conj(m_nk)
 * (pplib.py:2136-2138, 1319-1322): where the model has no power the cross-spectrum carries nothing.  For every
 * channel the kernels compute, store and stream only the leading groups of 16 harmonics outside which the model
 * holds less than eps^2 of its k^2-weighted power sum_k k^2 |m_nk|^2 (default eps = 1e-10: chi^2 moves by < 2e-10
 * relative, the parameters by ~1e-9 sigma; the noise level and Sd always use every harmonic of the data).  Smooth
 * templates (Gaussian / spline models) keep a quarter of the harmonics or less; a template with a noise floor
 * keeps them all.  eps = 0 keeps every harmonic of every channel.  pp_stats_t.x_keep_frac reports the kept share. */
int pp_plan_set_model_cutoff(pp_plan_t* plan, double eps);

/* Channel frequencies [nchan] MHz only (enough for pp_rotate_batch).  After pp_set_models these replace model 0's
 * table. */
int pp_set_freqs(pp_plan_t* plan, const double* freqs);

/* Model portrait [nchan, nbin] float32 and channel frequencies [nchan] MHz.
 * Computes conj(rfft(model)), |rfft(model)|^2 and p_n = sum_k |m_nk|^2 once
 * (pplib.py:2129-2130, 2138; pptoaslib.py:978-979). */
int pp_set_model(pp_plan_t* plan, const float* model, const double* freqs);

/* The same with the model portrait in float64, the reference's array type (pplib.py:2129): its spectrum then has
 * no float32 rounding floor (~1e-15 of the peak power in every harmonic), which is what lets the harmonic cut-off
 * above drop the harmonics an analytic template has no power in.  (Arbitrary nbin: rounded to float32 on the
 * device, as pp_set_model.) */
int pp_set_model_f64(pp_plan_t* plan, const double* model, const double* freqs);

/* nmodel model portraits [nmodel, nchan, nbin] and their frequency tables [nmodel, nchan] MHz (host or device).
 * Model m is everything pp_set_model computes, for table m; pp_set_model is the nmodel = 1 case.  Replaces the
 * per-subint read_model of pptoas.py:356-394: pp_fit_batch_models then fits each subint of one batch against its own
 * model and table.  Every frequency of every table must be positive.
 * Device memory per model, N = nbin/2 for power-of-two nbin (other nbin: N = the padded row length, the smallest
 * power of two above nbin/2):  nchan * (32 N + 36) + 8 N + 12 bytes (conj(m) in float and double, |m|^2, p_n, the
 * harmonic cut-off and three frequency tables per channel; the mean spectrum, the cut-off and the coarse levels per
 * model); other nbin add 16 N bytes per channel of transform scratch.  A staging copy of the portraits themselves
 * (nchan * nbin * 4 or 8 bytes per model) is kept when they come from host memory.  The plan keeps the largest model
 * set it has held.
 * pp_rotate_batch, pp_rotate_full_batch, pp_apply_response_batch, pp_align_accumulate, the noise entry points and
 * the model generators use one table: model 0's, or that of the last pp_set_freqs call.
 * pp_plan_set_model_cutoff recomputes the cut-offs of every model; pp_stats_t.x_keep_frac is the kept share over
 * all models' channels. */
int pp_set_models(pp_plan_t* plan, int32_t nmodel, const float* models, const double* freqs);
int pp_set_models_f64(pp_plan_t* plan, int32_t nmodel, const double* models, const double* freqs);

/* ---- batched wideband fit ------------------------------------------------
 * Replaces, per subint, the sequence of pptoas.GetTOAs.get_TOAs
 * (pptoas.py:402-486): [FFTFIT initial guess] -> fit_portrait_full
 * (pptoaslib.py:928-1096); with fit_flags = {1,1,0,0,0} and
 * semantics = PP_SEM_FIT_PORTRAIT it is pplib.fit_portrait
 * (pplib.py:2102-2204). */
enum { PP_DATA_F32 = 0, PP_DATA_I16 = 1, PP_DATA_F64 = 2 };   /* pp_fit_args_t.data_type */
enum {
  PP_SEM_FIT_PORTRAIT_FULL = 0, /* pptoaslib.py:928: covariance incl. amplitudes */
  PP_SEM_FIT_PORTRAIT = 1       /* pplib.py:2102: scale_errs = (p_n/sigma^2)^-1/2 */
};

typedef struct {
  const float* data;        /* [nsub,nchan,nbin] float32                       */
  int32_t nsub;
  int32_t semantics;        /* PP_SEM_*                                        */
  const double* P;          /* [nsub] spin period [s]                          */
  const double* errs;       /* [nsub,nchan] time-domain noise sigma, or NULL:
                               measured as get_noise_PS (pplib.py:2227-2253)   */
  const uint8_t* chan_mask; /* [nsub,nchan] 1 = use channel; NULL = all        */
  const double* weights;    /* [nsub,nchan] weights of the frequency average
                               used for the initial guess (pptoas.py:424);
                               NULL = 1                                        */
  const double* init;       /* [nsub,5] phi,DM,GM,tau(or log10),alpha at
                               nu_fits; NULL = FFTFIT guess (pptoas.py:421-456)*/
  const double* DM_guess;   /* [nsub] DM used to dedisperse for the guess and
                               as DM start value (pptoas.py:421); NULL = 0     */
  const double* snrs;       /* [nsub,nchan] per-channel S/N for guess_fit_freq
                               (pplib.py:2618) when nu_fits==NULL and
                               nu_fit_mode==1; NULL = ones                     */
  const double* nu_fits;    /* [nsub,3] fit reference freqs or NULL            */
  int32_t nu_fit_mode;      /* with nu_fits==NULL: 0 = mean of used freqs
                               (pptoaslib.py:986-989); 1 = guess_fit_freq
                               (pptoas.py:402)                                 */
  const double* nu_outs;    /* [nsub,3] output reference freqs; NaN (or NULL)
                               = zero-covariance frequency (pptoaslib.py:1040) */
  uint8_t fit_flags[5];     /* phi, DM, GM, tau, alpha                         */
  int32_t log10_tau;        /* pptoaslib.py:931                                */
  int32_t option;           /* get_nu_zeros option (pptoaslib.py:734)          */
  int32_t is_toa;           /* pptoaslib.py:1048-1050                          */
  int32_t Ns;               /* FFTFIT grid size (pplib.py:2054), default 100   */
  int32_t max_iter;         /* Newton passes per subint (0 = default 40; passes run
                               only while some subint has not converged).
                               < 0: evaluate only: one pass at init (or at the
                               FFTFIT guess), the epilogue (chi2, scales, snr,
                               errors, nu_out, chan_sums) at that point, no
                               step; return code 0 (pplib.get_scales)         */
  double tol;               /* convergence: |step| < tol * 1-sigma (0 = default:
                               1e-3; the (phi, DM) solver's model-based steps
                               stop at min(tol, 1e-4), see
                               pp_plan_set_model_steps)                        */
  const double* scat_guess; /* [nsub,2] with init==NULL: tau start value [rot,
                               linear] at nu_fit_tau and alpha start value
                               (pptoas.py:427-452); NULL = 0, 0                */
  int32_t data_type;        /* PP_DATA_F32 (0): data is float32.  PP_DATA_I16:
                               data points to int16 [nsub,nchan,nbin], the
                               PSRFITS DATA column as stored; samples are
                               raw*dat_scl + dat_offs evaluated in float32 as
                               PSRCHIVE decodes them (what load_data,
                               pplib.py:2669-2700, hands to the reference).
                               PP_DATA_F64: data is float64 (the reference's own
                               array type, pplib.py:2803); rounded to float32
                               on the device, chunk by chunk, so that a caller
                               holding float64 portraits needs no host pass    */
  const float* dat_scl;     /* [nsub,nchan] PSRFITS DAT_SCL (int16 only)       */
  const float* dat_offs;    /* [nsub,nchan] PSRFITS DAT_OFFS (int16 only)      */
  const double* bounds;     /* HOST [5,2] (lower, upper) for phi, DM, GM, tau
                               (log10 tau with log10_tau) and alpha, applied to
                               the parameters at the FIT reference frequencies
                               as scipy's TNC applies them (pplib.py:2146-2148,
                               pptoaslib.py:1008-1014; defaults of
                               pptoas.py:461-469).  NaN or +-inf = unbounded;
                               NULL = no bounds.  Parameters at a bound still
                               get their Hessian-based errors, as in the
                               reference                                       */
} pp_fit_args_t;

typedef struct {
  double* params;       /* [nsub,5] at the output reference frequencies        */
  double* param_errs;   /* [nsub,5] (0 for parameters not fit)                 */
  double* nu_out;       /* [nsub,3] nu_DM, nu_GM, nu_tau                       */
  double* cov;          /* [nsub,5,5] parameter covariance (0 rows if not fit) */
  double* chi2;         /* [nsub]                                              */
  double* red_chi2;     /* [nsub]                                              */
  double* snr;          /* [nsub]                                              */
  int32_t* nfeval;      /* [nsub] objective passes used                        */
  int32_t* return_code; /* [nsub] 0 converged, 1 max_iter, 3 non-finite        */
  double* scales;       /* [nsub,nchan]                                        */
  double* scale_errs;   /* [nsub,nchan]                                        */
  double* channel_snrs; /* [nsub,nchan]                                        */
  double* noise;        /* [nsub,nchan] time-domain sigma actually used        */
  int32_t* lag_index;   /* [nsub] FFTFIT integer grid argmin (-1 if init given)*/
  double* phi_guess;    /* [nsub] initial phase handed to the solver           */
  double* chan_sums;    /* [nsub,nchan,9] per-channel C,Cth,Cthth,Ct,Ctt,Ctht,
                           S,St,Stt at the last evaluated point (for host
                           epilogues); for the (phi, DM) solver slots 3, 4 hold
                           the third and fourth theta-derivatives of C instead
                           and slots 5-8 are 0.  The (phi, DM) solver runs when
                           GM, tau and alpha are not fit, GM and tau are 0 in a
                           host init, log10_tau is off and scat_guess is NULL
                           (a device init takes the general solver)           */
  double* align_sum;    /* [nchan,nbin] ppalign (ppalign.py:197-213), fused: the
                           sum over the batch of w_sn * rotate(data_sn, phi_s,
                           DM_s about nu_out_s) with the FITTED phi_s, DM_s and
                           w_sn = scales_sn / sigma_sn^2 (0 for unused channels
                           and failed subints); not normalised                 */
  double* align_wsum;   /* [nchan] sum_s w_sn (required with align_sum)        */
} pp_fit_out_t;          /* any member may be NULL                              */

int pp_fit_batch(pp_plan_t* plan, const pp_fit_args_t* args,
                 const pp_fit_out_t* out);

/* pp_fit_batch with model_index [nsub] int32 in [0, nmodel) (host or device): subint s is fit against model
 * model_index[s] on frequency table model_index[s] (pp_set_models).  pp_fit_batch(plan, a, o) is
 * pp_fit_batch_models(plan, a, NULL, o); NULL is valid only when the plan holds one model.  The index is checked
 * before any kernel reads it (a device index costs one small copy to the host): an entry out of range is an error.
 * The FFTFIT guess uses each subint's own model (its mean spectrum and harmonic cut-off); the coarse levels of the
 * general solver are chosen per model present in a chunk, from that model's first subint of the chunk.  Results of a
 * subint are those of a pp_fit_batch call on its model's subints alone, bit for bit, when the batch is one chunk (the
 * (phi, DM) fit: for any chunking).  align_sum needs one model (ppalign has one template and one table). */
int pp_fit_batch_models(pp_plan_t* plan, const pp_fit_args_t* args, const int32_t* model_index,
                        const pp_fit_out_t* out);

/* ---- batched 1-D FFTFIT ---------------------------------------------------
 * Replaces pplib.fit_phase_shift (pplib.py:2054-2100) for n profiles.
 * models: [nmodel, nbin] with nmodel a divisor of n: profile i is fit against
 * model i mod nmodel (1 = one template; nchan = the per-channel fits of
 * get_narrowband_TOAs, pptoas.py:980-992, with profiles [nsub*nchan, nbin];
 * n = one model per profile).  noise: [n] time-domain
 * sigma or NULL (-> get_noise, pplib.py:2076).  The brute-force grid is
 * np.mgrid[-0.5:0.5:Ns*1j]; lag_index is its argmin; phase is the exact
 * minimiser reached from there (the reference's Nelder-Mead polish is only
 * 1e-4 accurate, SURVEY 8c). */
typedef struct {
  double* phase; double* phase_err; double* scale; double* scale_err;
  double* snr; double* red_chi2; int32_t* lag_index;
} pp_pshift_out_t;

int pp_fit_phase_shift_batch(pp_plan_t* plan, const float* profiles, int32_t n,
                             const float* models, int32_t nmodel,
                             const double* noise, int32_t Ns,
                             const pp_pshift_out_t* out);

/* Same with the `bounds` argument of pplib.fit_phase_shift (pplib.py:2054,
 * 2085): the brute-force grid is np.mgrid[phi_lo:phi_hi:Ns*1j].  As in the
 * reference the polish is not confined to the bounds. */
int pp_fit_phase_shift_batch_bounds(pp_plan_t* plan, const float* profiles,
                                    int32_t n, const float* models,
                                    int32_t nmodel, const double* noise,
                                    int32_t Ns, double phi_lo, double phi_hi,
                                    const pp_pshift_out_t* out);

/* ---- batched Fourier-domain rotation -------------------------------------
 * Replaces pplib.rotate_data / rotate_portrait (pplib.py:2338-2460) for
 * [nsub,nchan,nbin] float32: harmonic k of channel n is multiplied by
 * exp(+2 pi i k (phase_s + Dconst*DM_s/P_s*(nu_n^-2 - nu_ref_s^-2))).
 * in/out may alias. */
int pp_rotate_batch(pp_plan_t* plan, const float* in, float* out, int32_t nsub,
                    const double* phase, const double* DM, const double* P,
                    const double* nu_ref);

/* Same with the nu^-4 ("GM") delay term: replaces pptoaslib.rotate_portrait_full
 * (pptoaslib.py:52-81).  GM / nu_GM may be NULL (= pp_rotate_batch). */
int pp_rotate_full_batch(pp_plan_t* plan, const float* in, float* out, int32_t nsub,
                         const double* phase, const double* DM, const double* GM,
                         const double* P, const double* nu_DM, const double* nu_GM);

/* Per-channel, per-harmonic real response applied in the Fourier domain:
 * out[s,n] = irfft(resp[n,:] * rfft(in[s,n])), resp float64 [nchan, nbin/2+1] (host or device).
 * Replaces the model multiply of pptoas.py:388-394, modelx = irfft(instrumental_response_port_FT(...)
 * * rfft(modelx)) (the response table itself, pptoaslib.py:112-179, is a few kB of host arithmetic:
 * pptoaslib.instrumental_response_port_FT).  in/out may alias. */
int pp_apply_response_batch(pp_plan_t* plan, const float* in, float* out, int32_t nsub,
                            const double* resp);

/* ---- align-and-accumulate (ppalign inner loop) ---------------------------------
 * Replaces the per-subint accumulation of ppalign.align_archives
 * (ppalign.py:202-208): aligned[n] = sum_s weights[s,n] * rotate_data(data[s,n],
 * phase_s, DM_s, P_s, freqs, nu_ref_s), accumulated in the Fourier domain in
 * double; rows with weight 0 are skipped (negative weights count, as in the reference).  aligned: [nchan,nbin] float64
 * (not normalised), wsum: [nchan] float64. */
int pp_align_accumulate(pp_plan_t* plan, const float* data, int32_t nsub,
                        const double* phase, const double* DM, const double* P,
                        const double* nu_ref, const double* weights,
                        double* aligned, double* wsum);

/* Evolving-Gaussian model portrait generated on the device: replaces
 * pplib.gen_gaussian_portrait (pplib.py:853-930) with evolve_parameter
 * (pplib.py:996-1046), gaussian_profile (pplib.py:770-825) and the analytic
 * scattering of pplib.py:4049-4095; what read_model (pplib.py:2867-2953) calls
 * per archive / per subint (pptoas.py:356-379).
 *   model_code  three characters '0' (power law) / '1' (linear) for loc, wid, amp
 *   params      HOST [2 + 6*ngauss]: DC, tau [bin], then per component
 *               loc, m_loc, wid, m_wid, amp, m_amp  (as read from a .gmodel file)
 *   out         float [nchan, nbin], host or device; frequencies from pp_set_freqs.
 * The result can be handed to pp_set_model without leaving the device. */
int pp_gen_gaussian_portrait(pp_plan_t* plan, const char* model_code,
                             const double* params, int32_t ngauss,
                             double scattering_index, double nu_ref, float* out);

/* The same portrait in float64 (an unscattered model is evaluated and stored in double: what pp_set_model_f64
 * and the harmonic cut-off want; a scattered one, tau != 0, passes through float32 rows). */
int pp_gen_gaussian_portrait_f64(pp_plan_t* plan, const char* model_code,
                             const double* params, int32_t ngauss,
                             double scattering_index, double nu_ref, double* out);

/* B-spline (PCA) model portrait on the device: replaces pplib.gen_spline_portrait
 * (pplib.py:932-956) as called by read_spline_model (pplib.py:2955-2987;
 * pptoas.py:376-379):  out[n,:] = mean_prof + sum_c s_c(freqs[n]) * eigvec[:,c]
 * with s_c = scipy.interpolate.splev(freqs, (knots, coefs, degree), ext=0).
 *   mean_prof HOST [nbin]; eigvec HOST [nbin, ncomp] row-major; knots HOST
 *   [nknots]; coefs HOST [ncomp, nknots-degree-1]; out float [nchan, nbin]
 *   host or device.  The model must already have the plan's nbin (the
 *   reference's optional ss.resample step is not provided). */
int pp_gen_spline_portrait(pp_plan_t* plan, const double* mean_prof,
                           const double* eigvec, int32_t ncomp,
                           const double* knots, int32_t nknots,
                           const double* coefs, int32_t degree, float* out);

/* get_noise_fit(data, fact, chans=True) of pplib.py:2255-2284: the noise floor of each row's power
 * spectrum starts at fact * find_kc(pows) (pplib.py:1465-1495, scipy.optimize.brute over a 20^3 grid of
 * the b exp(-a k) + dc model of log10 pows, evaluated on the device). */
int pp_get_noise_fit_batch(pp_plan_t* plan, const float* data, int32_t nsub, double fact,
                           double* noise_out);

/* Measured FP64 yardstick for the roofline record: DFMA thread-instructions per second of a kernel
 * of independent DFMA chains on the plan's device (no reference counterpart: measurement support). */
int pp_measure_fp64(pp_plan_t* plan, double* dfma_per_second);

/* ---- per-channel noise -----------------------------------------------------
 * Replaces pplib.get_noise(data, chans=True) (pplib.py:2227-2245). */
int pp_get_noise_batch(pp_plan_t* plan, const float* data, int32_t nsub,
                       double* noise_out);

/* The same estimate from the harmonics k >= kc of each row (kc < 0: the default int(0.75 nharm));
 * get_noise_PS(data, frac) of pplib.py:2227-2253 is kc = int((1 - 1/frac) * (nbin/2 + 1)). */
int pp_get_noise_cut_batch(pp_plan_t* plan, const float* data, int32_t nsub, int32_t kc,
                           double* noise_out);

/* ---- evolving-Gaussian model fit (ppgauss) ----------------------------------------
 * Replaces the numerical core of pplib.fit_gaussian_portrait (pplib.py:1924-2052): a weighted least-squares
 * fit of the evolving-Gaussian portrait of gen_gaussian_portrait (pplib.py:853-930), scattered when tau or
 * alpha is free or tau != 0, to nport portraits at once.  P = 3 + 6*ngauss parameters per portrait:
 *   [DC, tau [bin at nu_ref], (loc, m_loc, wid, m_wid, amp, m_amp) x ngauss, alpha]
 * chi^2 = sum_n sum_t (d_nt - m_nt)^2 / sigma_n^2, the DC harmonic included, evaluated in the Fourier domain
 * (Parseval) in FP64 with analytic derivatives.  Levenberg-Marquardt on the Marquardt-scaled normal
 * equations; bounds as an active set (starts are moved into the box, a parameter on a bound whose gradient
 * points outwards is held, steps are clipped to the box).  Stops when every free parameter's Gauss-Newton
 * step is below tol x its sigma.  Frequencies from pp_set_freqs; nbin a power of two (64..4096).  Results of
 * a portrait do not depend on the batch or chunk it is fit in (pp_plan_set_chunk: portraits per chunk). */
typedef struct {
  int32_t nport;
  const double* data;       /* [nport,nchan,nbin] float64, host or device         */
  const double* errs;       /* [nport,nchan] sigma_n > 0, host or device         */
  const char* model_code;   /* three characters '0' (power law) / '1' (linear)
                               for loc, wid, amp                                 */
  int32_t ngauss;           /* 1..16                                             */
  double nu_ref;            /* reference frequency of the parameters [MHz] > 0   */
  const double* init;       /* [nport,P] start values, host or device            */
  const uint8_t* fit_flags; /* HOST [P] nonzero = free; alpha's flag last        */
  const double* bounds;     /* HOST [P,2] (lower, upper); NaN = unbounded; NULL =
                               no bounds                                         */
  int32_t max_iter;         /* objective evaluations per portrait (0 = default
                               200); < 0: evaluate only: chi2, jtr, jtj at the
                               (boxed) start point, no step, return code 0       */
  double tol;               /* 0 = default 1e-4                                  */
} pp_gfit_args_t;

typedef struct {
  double* params;       /* [nport,P]                                              */
  double* param_errs;   /* [nport,P] sqrt(diag(cov)); 0 for fixed parameters      */
  double* cov;          /* [nport,P,P] (J^T J)^-1 red_chi2 over the free parameters
                           (lmfit's scale_covar); 0 rows / columns for fixed ones */
  double* chi2;         /* [nport]                                                */
  double* red_chi2;     /* [nport] chi2 / (nchan nbin - n_free)                   */
  int32_t* nfeval;      /* [nport] model + Jacobian evaluations                   */
  int32_t* return_code; /* [nport] 0 converged, 1 max_iter, 3 non-finite          */
  double* jtr;          /* [nport,P] J^T (d - m) / sigma^2 at params (free only)  */
  double* jtj;          /* [nport,P,P] J^T J / sigma^2 at params (free only)      */
  double* model;        /* [nport,nchan,nbin] float64 model portrait at params    */
} pp_gfit_out_t;        /* any member may be NULL; host or device pointers        */

int pp_fit_gaussian_portraits(pp_plan_t* plan, const pp_gfit_args_t* args,
                              const pp_gfit_out_t* out);

/* Join parameters (ppgauss's multi-receiver fit): one evolving-Gaussian model fit to a portrait whose channels
 * come from several archives, each archive after the first with its own phase and DM offset.  Channel n of group
 * j = join_chan[n] is rotated as rotate_data(row, phi_j, DM_j, P, freqs, nu_ref) after scattering: harmonic k is
 * multiplied by e^{2 pi i k theta_n}, theta_n = phi_j + Dconst DM_j / P (nu_n^-2 - nu_ref^-2), and the Nyquist term
 * (irfft keeps its real part) by cos(2 pi N theta_n).  Channels with join_chan[n] = -1 are not rotated.  The
 * parameter vector grows to P = 3 + 6*ngauss + 2*njoin:
 *   [DC, tau, (loc, m_loc, wid, m_wid, amp, m_amp) x ngauss, alpha, (phi_j, DM_j) x njoin]
 * and fit_flags, bounds, init and every output of pp_fit_gaussian_portraits_join cover all P entries.
 * NULL join or njoin = 0: exactly pp_fit_gaussian_portraits.  data (and errs) may be NULL when max_iter < 0 and
 * out->model is the only output: the model portraits at init (the device generator of joined models, FP64).
 * Errors: njoin > 8, P <= 0, a join_chan entry outside [-1, njoin), a group with no channel. */
typedef struct {
  int32_t njoin;              /* 0..8 groups                                            */
  const int32_t* join_chan;   /* HOST [nchan] group of each channel, -1 = none          */
  double P;                   /* spin period [s] of the DM term, > 0                    */
} pp_gfit_join_t;

int pp_fit_gaussian_portraits_join(pp_plan_t* plan, const pp_gfit_args_t* args,
                                   const pp_gfit_join_t* join, const pp_gfit_out_t* out);

/* ---- simulated archives ---------------------------------------------------------
 * Replaces the data generation of pplib.make_fake_pulsar (pplib.py:3183-3378) for a batch of subints, without the
 * PSRFITS writing.  Row (s, n), m = model_index[s]:
 *   Y_k = S_sn M_mnk e^{-2 pi i k theta_sn} B_snk  (k = 0..nbin/2),   out = irfft(Y) + sigma_sn z(seed, s_global, n, b)
 *   theta_sn = phase_s + Dconst DM_s (nu_n^-2 - nu_DM_s^-2)/P_s + Dconst^2 GM_s (nu_n^-4 - nu_GM_s^-4)/P_s
 *   B_snk = 1/(1 + 2 pi i k tau_sn),  tau_sn = tau_s (nu_n/nu_tau_s)^alpha_s [rot]
 * with M = rfft(models) in double (the DC and Nyquist terms included; irfft keeps the real part of the Nyquist
 * term).  The parameters are the injected ones: pp_fit_batch on the output recovers phase, DM, GM, tau and alpha
 * (a row is rotate_data(model, -phase, -DM), scattered).  The inverse transform is FP64.
 * Noise z: Philox4x32-10 with key (seed low, seed high) and counter (b/4, n, s_global low, s_global high),
 * s_global = first_subint + s, four uint32 per quad of bins 4q..4q+3, each mapped to u = f32((x >> 8) 2^-24 + 2^-25)
 * and pairs through Box-Muller in float32 (accurate logf, sqrtf, sincospif): (z0, z1) = sqrt(-2 ln u0) (cos 2 pi u1,
 * sin 2 pi u1); |z| <= 5.89.  A subint's samples depend only on (seed, s_global, its model and its parameters): not
 * on the batch, the chunk (pp_plan_set_chunk) or the device, so a study can be split over calls and GPUs.
 * Outputs: float32 rows and / or int16 rows with DAT_SCL / DAT_OFFS that are pptoas.quantize_subints of the float32
 * rows bit for bit (offs = f32((hi + lo)/2), scl = f32((hi - lo)/65000) or 1, raw = clip(rint((x - offs)/scl)) in
 * double).  Each array is taken for what it is, host or device, independently of the others: device outputs are
 * written in place, host outputs go through the plan's page-locked staging chunk by chunk, and host per-subint inputs
 * are staged chunk by chunk, so that device scratch is bounded independently of nsub.  The fit's model set and
 * frequency tables are not touched.
 * Errors (nothing is launched): nmodel < 1, a model index out of range, P <= 0, a frequency <= 0 (freqs, nu_DM,
 * nu_GM, nu_tau), a negative sigma, no output.  nsub = 0 does nothing. */
typedef struct {
  const double* models;       /* [nmodel,nchan,nbin] float64 model portraits (host or device)       */
  const double* freqs;        /* [nmodel,nchan] MHz                                                  */
  int32_t nmodel;
  const int32_t* model_index; /* [nsub] in [0, nmodel) or NULL (model 0)                             */
  int32_t nsub;
  int64_t first_subint;       /* global index of subint 0: the noise counter                         */
  uint64_t seed;
  const double* phase;        /* [nsub] rot                                                          */
  const double* DM;           /* [nsub]                                                              */
  const double* P;            /* [nsub] s, > 0                                                       */
  const double* nu_DM;        /* [nsub] MHz (inf allowed)                                            */
  const double* GM;           /* [nsub] or NULL, with nu_GM                                          */
  const double* nu_GM;
  const double* tau;          /* [nsub] rot at nu_tau, or NULL (unscattered), with alpha and nu_tau  */
  const double* alpha;
  const double* nu_tau;
  const double* scales;       /* [nsub,nchan] or NULL (= 1)                                          */
  const double* noise_std;    /* [nsub,nchan] time-domain sigma >= 0, or NULL (= 0)                  */
} pp_sim_args_t;

typedef struct {
  float* data;                /* [nsub,nchan,nbin] float32 or NULL                                   */
  int16_t* raw;               /* [nsub,nchan,nbin] int16 or NULL; dat_scl and dat_offs with it        */
  float* dat_scl;             /* [nsub,nchan]                                                        */
  float* dat_offs;            /* [nsub,nchan]                                                        */
} pp_sim_out_t;               /* host or device pointers; data or raw must be given                  */

int pp_simulate_batch(pp_plan_t* plan, const pp_sim_args_t* args, const pp_sim_out_t* out);

/* ---- PCA / B-spline model building ----------------------------------------------
 * The device steps of pplib.make_spline_model (after ppspline.py make_spline_model), FP64, on the plan's
 * [nchan, nbin] shape (any even nbin the plan takes).  With d_n = sqrt(w_n) (x_n - mu), W = sum_n w_n:
 *   pp_pca_moments: mu = sum_n w_n x_n / W [nbin], and C = sum_n d_n d_n^T / W [nbin, nbin] (gram = 0) or
 *     G = D D^T / W [nchan, nchan] (gram != 0), both triangles written and bit-symmetric.  Weights >= 0 (0 = excluded);
 *     W must be positive.
 *   pp_pca_project, back != 0: e_j = D^T u_j for the columns of vecs = U [nchan, m] (mean = mu, weights = w), each
 *     normalised to unit norm with its entry of largest |value| positive: out = E [nbin, m].
 *   pp_pca_project, back == 0: out = P [nchan, m], P_nj = sum_b (x_nb - mean_b) E_bj for vecs = E [nbin, m]
 *     (unweighted; weights unused).
 *   pp_lowpass_rows: per row of nbin samples: rfft, k_c = find_kc of the row's power spectrum (the rule of
 *     pp_get_noise_fit_batch, fact = 1), harmonics above k_c set to zero (DC kept, the Nyquist term kept only when
 *     k_c = nbin/2), irfft.  out [nrows, nbin], kc [nrows].
 * No floating-point atomics and a fixed summation order: outputs are bit-identical run to run.  Inputs and outputs
 * may be host or device pointers. */
int pp_pca_moments(pp_plan_t* plan, const double* port, const double* weights, int32_t gram, double* mean_out,
                   double* moment_out);
int pp_pca_project(pp_plan_t* plan, const double* port, const double* weights, const double* mean,
                   const double* vecs, int32_t m, int32_t back, double* out);
int pp_lowpass_rows(pp_plan_t* plan, const double* rows, int32_t nrows, double* out, int32_t* kc);

/* ---- diagnostics ------------------------------------------------------------ */
typedef struct {
  int64_t launches;        /* kernels launched by the last pp_* call            */
  int64_t pass_launches;   /* of which objective-pass kernels                   */
  int64_t pass_rows;       /* channel rows actually streamed by pass kernels    */
  double ms_spectra;       /* CUDA-event time of the FFT/precompute kernels     */
  double ms_guess;         /* ... FFTFIT guess kernels                          */
  double ms_pass;          /* ... objective pass kernels                        */
  double ms_update;        /* ... Newton update / epilogue kernels              */
  double ms_total;         /* first launch -> last kernel of the call           */
  int32_t chunk;           /* subints per chunk used                            */
  int32_t timing_enabled;
  int64_t coarse_launches; /* coarse (low-harmonic) iterations of the general solver, not in pass_launches */
  double ms_coarse;        /* ... their pass + update kernels                   */
  double x_keep_frac;      /* share of the cross-spectrum kept by the model's harmonic cut-off */
} pp_stats_t;

int pp_plan_enable_timing(pp_plan_t* plan, int32_t on);
int pp_get_stats(pp_plan_t* plan, pp_stats_t* stats);

/* Page-locked host memory for result / input buffers (makes the D2H / H2D
 * copies of pp_fit_batch asynchronous and full-speed). */
void* pp_host_alloc(uint64_t bytes);
void pp_host_free(void* p);

const char* pp_last_error(void);
int pp_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PPB200_H */
