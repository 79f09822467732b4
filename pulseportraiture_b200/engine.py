"""Batch-first Python front end of the C ABI (one plan per device).

``WidebandPlan`` is what the reference-compatible facade functions
(``pplib.fit_portrait``, ``pptoaslib.fit_portrait_full``,
``pplib.fit_phase_shift``, ``pptoas.GetTOAs``) are built on: they are the
``nsub = 1`` views of these batched calls.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _ffi

_KEEP = "_keepalive"


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x, dtype, keep, name, shape=None):
    """Raw pointer of a numpy array / torch tensor (host or CUDA); None->NULL."""
    if x is None:
        return None
    if _is_torch(x):
        import torch
        want = {np.float32: torch.float32, np.float64: torch.float64,
                np.uint8: torch.uint8, np.int32: torch.int32, np.int16: torch.int16}[dtype]
        if x.dtype != want:
            raise TypeError("%s: expected torch dtype %s, got %s" % (name, want, x.dtype))
        if not x.is_contiguous():
            raise ValueError("%s must be contiguous" % name)
        if shape is not None and tuple(x.shape) != tuple(shape):
            raise ValueError("%s: expected shape %s, got %s" % (name, shape, tuple(x.shape)))
        if x.is_cuda:
            # the plan works on its own stream: whatever torch still has queued for this tensor
            # on the caller's current stream must be finished before the kernels read it
            torch.cuda.current_stream(x.device).synchronize()
        keep.append(x)
        return x.data_ptr()
    a = np.ascontiguousarray(x, dtype=dtype)
    if shape is not None:
        a = a.reshape(shape)
    keep.append(a)
    return a.ctypes.data


class PinnedPool(object):
    """Named page-locked host arrays (pp_host_alloc), grown on demand."""

    def __init__(self, lib):
        self._lib, self._bufs = lib, {}

    def array(self, name, shape, dtype):
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        ent = self._bufs.get(name)
        if ent is None or ent[1] < nbytes:
            if ent is not None:
                self._lib.pp_host_free(C.c_void_p(ent[0]))
            cap = max(nbytes, 64)
            ptr = self._lib.pp_host_alloc(cap)
            if not ptr:
                raise _ffi.PPError("pp_host_alloc(%d) failed" % cap)
            ent = (ptr, cap)
            self._bufs[name] = ent
        raw = (C.c_char * nbytes).from_address(ent[0])
        return np.frombuffer(raw, dtype=dtype).reshape(shape)

    def close(self):
        for ptr, _ in self._bufs.values():
            self._lib.pp_host_free(C.c_void_p(ptr))
        self._bufs = {}


def bounds_array(bounds):
    """scipy-style bounds [(lo, hi), ...] (None = open) for the leading parameters -> float64
    [5, 2] with NaN for open ends, or None when nothing is bounded."""
    if bounds is None:
        return None
    out = np.full((5, 2), np.nan)
    for i, b in enumerate(bounds):
        if b is None:
            continue
        lo, hi = b
        out[i, 0] = np.nan if lo is None else float(lo)
        out[i, 1] = np.nan if hi is None else float(hi)
    return None if np.all(np.isnan(out)) else out


def model_bytes(nchan, nbin):
    """Device memory one model of pp_set_models costs on a [nchan, nbin] plan (include/ppb200.h): nchan * (32 N + 36)
    + 8 N + 12 bytes, N = nbin/2 slots per spectrum row (other than power-of-two nbin: the smallest power of two above
    nbin/2, plus 16 N bytes per channel of transform scratch).  The portraits' staging copy is not counted."""
    nchan, nbin = int(nchan), int(nbin)
    pow2 = nbin & (nbin - 1) == 0
    N = nbin // 2
    if not pow2:
        N = 1
        while N < nbin // 2 + 1:
            N *= 2
    per_chan = 32 * N + 36 + (0 if pow2 else 16 * N)
    return nchan * per_chan + 8 * N + 12


class WidebandPlan(object):
    """Device plan for portraits of shape [nchan, nbin] (C ABI pp_plan_*)."""

    def __init__(self, nchan, nbin, device=0, stream=None):
        self._lib = _ffi.lib()
        self._h = C.c_void_p()
        _ffi.check(self._lib.pp_plan_create(int(nchan), int(nbin), int(device),
                                            C.byref(self._h)), "pp_plan_create")
        self.nchan, self.nbin, self.device = int(nchan), int(nbin), int(device)
        self.freqs = None
        self.nmodel = 0
        self._pool = PinnedPool(self._lib)
        if stream is not None:
            self.set_stream(stream)

    def close(self):
        if getattr(self, "_pool", None) is not None:
            self._pool.close()
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.pp_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- configuration -------------------------------------------------------
    def set_stream(self, stream):
        """stream: torch.cuda.Stream, raw cudaStream_t int, or None."""
        h = getattr(stream, "cuda_stream", stream)
        _ffi.check(self._lib.pp_plan_set_stream(self._h, C.c_void_p(h or 0)),
                   "pp_plan_set_stream")

    def set_chunk(self, n):
        _ffi.check(self._lib.pp_plan_set_chunk(self._h, int(n)), "pp_plan_set_chunk")

    def set_fft_precision(self, bits):
        """0 = automatic, 32 = float FFT, 64 = double FFT (data rows)."""
        _ffi.check(self._lib.pp_plan_set_fft_precision(self._h, int(bits)),
                   "pp_plan_set_fft_precision")

    def set_model_steps(self, steps):
        """(phi, DM) solver: Newton steps per pass on the local fourth-order model (0 = default,
        1 = every step evaluated on the data)."""
        _ffi.check(self._lib.pp_plan_set_model_steps(self._h, int(steps)), "pp_plan_set_model_steps")

    def set_coarse(self, frac):
        """General solver: share of the model's phase information kept by the coarse (low-harmonic)
        objective its first iterations run on (default 0.99; 0 = no coarse stage)."""
        _ffi.check(self._lib.pp_plan_set_coarse(self._h, float(frac)), "pp_plan_set_coarse")

    def set_model_cutoff(self, eps):
        """Harmonics outside which a model channel holds less than eps^2 of its k^2-weighted power are
        neither computed, stored nor streamed (default 1e-10; 0 = keep every harmonic)."""
        _ffi.check(self._lib.pp_plan_set_model_cutoff(self._h, float(eps)), "pp_plan_set_model_cutoff")

    def set_freqs(self, freqs):
        keep = []
        fp = _ptr(np.asarray(freqs, dtype=np.float64), np.float64, keep, "freqs",
                  (self.nchan,))
        _ffi.check(self._lib.pp_set_freqs(self._h, fp), "pp_set_freqs")
        self.freqs = np.array(freqs, dtype=np.float64)

    def measure_fp64(self):
        """DFMA thread-instructions per second of an FP64-only kernel on this device (roofline yardstick)."""
        v = C.c_double(0.0)
        _ffi.check(self._lib.pp_measure_fp64(self._h, C.byref(v)), "pp_measure_fp64")
        return float(v.value)

    def enable_timing(self, on=True):
        _ffi.check(self._lib.pp_plan_enable_timing(self._h, 1 if on else 0),
                   "pp_plan_enable_timing")

    def stats(self):
        st = _ffi.Stats()
        _ffi.check(self._lib.pp_get_stats(self._h, C.byref(st)), "pp_get_stats")
        return {n: getattr(st, n) for n, _ in st._fields_}

    def set_model(self, model, freqs):
        """Model portrait [nchan, nbin] (numpy array or torch tensor, host or CUDA).  float64 models go to the
        device as they are (pp_set_model_f64: no float32 rounding floor in the model spectrum, which the
        harmonic cut-off needs to be effective); anything else is taken as float32."""
        self._set_models(1, model, freqs, (self.nchan, self.nbin), (self.nchan,))

    def set_models(self, models, freqs):
        """nmodel model portraits [nmodel, nchan, nbin] and their frequency tables [nmodel, nchan] MHz
        (pp_set_models; dtypes as set_model).  fit_batch(..., model_index) then fits subint s against model
        model_index[s].  Each model costs model_bytes(nchan, nbin) of device memory."""
        nmodel = int(models.shape[0])
        self._set_models(nmodel, models, freqs, (nmodel, self.nchan, self.nbin), (nmodel, self.nchan))

    def _set_models(self, nmodel, models, freqs, mshape, fshape):
        keep = []
        fp = _ptr(freqs if _is_torch(freqs) else np.asarray(freqs, dtype=np.float64), np.float64, keep, "freqs",
                  fshape)
        is64 = (str(models.dtype).endswith("float64")) if hasattr(models, "dtype") else False
        if is64:
            mp = _ptr(models, np.float64, keep, "model", mshape)
            _ffi.check(self._lib.pp_set_models_f64(self._h, nmodel, mp, fp), "pp_set_model_f64")
        else:
            mp = _ptr(models, np.float32, keep, "model", mshape)
            _ffi.check(self._lib.pp_set_models(self._h, nmodel, mp, fp), "pp_set_model")
        f = freqs.detach().cpu().numpy() if _is_torch(freqs) else freqs
        # the table of the rotation, alignment and model-generation calls: model 0's
        self.freqs = np.array(f, dtype=np.float64).reshape(-1, self.nchan)[0]
        self.nmodel = nmodel

    # ---- batched wideband fit ---------------------------------------------------
    def fit_batch(self, data, P, errs=None, chan_mask=None, weights=None,
                  init=None, DM_guess=None, snrs=None, nu_fits=None,
                  nu_fit_mode=0, nu_outs=None, fit_flags=(1, 1, 0, 0, 0),
                  log10_tau=False, option=0, is_toa=True, Ns=100, max_iter=0,
                  tol=0.0, semantics="full", want_chan_sums=False, nsub=None,
                  pinned_results=False, scat_guess=None, align=False, dat_scl=None, dat_offs=None,
                  bounds=None, model_index=None):
        """Fit every subint of data[nsub, nchan, nbin] (float32, host numpy or
        CUDA torch tensor).  Returns a dict of numpy arrays.

        model_index: [nsub] int32 (numpy or torch, host or CUDA) after set_models: subint s is fit against
        model model_index[s] and its frequency table.  None: the plan's one model.

        bounds: up to five (lower, upper) pairs for phi, DM, GM, tau (log10 tau with
        log10_tau) and alpha as scipy's TNC takes them (None = unbounded).

        pinned_results=True returns views of plan-owned page-locked buffers
        (full-speed D2H); they are overwritten by the next call on this plan and freed with it
        (copy what must outlive the plan)."""
        keep = []
        if nsub is None:
            nsub = int(data.shape[0]) if hasattr(data, "shape") and len(data.shape) == 3 else 1
        nchan, nbin = self.nchan, self.nbin
        a = _ffi.FitArgs()
        is_i16 = (data.dtype == np.int16) if isinstance(data, np.ndarray) else \
            (_is_torch(data) and str(data.dtype) == "torch.int16")
        if is_i16:
            # PSRFITS DATA column as stored: value = raw * DAT_SCL + DAT_OFFS per (subint, channel)
            if dat_scl is None or dat_offs is None:
                raise ValueError("int16 data need dat_scl and dat_offs [nsub, nchan]")
            a.data = _ptr(data, np.int16, keep, "data", (nsub, nchan, nbin))
            a.data_type = 1
            a.dat_scl = _ptr(dat_scl, np.float32, keep, "dat_scl", (nsub, nchan))
            a.dat_offs = _ptr(dat_offs, np.float32, keep, "dat_offs", (nsub, nchan))
        elif (isinstance(data, np.ndarray) and data.dtype == np.float64) or \
                (_is_torch(data) and str(data.dtype) == "torch.float64"):
            # the reference's array type: rounded to float32 on the device (PP_DATA_F64), no host pass
            a.data = _ptr(data, np.float64, keep, "data", (nsub, nchan, nbin))
            a.data_type = 2
        else:
            a.data = _ptr(data, np.float32, keep, "data", (nsub, nchan, nbin))
        a.nsub = nsub
        a.semantics = {"full": 0, "fit_portrait": 1}[semantics]
        Parr = np.broadcast_to(np.asarray(P, dtype=np.float64), (nsub,)) \
            if not _is_torch(P) else P
        a.P = _ptr(Parr, np.float64, keep, "P", (nsub,))
        a.errs = _ptr(errs, np.float64, keep, "errs", (nsub, nchan))
        a.chan_mask = _ptr(chan_mask, np.uint8, keep, "chan_mask", (nsub, nchan))
        a.weights = _ptr(weights, np.float64, keep, "weights", (nsub, nchan))
        a.init = _ptr(init, np.float64, keep, "init", (nsub, 5))
        a.DM_guess = _ptr(None if DM_guess is None else
                          (DM_guess if _is_torch(DM_guess) else
                           np.broadcast_to(np.asarray(DM_guess, dtype=np.float64), (nsub,))),
                          np.float64, keep, "DM_guess", (nsub,))
        a.snrs = _ptr(snrs, np.float64, keep, "snrs", (nsub, nchan))
        a.nu_fits = _ptr(nu_fits, np.float64, keep, "nu_fits", (nsub, 3))
        a.nu_fit_mode = int(nu_fit_mode)
        a.nu_outs = _ptr(nu_outs, np.float64, keep, "nu_outs", (nsub, 3))
        for i in range(5):
            a.fit_flags[i] = 1 if fit_flags[i] else 0
        a.log10_tau = 1 if log10_tau else 0
        a.option = int(option)
        a.is_toa = 1 if is_toa else 0
        a.Ns = int(Ns)
        a.max_iter = int(max_iter)
        a.tol = float(tol)
        a.scat_guess = _ptr(scat_guess, np.float64, keep, "scat_guess", (nsub, 2))
        a.bounds = _ptr(bounds_array(bounds), np.float64, keep, "bounds", (5, 2))
        mi = _ptr(model_index, np.int32, keep, "model_index", (nsub,))

        spec = {
            "params": ((nsub, 5), np.float64), "param_errs": ((nsub, 5), np.float64),
            "nu_out": ((nsub, 3), np.float64), "cov": ((nsub, 5, 5), np.float64),
            "chi2": ((nsub,), np.float64), "red_chi2": ((nsub,), np.float64),
            "snr": ((nsub,), np.float64), "nfeval": ((nsub,), np.int32),
            "return_code": ((nsub,), np.int32),
            "scales": ((nsub, nchan), np.float64), "scale_errs": ((nsub, nchan), np.float64),
            "channel_snrs": ((nsub, nchan), np.float64), "noise": ((nsub, nchan), np.float64),
            "lag_index": ((nsub,), np.int32), "phi_guess": ((nsub,), np.float64),
        }
        if want_chan_sums:
            spec["chan_sums"] = ((nsub, nchan, 9), np.float64)
        if align:   # fused ppalign accumulation (ppalign.py:197-213): sum_s w rotate(data) and sum_s w
            spec["align_sum"] = ((nchan, nbin), np.float64)
            spec["align_wsum"] = ((nchan,), np.float64)
        if pinned_results:
            res = {k: self._pool.array(k, sh, dt) for k, (sh, dt) in spec.items()}
        else:
            res = {k: np.empty(sh, dtype=dt) for k, (sh, dt) in spec.items()}
        o = _ffi.FitOut()
        for k, v in res.items():
            setattr(o, k, v.ctypes.data)
        _ffi.check(self._lib.pp_fit_batch_models(self._h, C.byref(a), mi, C.byref(o)),
                   "pp_fit_batch")
        del keep
        return res

    # ---- evolving-Gaussian model fit ----------------------------------------------------
    def fit_gaussian_portraits(self, data, errs, model_code, init, fit_flags, nu_ref, bounds=None,
                               max_iter=0, tol=0, want_model=False, want_sums=False):
        """Fit evolving-Gaussian portraits (pplib.py:1924-2052) to ``data`` [nport, nchan, nbin] float64
        with per-channel sigma ``errs`` [nport, nchan], on the plan's frequencies (set_freqs first).
        ``init`` [nport, P] and ``fit_flags`` [P] use the layout [DC, tau [bin], (loc, m_loc, wid, m_wid,
        amp, m_amp) * ngauss, alpha], P = 3 + 6 ngauss; ``bounds`` [P, 2] with NaN (or None) for open
        ends.  ``max_iter`` < 0 evaluates chi2, J^T r and J^T J at the start point only (0: default 200);
        ``tol`` 0 = 1e-4.  numpy arrays or CUDA tensors.  Returns a dict of numpy arrays: params,
        param_errs, cov, chi2, red_chi2, dof, nfeval, return_code, and with ``want_model`` the model
        portraits [nport, nchan, nbin], with ``want_sums`` jtr [nport, P] and jtj [nport, P, P]."""
        fit_flags = np.ascontiguousarray(np.asarray(fit_flags) != 0, dtype=np.uint8).ravel()
        P = fit_flags.size
        if P < 9 or (P - 3) % 6:
            raise ValueError("fit_flags must have 3 + 6*ngauss entries")
        ngauss = (P - 3) // 6
        nport = int(data.shape[0])
        nchan, nbin = self.nchan, self.nbin
        keep = []
        a = _ffi.GfitArgs()
        a.nport = nport
        a.data = _ptr(data, np.float64, keep, "data", (nport, nchan, nbin))
        a.errs = _ptr(errs, np.float64, keep, "errs", (nport, nchan))
        a.model_code = str(model_code).encode("ascii")
        a.ngauss = ngauss
        a.nu_ref = float(nu_ref)
        a.init = _ptr(init, np.float64, keep, "init", (nport, P))
        a.fit_flags = fit_flags.ctypes.data
        if bounds is not None:
            b = np.array([[np.nan if v is None else v for v in pair] for pair in bounds], dtype=np.float64)
            if b.shape != (P, 2):
                raise ValueError("bounds must be [P, 2]")
            a.bounds = _ptr(b, np.float64, keep, "bounds")
        a.max_iter = int(max_iter)
        a.tol = float(tol)
        spec = {"params": ((nport, P), np.float64), "param_errs": ((nport, P), np.float64),
                "cov": ((nport, P, P), np.float64), "chi2": ((nport,), np.float64),
                "red_chi2": ((nport,), np.float64), "nfeval": ((nport,), np.int32),
                "return_code": ((nport,), np.int32)}
        if want_model:
            spec["model"] = ((nport, nchan, nbin), np.float64)
        if want_sums:
            spec["jtr"] = ((nport, P), np.float64)
            spec["jtj"] = ((nport, P, P), np.float64)
        res = {k: np.empty(sh, dtype=dt) for k, (sh, dt) in spec.items()}
        o = _ffi.GfitOut()
        for k, v in res.items():
            setattr(o, k, v.ctypes.data)
        _ffi.check(self._lib.pp_fit_gaussian_portraits(self._h, C.byref(a), C.byref(o)),
                   "pp_fit_gaussian_portraits")
        del keep
        res["dof"] = np.full(nport, nchan * nbin - int(fit_flags.sum()), dtype=np.int64)
        return res

    # ---- batched 1-D FFTFIT --------------------------------------------------------
    def fit_phase_shift_batch(self, profiles, models, noise=None, Ns=100, bounds=(-0.5, 0.5)):
        """Batched pplib.fit_phase_shift; ``bounds`` = ends of the brute-force grid (pplib.py:2085)."""
        keep = []
        n = int(profiles.shape[0])
        nmodel = int(models.shape[0]) if len(models.shape) == 2 else 1
        pp = _ptr(profiles, np.float32, keep, "profiles", (n, self.nbin))
        mp = _ptr(models, np.float32, keep, "models", (nmodel, self.nbin))
        nz = _ptr(noise, np.float64, keep, "noise", (n,))
        res = {k: np.empty(n) for k in ("phase", "phase_err", "scale",
                                        "scale_err", "snr", "red_chi2")}
        res["lag_index"] = np.empty(n, dtype=np.int32)
        o = _ffi.PShiftOut()
        for k, v in res.items():
            setattr(o, k, v.ctypes.data)
        _ffi.check(self._lib.pp_fit_phase_shift_batch_bounds(self._h, pp, n, mp, nmodel, nz, int(Ns),
                                                             float(bounds[0]), float(bounds[1]), C.byref(o)),
                   "pp_fit_phase_shift_batch_bounds")
        return res

    # ---- batched rotation -------------------------------------------------------------
    def align_accumulate(self, data, phase, DM, P, nu_ref, weights):
        """sum_s weights[s,n] * rotate(data[s,n], phase_s, DM_s) (ppalign.py:202-208).
        Returns (aligned[nchan,nbin] float64 un-normalised, wsum[nchan])."""
        keep = []
        nsub = int(data.shape[0])
        ip = _ptr(data, np.float32, keep, "data", (nsub, self.nchan, self.nbin))
        bc = lambda v: np.broadcast_to(np.asarray(v, dtype=np.float64), (nsub,))  # noqa: E731
        aligned = np.empty((self.nchan, self.nbin))
        wsum = np.empty(self.nchan)
        _ffi.check(self._lib.pp_align_accumulate(
            self._h, ip, nsub, _ptr(bc(phase), np.float64, keep, "phase"),
            _ptr(bc(DM), np.float64, keep, "DM"), _ptr(bc(P), np.float64, keep, "P"),
            _ptr(bc(nu_ref), np.float64, keep, "nu_ref"),
            _ptr(weights, np.float64, keep, "weights", (nsub, self.nchan)),
            aligned.ctypes.data, wsum.ctypes.data), "pp_align_accumulate")
        return aligned, wsum

    def get_noise_fit_batch(self, data, fact=1.1):
        """get_noise_fit(chans=True) per row (pplib.py:2255-2284; the find_kc grid search runs on the device)."""
        keep = []
        nsub = int(data.shape[0])
        ip = _ptr(data, np.float32, keep, "data", (nsub, self.nchan, self.nbin))
        out = np.empty((nsub, self.nchan))
        _ffi.check(self._lib.pp_get_noise_fit_batch(self._h, ip, nsub, float(fact), out.ctypes.data),
                   "pp_get_noise_fit_batch")
        return out

    def gen_gaussian_portrait(self, model_code, params, scattering_index, nu_ref, out=None, device_out=False,
                              dtype=np.float32):
        """Evolving-Gaussian model portrait on the device (pplib.py:853-930) for the plan's
        frequencies (set_freqs first).  ``params`` = [DC, tau_bin, (loc, m_loc, wid, m_wid, amp,
        m_amp) * ngauss].  Returns [nchan, nbin] of ``dtype`` (float32, or float64: evaluated and stored in
        double): a numpy array, or a torch CUDA tensor with ``device_out=True`` (ready for set_model without a
        host round trip)."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.ndim != 1 or (params.size - 2) % 6:
            raise ValueError("params must have 2 + 6*ngauss entries")
        ngauss = (params.size - 2) // 6
        f64 = np.dtype(dtype) == np.float64
        if out is None:
            if device_out:
                import torch
                out = torch.empty((self.nchan, self.nbin), dtype=torch.float64 if f64 else torch.float32,
                                  device=torch.device("cuda", self.device))
            else:
                out = np.empty((self.nchan, self.nbin), dtype=np.float64 if f64 else np.float32)
        else:
            f64 = str(out.dtype).endswith("float64")
        op = out.data_ptr() if _is_torch(out) else out.ctypes.data
        fn = self._lib.pp_gen_gaussian_portrait_f64 if f64 else self._lib.pp_gen_gaussian_portrait
        _ffi.check(fn(self._h, str(model_code).encode("ascii"), params.ctypes.data, int(ngauss),
                      float(scattering_index), float(nu_ref), op), "pp_gen_gaussian_portrait")
        return out

    def gen_spline_portrait(self, mean_prof, eigvec, tck, out=None, device_out=False):
        """B-spline (PCA) model portrait on the device (pplib.py:932-956) for the plan's
        frequencies.  ``tck`` = (knots, [coefficient arrays], degree) as returned by
        scipy.interpolate.splprep; eigvec is [nbin, ncomp].  Returns float32 [nchan, nbin]."""
        mean_prof = np.ascontiguousarray(mean_prof, dtype=np.float64)
        eigvec = np.ascontiguousarray(eigvec, dtype=np.float64).reshape(len(mean_prof), -1)
        if mean_prof.shape != (self.nbin,):
            raise ValueError("the spline model has %d bins, the plan %d (resampling is not provided)"
                             % (len(mean_prof), self.nbin))
        ncomp = eigvec.shape[1]
        knots = np.ascontiguousarray(tck[0], dtype=np.float64)
        degree = int(tck[2])
        ncoef = len(knots) - degree - 1
        coefs = np.ascontiguousarray([np.asarray(c, dtype=np.float64)[:ncoef] for c in tck[1]],
                                     dtype=np.float64).reshape(ncomp, ncoef) if ncomp else np.zeros((0, 0))
        if out is None:
            if device_out:
                import torch
                out = torch.empty((self.nchan, self.nbin), dtype=torch.float32,
                                  device=torch.device("cuda", self.device))
            else:
                out = np.empty((self.nchan, self.nbin), dtype=np.float32)
        op = out.data_ptr() if _is_torch(out) else out.ctypes.data
        _ffi.check(self._lib.pp_gen_spline_portrait(
            self._h, mean_prof.ctypes.data, eigvec.ctypes.data if ncomp else None, int(ncomp),
            knots.ctypes.data if ncomp else None, int(len(knots)), coefs.ctypes.data if ncomp else None,
            degree, op), "pp_gen_spline_portrait")
        return out

    def pca_moments(self, port, weights, gram=False):
        """Weighted mean profile mu [nbin] and second-moment matrix of d_n = sqrt(w_n) (x_n - mu), normalised by
        sum(w): the covariance [nbin, nbin], or with ``gram`` the Gram matrix [nchan, nchan] (pp_pca_moments).
        ``port`` [nchan, nbin] and ``weights`` [nchan] (>= 0, 0 = excluded) are float64 numpy arrays or CUDA
        tensors."""
        keep = []
        if not _is_torch(weights) and np.any(np.asarray(weights, dtype=np.float64) < 0):
            raise ValueError("weights must be >= 0")
        dim = self.nchan if gram else self.nbin
        mean = np.empty(self.nbin)
        mat = np.empty((dim, dim))
        _ffi.check(self._lib.pp_pca_moments(
            self._h, _ptr(port, np.float64, keep, "port", (self.nchan, self.nbin)),
            _ptr(weights, np.float64, keep, "weights", (self.nchan,)), int(bool(gram)),
            mean.ctypes.data, mat.ctypes.data), "pp_pca_moments")
        return mean, mat

    def pca_backproject(self, port, weights, mean, U):
        """Unit basis vectors e_j = D^T u_j / ||D^T u_j|| [nbin, m] from Gram eigenvectors U [nchan, m], with
        d_n = sqrt(w_n) (x_n - mean); each with its entry of largest |value| positive (pp_pca_project)."""
        keep = []
        m = int(U.shape[1])
        out = np.empty((self.nbin, m))
        _ffi.check(self._lib.pp_pca_project(
            self._h, _ptr(port, np.float64, keep, "port", (self.nchan, self.nbin)),
            _ptr(weights, np.float64, keep, "weights", (self.nchan,)),
            _ptr(mean, np.float64, keep, "mean", (self.nbin,)), _ptr(U, np.float64, keep, "U", (self.nchan, m)),
            m, 1, out.ctypes.data), "pp_pca_project")
        return out

    def pca_project(self, port, mean, E):
        """Projections P [nchan, m] of x_n - mean onto the columns of E [nbin, m] (pp_pca_project)."""
        keep = []
        m = int(E.shape[1])
        out = np.empty((self.nchan, m))
        _ffi.check(self._lib.pp_pca_project(
            self._h, _ptr(port, np.float64, keep, "port", (self.nchan, self.nbin)), None,
            _ptr(mean, np.float64, keep, "mean", (self.nbin,)), _ptr(E, np.float64, keep, "E", (self.nbin, m)),
            m, 0, out.ctypes.data), "pp_pca_project")
        return out

    def lowpass_rows(self, rows):
        """Low-pass float64 rows [nrows, nbin]: rfft, k_c from find_kc (get_noise_fit's rule, fact = 1), harmonics
        above k_c zeroed (DC kept, Nyquist only when k_c reaches it), irfft (pp_lowpass_rows).  Returns (smoothed
        rows [nrows, nbin], kc [nrows] int32)."""
        keep = []
        nrows = int(rows.shape[0])
        out = np.empty((nrows, self.nbin))
        kc = np.empty(nrows, dtype=np.int32)
        _ffi.check(self._lib.pp_lowpass_rows(
            self._h, _ptr(rows, np.float64, keep, "rows", (nrows, self.nbin)), nrows, out.ctypes.data,
            kc.ctypes.data), "pp_lowpass_rows")
        return out, kc

    def rotate_batch(self, data, phase, DM, P, nu_ref, out=None, GM=None, nu_GM=None):
        if GM is not None:
            return self._rotate_full(data, phase, DM, GM, P, nu_ref, nu_GM, out)
        keep = []
        nsub = int(data.shape[0])
        ip = _ptr(data, np.float32, keep, "data", (nsub, self.nchan, self.nbin))
        if out is None:
            if _is_torch(data):
                import torch
                out = torch.empty_like(data)
            else:
                out = np.empty((nsub, self.nchan, self.nbin), dtype=np.float32)
        op = out.data_ptr() if _is_torch(out) else out.ctypes.data
        bc = lambda v: np.broadcast_to(np.asarray(v, dtype=np.float64), (nsub,))  # noqa: E731
        _ffi.check(self._lib.pp_rotate_batch(
            self._h, ip, op, nsub,
            _ptr(bc(phase), np.float64, keep, "phase"),
            _ptr(bc(DM), np.float64, keep, "DM"),
            _ptr(bc(P), np.float64, keep, "P"),
            _ptr(bc(nu_ref), np.float64, keep, "nu_ref")), "pp_rotate_batch")
        return out

    def apply_response_batch(self, data, resp, out=None):
        """out[s, n] = irfft(resp[n] * rfft(data[s, n])): a real per-channel, per-harmonic response
        [nchan, nbin/2 + 1] applied in the Fourier domain (pp_apply_response_batch; the model
        multiply of pptoas.py:388-394)."""
        keep = []
        nsub = int(data.shape[0])
        ip = _ptr(data, np.float32, keep, "data", (nsub, self.nchan, self.nbin))
        if out is None:
            if _is_torch(data):
                import torch
                out = torch.empty_like(data)
            else:
                out = np.empty((nsub, self.nchan, self.nbin), dtype=np.float32)
        op = out.data_ptr() if _is_torch(out) else out.ctypes.data
        _ffi.check(self._lib.pp_apply_response_batch(
            self._h, ip, op, nsub,
            _ptr(resp, np.float64, keep, "resp", (self.nchan, self.nbin // 2 + 1))), "pp_apply_response_batch")
        return out

    def _rotate_full(self, data, phase, DM, GM, P, nu_DM, nu_GM, out=None):
        keep = []
        nsub = int(data.shape[0])
        ip = _ptr(data, np.float32, keep, "data", (nsub, self.nchan, self.nbin))
        if out is None:
            if _is_torch(data):
                import torch
                out = torch.empty_like(data)
            else:
                out = np.empty((nsub, self.nchan, self.nbin), dtype=np.float32)
        op = out.data_ptr() if _is_torch(out) else out.ctypes.data
        bc = lambda v: np.broadcast_to(np.asarray(v, dtype=np.float64), (nsub,))  # noqa: E731
        _ffi.check(self._lib.pp_rotate_full_batch(
            self._h, ip, op, nsub, _ptr(bc(phase), np.float64, keep, "phase"),
            _ptr(bc(DM), np.float64, keep, "DM"), _ptr(bc(GM), np.float64, keep, "GM"),
            _ptr(bc(P), np.float64, keep, "P"), _ptr(bc(nu_DM), np.float64, keep, "nu_DM"),
            _ptr(bc(nu_GM), np.float64, keep, "nu_GM")), "pp_rotate_full_batch")
        return out

    # ---- simulated archives -------------------------------------------------------------
    def simulate_batch(self, models, freqs, phase, DM, P, nu_DM=np.inf, GM=None, nu_GM=None, tau=None,
                       alpha=None, nu_tau=None, scales=None, noise_stds=None, seed=0, first_subint=0,
                       model_index=None, quantize=False, out=None, device_out=False):
        """Simulated subints (pp_simulate_batch): row (s, n) is the model portrait model_index[s] rotated by the
        injected phase, DM (about nu_DM) and GM (about nu_GM, default inf), scattered by tau [rot at nu_tau] with
        index alpha (default -4), times scales, plus noise_stds * N(0, 1) from the counter-based generator keyed by
        ``seed`` (subint s draws as global subint first_subint + s, whatever the batch).  fit_batch recovers the
        injected parameters.

        models: float64 [nchan, nbin] or [nmodel, nchan, nbin] with freqs [nchan] or [nmodel, nchan] (numpy or
        torch, host or CUDA).  phase, DM, P, nu_DM, GM, nu_GM, tau, alpha, nu_tau: scalars or [nsub]; scales,
        noise_stds: scalars, [nchan] or [nsub, nchan] (None: 1 and 0).  nsub is the longest of these (1 when all
        are scalars), or out's.

        Returns float32 [nsub, nchan, nbin], or with ``quantize`` (raw int16 [nsub, nchan, nbin], dat_scl,
        dat_offs float32 [nsub, nchan]) = pptoas.quantize_subints of the float32 rows: numpy arrays, or torch
        CUDA tensors with ``device_out`` (which fit_batch takes as they are).  ``out`` (an array, or the
        (raw, dat_scl, dat_offs) tuple) receives the result instead."""
        nchan, nbin = self.nchan, self.nbin
        keep = []
        mshape = tuple(models.shape)
        nmodel = 1 if len(mshape) == 2 else int(mshape[0])
        if mshape[-2:] != (nchan, nbin) or len(mshape) not in (2, 3):
            raise ValueError("models must be [nchan, nbin] or [nmodel, nchan, nbin] with (nchan, nbin) = (%d, %d)"
                             % (nchan, nbin))
        if GM is not None and nu_GM is None:
            nu_GM = np.inf
        if tau is not None:
            if nu_tau is None:
                raise ValueError("tau needs nu_tau, the frequency it refers to")
            if alpha is None:
                alpha = -4.0
        elif alpha is not None or nu_tau is not None:
            raise ValueError("alpha and nu_tau describe tau: give tau too")
        per_sub = dict(phase=phase, DM=DM, P=P, nu_DM=nu_DM, GM=GM, nu_GM=nu_GM, tau=tau, alpha=alpha, nu_tau=nu_tau)
        lens = [int(np.shape(v)[0]) for v in list(per_sub.values()) + [model_index] if v is not None and np.ndim(v) >= 1]
        lens += [int(np.shape(v)[0]) for v in (scales, noise_stds) if v is not None and np.ndim(v) == 2]
        if out is not None:
            lens.append(int(np.shape(out[0] if quantize else out)[0]))
        nsub = max(lens) if lens else 1

        def sub(v, name):
            if v is None:
                return None
            if _is_torch(v):
                return _ptr(v, np.float64, keep, name, (nsub,))
            return _ptr(np.broadcast_to(np.asarray(v, dtype=np.float64), (nsub,)), np.float64, keep, name)

        def chan(v, name):
            if v is None:
                return None
            if _is_torch(v):
                return _ptr(v, np.float64, keep, name, (nsub, nchan))
            return _ptr(np.broadcast_to(np.asarray(v, dtype=np.float64), (nsub, nchan)), np.float64, keep, name)

        a = _ffi.SimArgs()
        a.models = _ptr(models, np.float64, keep, "models", (nmodel, nchan, nbin))
        a.freqs = _ptr(freqs if _is_torch(freqs) else np.asarray(freqs, dtype=np.float64), np.float64, keep,
                       "freqs", (nmodel, nchan))
        a.nmodel = nmodel
        a.model_index = _ptr(model_index, np.int32, keep, "model_index", (nsub,))
        a.nsub = nsub
        a.first_subint = int(first_subint)
        a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        for k, v in per_sub.items():
            setattr(a, k, sub(v, k))
        a.scales = chan(scales, "scales")
        a.noise_std = chan(noise_stds, "noise_stds")
        if out is None:
            shapes = [((nsub, nchan, nbin), np.int16), ((nsub, nchan), np.float32), ((nsub, nchan), np.float32)] \
                if quantize else [((nsub, nchan, nbin), np.float32)]
            if device_out:
                import torch
                tdt = {np.int16: torch.int16, np.float32: torch.float32}
                res = [torch.empty(sh, dtype=tdt[dt], device=torch.device("cuda", self.device)) for sh, dt in shapes]
            else:
                res = [np.empty(sh, dtype=dt) for sh, dt in shapes]
        else:
            res = list(out) if quantize else [out]
        o = _ffi.SimOut()
        if quantize:
            o.raw = _ptr(res[0], np.int16, keep, "raw", (nsub, nchan, nbin))
            o.dat_scl = _ptr(res[1], np.float32, keep, "dat_scl", (nsub, nchan))
            o.dat_offs = _ptr(res[2], np.float32, keep, "dat_offs", (nsub, nchan))
        else:
            o.data = _ptr(res[0], np.float32, keep, "out", (nsub, nchan, nbin))
        for r in res:
            if isinstance(r, np.ndarray) and not (r.flags.c_contiguous and r.flags.writeable):
                raise ValueError("outputs must be writeable C-contiguous arrays")
        _ffi.check(self._lib.pp_simulate_batch(self._h, C.byref(a), C.byref(o)), "pp_simulate_batch")
        del keep
        return tuple(res) if quantize else res[0]

    def get_noise_batch(self, data, kc=-1):
        """Per-row noise level from the harmonics k >= kc (default int(0.75 nharm), pplib.py:2244)."""
        keep = []
        nsub = int(data.shape[0])
        ip = _ptr(data, np.float32, keep, "data", (nsub, self.nchan, self.nbin))
        out = np.empty((nsub, self.nchan))
        _ffi.check(self._lib.pp_get_noise_cut_batch(self._h, ip, nsub, int(kc), out.ctypes.data),
                   "pp_get_noise_cut_batch")
        return out
