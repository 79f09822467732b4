"""Reference-compatible facade for the hot-path functions of ``pplib``.

Same names, argument meaning, units and return fields as the reference
(pennucci/PulsePortraiture ``pplib.py``; line numbers cited per function), but
the arithmetic runs in the sm_100a CUDA library behind the C ABI
(``include/ppb200.h``).  Inputs are converted to float32 on entry (the device
storage type); parameters and accumulators are float64.

Not accelerated (plain host helpers kept so that scripts run): model
generation from ``.gmodel`` files and scalar reference-frequency transforms.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np

from .engine import WidebandPlan

# ---- settings (pplib.py:44-83) ---------------------------------------------
Dconst_exact = 4.148808e3
Dconst_trad = 0.000241 ** -1
Dconst = Dconst_trad
scattering_alpha = -4.0
use_get_noise = True
default_noise_method = "PS"
F0_fact = 0
wid_max = 0.25
default_model = "000"
binshift = 1.0

# Return codes.  The device solver reports 0 converged / 1 pass limit / 3 non-finite objective
# (DEVICE_RCSTRINGS).  The facades hand callers the scipy status the reference's minimiser would
# have returned for the same outcome (pplib.py:2159-2171, pptoaslib.py:1018-1033: callers treat
# TNC's {1, 2, 4} and trust-ncg's 2 as the normal exits), with the messages of pplib.py:111-119;
# the device's own code stays available as the extra DataBunch field ``device_return_code``.
DEVICE_RCSTRINGS = {"0": "CONVERGED: Newton step below tolerance.",
                    "1": "MAXITER: Maximum number of objective passes reached.",
                    "3": "NONFINITE: Objective is not finite."}
RCSTRINGS = {'-1': 'INFEASIBLE: Infeasible (low > up).',
             '0': 'LOCALMINIMUM: Local minima reach (|pg| ~= 0).',
             '1': 'FCONVERGED: Converged (|f_n-f_(n-1)| ~= 0.)',
             '2': 'XCONVERGED: Converged (|x_n-x_(n-1)| ~= 0.)',
             '3': 'MAXFUN: Max. number of function evaluations reach.',
             '4': 'LSFAIL: Linear search failed.',
             '5': 'CONSTANT: All lower bounds are equal to the upper bounds.',
             '6': 'NOPROGRESS: Unable to progress.',
             '7': 'USERABORT: User requested end of minimization.'}
# device code -> scipy status, per minimiser
_RC_MAP = {'TNC': {0: 1, 1: 3, 3: 6},            # FCONVERGED / MAXFUN / NOPROGRESS
           'trust-ncg': {0: 2, 1: 1, 3: 3},      # "failure to predict improvement" is the normal exit
           'Newton-CG': {0: 0, 1: 1, 3: 3}}      # success / maxiter / NaN result encountered
_RC_BENIGN = {'TNC': (0, 1, 2, 4), 'trust-ncg': (0, 1, 2, 4), 'Newton-CG': (0, 1, 2, 4)}


def scipy_return_code(device_rc, method='TNC'):
    """The status scipy's ``method`` reports for the outcome the device solver reports as ``device_rc``
    (scalar or array)."""
    m = _RC_MAP[method]
    if np.ndim(device_rc) == 0:
        return m.get(int(device_rc), int(device_rc))
    return np.array([m.get(int(v), int(v)) for v in np.asarray(device_rc).ravel()],
                    dtype=int).reshape(np.shape(device_rc))


class DataBunch(dict):
    """dict with attribute access (pplib.py:125-136)."""

    def __init__(self, **kwds):
        dict.__init__(self, kwds)
        self.__dict__ = self


# ---- plan cache ---------------------------------------------------------------
_plans = {}
_device = 0


def set_device(device):
    """Select the CUDA device used by the single-portrait facade calls."""
    global _device
    _device = int(device)


def get_plan(nchan, nbin, device=None):
    device = _device if device is None else int(device)
    key = (int(nchan), int(nbin), device)
    pl = _plans.get(key)
    if pl is None:
        pl = WidebandPlan(nchan, nbin, device)
        _plans[key] = pl
    return pl


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _mdl(a):
    """A model portrait as set_model takes it: float32 arrays as they are, everything else as float64 (the
    reference's array type; no float32 rounding floor in the model spectrum)."""
    a = np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float32 if a.dtype == np.float32 else np.float64)


def _dev(a):
    """Portrait data as the device takes them without a host pass: float32 and float64 arrays go as
    they are (float64 is rounded to float32 on the device, PP_DATA_F64), anything else via float64."""
    a = np.asarray(a)
    if a.dtype not in (np.float32, np.float64):
        a = a.astype(np.float64)
    return np.ascontiguousarray(a)


def _check_bounds(bounds, nparam):
    """scipy-style bounds -> what WidebandPlan.fit_batch takes (None when nothing is bounded)."""
    bounds = list(bounds or [])
    if len(bounds) > nparam:
        raise ValueError("bounds has %d entries for %d parameters" % (len(bounds), nparam))
    for b in bounds:
        if b is not None and len(b) != 2:
            raise ValueError("each bound is a (lower, upper) pair")
    return bounds if any(b is not None and any(v is not None for v in b) for b in bounds) else None


# ---- A3: 1-D FFTFIT -------------------------------------------------------------
def fit_phase_shift(data, model, noise=None, bounds=[-0.5, 0.5], Ns=100):
    """Fit a phase shift between data and model (pplib.py:2054-2100).

    Returns DataBunch(phase, phase_err, scale, scale_err, snr, red_chi2,
    duration).  The brute-force grid (Ns points on ``bounds``, both ends) is
    evaluated on the device; ``phase`` is the exact minimiser reached from the
    grid argmin (the reference's Nelder-Mead polish is accurate to ~1e-4 rot).
    The integer argmin is returned as the extra field ``lag_index``.
    """
    data = np.asarray(data)
    if len(bounds) != 2 or not bounds[1] > bounds[0]:
        raise ValueError("bounds = [lower, upper]")
    nbin = data.shape[-1]
    pl = get_plan(1, nbin)
    start = time.time()
    r = pl.fit_phase_shift_batch(_f32(data).reshape(1, nbin),
                                 _f32(model).reshape(1, nbin),
                                 None if noise is None else np.array([noise], dtype=np.float64),
                                 Ns=Ns, bounds=bounds)
    duration = time.time() - start
    return DataBunch(phase=r["phase"][0], phase_err=r["phase_err"][0],
                     scale=r["scale"][0], scale_err=r["scale_err"][0],
                     snr=r["snr"][0], red_chi2=r["red_chi2"][0],
                     duration=duration, lag_index=int(r["lag_index"][0]))


# ---- A1: phi + DM fit --------------------------------------------------------------
def fit_portrait(data, model, init_params, P, freqs, nu_fit=None, nu_out=None,
                 errs=None, bounds=[(None, None), (None, None)], id=None,
                 quiet=True):
    """Fit a phase offset and DM between data and model portraits
    (pplib.py:2102-2204).  Same arguments and DataBunch fields as the
    reference; the TNC minimiser is replaced by the on-device Newton solver
    (``return_code`` 0 = converged, 1 = max passes, 3 = non-finite), which
    honours ``bounds`` as an active set."""
    bounds = _check_bounds(bounds, 2)
    data = np.asarray(data)
    nchan, nbin = data.shape
    freqs = np.asarray(freqs, dtype=np.float64)
    pl = get_plan(nchan, nbin)
    pl.set_model(_mdl(model), freqs)
    init = np.zeros((1, 5))
    init[0, 0], init[0, 1] = init_params[0], init_params[1]
    nu_fits = None if nu_fit is None else np.full((1, 3), float(nu_fit))
    nu_outs = None if nu_out is None else np.full((1, 3), float(nu_out))
    start = time.time()
    r = pl.fit_batch(_dev(data)[None], P,
                     errs=None if errs is None else np.asarray(errs, dtype=np.float64)[None],
                     init=init, nu_fits=nu_fits, nu_outs=nu_outs,
                     fit_flags=(1, 1, 0, 0, 0), semantics="fit_portrait", bounds=bounds)
    duration = time.time() - start
    drc = int(r["return_code"][0])
    rc = scipy_return_code(drc, 'TNC')
    if not quiet and rc not in _RC_BENIGN['TNC']:
        if id is not None:
            ii = id[::-1].index("_")
            isub, filename = id[-ii:], id[:-ii - 1]
            sys.stderr.write("Fit failed with return code %d: %s -- %s subint %s\n"
                             % (rc, RCSTRINGS[str(rc)], filename, isub))
        else:
            sys.stderr.write("Fit failed with return code %d -- %s" % (rc, RCSTRINGS[str(rc)]))
    return DataBunch(phase=r["params"][0, 0], phase_err=r["param_errs"][0, 0],
                     DM=r["params"][0, 1], DM_err=r["param_errs"][0, 1],
                     scales=r["scales"][0], scale_errs=r["scale_errs"][0],
                     nu_ref=r["nu_out"][0, 0], covariance=r["cov"][0, 0, 1],
                     chi2=r["chi2"][0], red_chi2=r["red_chi2"][0],
                     snr=r["snr"][0], duration=duration,
                     nfeval=int(r["nfeval"][0]), return_code=rc, device_return_code=drc)


def get_scales(data, model, phase, DM, P, freqs, nu_ref=np.inf):
    """Best-fit per-channel amplitudes at given (phase, DM) (pplib.py:2310-2336)."""
    data = np.asarray(data)
    nchan, nbin = data.shape
    pl = get_plan(nchan, nbin)
    pl.set_model(_mdl(model), np.asarray(freqs, dtype=np.float64))
    init = np.zeros((1, 5))
    init[0, 0], init[0, 1] = phase, DM
    nu = 1e300 if np.isinf(nu_ref) else float(nu_ref)
    r = pl.fit_batch(_f32(data)[None], P, init=init, nu_fits=np.full((1, 3), nu),
                     nu_outs=np.full((1, 3), nu), fit_flags=(1, 1, 0, 0, 0),
                     max_iter=-1, semantics="fit_portrait")
    return r["scales"][0]


# ---- A9: noise ------------------------------------------------------------------------
def get_noise(data, method=default_noise_method, **kwargs):
    """Off-pulse noise estimate (pplib.py:2206-2225): "PS" or "fit"."""
    if method == "PS":
        return get_noise_PS(data, **kwargs)
    if method == "fit":
        return get_noise_fit(data, **kwargs)
    print("Unknown get_noise method.")
    return 0


def _power_spectrum(data):
    """|rfft(data.ravel())|^2 / n in float64, on the facade's device.  The whole-portrait estimate is one
    row of nchan * nbin samples, longer than any row plan takes, so it is transformed as one float64 rfft."""
    import torch
    x = torch.as_tensor(np.ascontiguousarray(np.ravel(data), dtype=np.float64), device=torch.device("cuda", _device))
    X = torch.fft.rfft(x)
    return (X.real * X.real + X.imag * X.imag) / x.numel()


def _find_kc(pows):
    """find_kc (pplib.py:1465-1495) of a power spectrum on the device: chi2 of b exp(-a k) + dc against
    log10 pows at every point of scipy.optimize.brute's 20 x 20 x 20 np.mgrid, in chunks of grid points (C
    order, a slowest); np.argmin's order picks the point (a NaN chi2 wins, the first one; otherwise the
    lowest chi2, the lowest index on ties); the first k with exp(-a k) < 0.005, or nharm - 1."""
    import torch
    y = torch.log10(pows)
    nh = y.numel()
    lo, hi = float(y.min()), float(y.max())
    with np.errstate(invalid="ignore"):    # an exactly zero harmonic: lo = -inf, the grid is NaN
        grid = np.mgrid[nh ** -1.0:1.0:20j, 0:hi - lo:20j, lo:hi:20j].reshape(3, -1)
    g = torch.as_tensor(grid, device=pows.device)
    k = torch.arange(nh, dtype=torch.float64, device=pows.device)
    c2 = torch.empty(g.shape[1], dtype=torch.float64, device=pows.device)
    step = max(1, (1 << 24) // nh)          # grid points per chunk: at most 2^24 terms
    for i0 in range(0, g.shape[1], step):
        a, b, dc = g[:, i0:i0 + step, None]
        c2[i0:i0 + step] = ((y - (b * torch.exp(-a * k) + dc)) ** 2).sum(-1)
    nan = torch.isnan(c2)
    i = int(torch.nonzero(nan)[0, 0]) if bool(nan.any()) else int(torch.argmin(c2))
    hit = np.nonzero(np.exp(-grid[0, i] * np.arange(nh)) < 0.005)[0]
    return int(hit[0]) if len(hit) else nh - 1


def get_noise_fit(data, fact=1.1, chans=False):
    """Noise from the harmonics above fact * the cutoff a fit of b exp(-a k) + dc to the log power
    spectrum finds (pplib.py:2255-2284, find_kc 1465-1495).  chans=False: the whole of data as one row of
    any length (_power_spectrum, _find_kc)."""
    data = np.asarray(data)
    if chans:
        nchan, nbin = data.shape
        return get_plan(nchan, nbin).get_noise_fit_batch(_f32(data)[None], fact)[0]
    pows = _power_spectrum(data)
    k_crit = fact * _find_kc(pows)
    if k_crit >= pows.numel():
        k_crit = min(int(0.99 * pows.numel()), k_crit)
    return np.float64(pows[int(k_crit):].mean().sqrt().item())


def get_noise_PS(data, frac=4, chans=False):
    """Mean of the highest 1/frac of the power spectrum (pplib.py:2227-2253).  chans=False: the whole of
    data as one row of any length (_power_spectrum)."""
    data = np.asarray(data)
    if chans:
        nchan, nbin = data.shape
        kc = int((1 - frac ** -1) * (nbin // 2 + 1))         # pplib.py:2244
        return get_plan(nchan, nbin).get_noise_batch(_f32(data)[None], kc=kc)[0]
    pows = _power_spectrum(data)
    kc = int((1 - frac ** -1) * pows.numel())
    return np.float64(pows[kc:].mean().sqrt().item())


# ---- A10: rotation ----------------------------------------------------------------------
def rotate_data(data, phase=0.0, DM=0.0, Ps=None, freqs=None, nu_ref=np.inf):
    """Rotate and/or dedisperse a profile, portrait or [nsub,npol,nchan,nbin]
    cube in the Fourier domain (pplib.py:2338-2426).  Positive phase/DM rotate
    to earlier phase."""
    data = np.asarray(data)
    shape = data.shape
    nbin = shape[-1]
    nu = 1e300 if np.isinf(nu_ref) else float(nu_ref)
    if data.ndim == 1:
        cube = data.reshape(1, 1, nbin)
        f = np.array([1.0 if freqs is None else float(np.atleast_1d(freqs)[0])])
        Pv = 1.0 if Ps is None else Ps
    elif data.ndim == 2:
        cube = data.reshape(1, shape[0], nbin)
        f = np.ones(shape[0]) if freqs is None else np.asarray(freqs, dtype=np.float64)
        Pv = 1.0 if Ps is None else Ps
    elif data.ndim == 4:
        nsub, npol, nchan, _ = shape
        cube = data.reshape(nsub * npol, nchan, nbin)
        f = np.asarray(freqs, dtype=np.float64)
        Pv = np.repeat(np.ones(nsub) * (1.0 if Ps is None else Ps), npol)
        if f.ndim == 2 and np.any(f != f[0]):
            # per-subint frequency arrays (pplib.py:2398-2411): one batch per distinct table
            if DM != 0.0 and Ps is None:
                raise ValueError("Ps and freqs are needed when DM != 0")
            tables, table_of = np.unique(f, axis=0, return_inverse=True)
            table_of = np.repeat(np.asarray(table_of).reshape(-1), npol)
            pl = get_plan(nchan, nbin)
            out = np.empty(cube.shape, dtype=np.float32)
            for t in range(len(tables)):
                sel = np.where(table_of == t)[0]
                pl.set_freqs(tables[t])
                out[sel] = pl.rotate_batch(_f32(cube[sel]), phase, DM if DM else 0.0, Pv[sel], nu)
            return out.astype(np.float64).reshape(shape)
        if f.ndim == 2:
            f = f[0]
    else:
        raise ValueError("Wrong number of dimensions.")
    if DM != 0.0 and (Ps is None or freqs is None):
        raise ValueError("Ps and freqs are needed when DM != 0")
    pl = get_plan(cube.shape[1], nbin)
    pl.set_freqs(f)
    out = pl.rotate_batch(_f32(cube), phase, DM if DM else 0.0, Pv, nu)
    return out.astype(np.float64).reshape(shape)


def rotate_portrait(port, phase=0.0, DM=None, P=None, freqs=None, nu_ref=np.inf):
    """pplib.py:2428-2460."""
    if DM is None and freqs is None:
        return rotate_data(port, phase)
    return rotate_data(port, phase, DM, P, freqs, nu_ref)


def rotate_profile(profile, phase=0.0):
    """pplib.py:2548-2559."""
    return rotate_data(profile, phase)


# ---- A11: scalar transforms (host arithmetic) --------------------------------------------
def DM_delay(DM, freq, freq_ref=np.inf, P=None):
    """pplib.py:2577-2590."""
    delay = Dconst * DM * ((freq ** -2.0) - (freq_ref ** -2.0))
    return delay / P if P else delay


def phase_transform(phi, DM, nu_ref1=np.inf, nu_ref2=np.inf, P=None, mod=False):
    """pplib.py:2592-2616."""
    if P is None:
        P, mod = 1.0, False
    phi_prime = phi + (Dconst * DM * P ** -1 * (nu_ref2 ** -2.0 - nu_ref1 ** -2.0))
    if mod:
        phi_prime = np.where(abs(phi_prime) >= 0.5, phi_prime % 1, phi_prime)
        phi_prime = np.where(phi_prime >= 0.5, phi_prime - 1.0, phi_prime)
        if not phi_prime.shape:
            phi_prime = np.float64(phi_prime)
    return phi_prime


def guess_fit_freq(freqs, SNRs=None):
    """pplib.py:2618-2632."""
    freqs = np.asarray(freqs, dtype=np.float64)
    nu0 = (freqs.min() + freqs.max()) * 0.5
    if SNRs is None:
        SNRs = np.ones(len(freqs))
    diff = np.sum((freqs - nu0) * SNRs * freqs ** -2) / np.sum(SNRs * freqs ** -2)
    return nu0 + diff


def guess_fit_freq_batch(freqs, SNRs, mask):
    """guess_fit_freq (pplib.py:2618-2632) of every row over its usable channels (mask != 0): [nsub, nchan] arrays
    in, [nsub] out; rows without usable channels give 0."""
    freqs = np.asarray(freqs, dtype=np.float64)
    m = np.asarray(mask) != 0
    w = np.where(m, np.asarray(SNRs, dtype=np.float64) * freqs ** -2, 0.0)
    den = w.sum(axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        nu0 = 0.5 * (np.where(m, freqs, np.inf).min(axis=1) + np.where(m, freqs, -np.inf).max(axis=1))
        out = nu0 + ((freqs - nu0[:, None]) * w).sum(axis=1) / den
    return np.where(m.any(axis=1) & (den != 0), out, 0.0)


def scattering_times(tau, alpha, freqs, nu_tau):
    """pplib.py:4049-4053."""
    return tau * (np.asarray(freqs, dtype=np.float64) / nu_tau) ** alpha


def scattering_portrait_FT(taus, nbin, binshift=binshift):
    """1/(1 + 2 pi i k tau_n) (pplib.py:4080-4095)."""
    taus = np.atleast_1d(np.asarray(taus, dtype=np.float64))
    nharm = nbin // 2 + 1
    if not np.any(taus):
        return np.ones([len(taus), nharm])
    return 1.0 / (1.0 + 2.0j * np.pi * np.outer(taus, np.arange(nharm)))


# ---- synthetic model portraits (host setup code, not on the hot path) ----------------------
def get_bin_centers(nbin, lo=0.0, hi=1.0):
    """pplib.py:671-684."""
    lo, hi = np.double(lo), np.double(hi)
    diff = hi - lo
    return np.linspace(lo + diff / (nbin * 2), hi - diff / (nbin * 2), nbin)


def _wrapped_gaussian(nbin, loc, wid):
    """Unit-amplitude wrapped Gaussian of FWHM wid at phase loc
    (gaussian_profile, pplib.py:770-825, norm=False)."""
    out = np.zeros(nbin)
    if not wid > 0.0:
        return out
    sigma = wid / (2 * np.sqrt(2 * np.log(2)))
    mean = loc % 1.0
    x = get_bin_centers(nbin)
    x = np.where(x > mean + 0.5, x - 1.0, x) if mean < 0.5 else \
        np.where(x < mean - 0.5, x + 1.0, x)
    z = (x - mean) / sigma
    near = np.fabs(z) < 20.0
    out[near] = np.exp(-0.5 * z[near] ** 2) / (sigma * np.sqrt(2 * np.pi))
    if np.max(np.abs(out)) == 0.0:
        return out
    ipk = out.argmax()
    return out * (np.exp(-0.5 * ((x[ipk] - loc) / sigma) ** 2) / out[ipk])


def evolve_parameter(freqs, nu_ref, parameter, evol_parameter, code):
    """Power-law ('0') or linear ('1') evolution (pplib.py:996-1046)."""
    freqs = np.asarray(freqs, dtype=np.float64)
    if code == "0":
        return np.exp(np.outer(np.log(freqs) - np.log(nu_ref), evol_parameter) +
                      np.outer(np.ones(len(freqs)), np.log(parameter)))
    if code == "1":
        return np.outer(freqs - nu_ref, evol_parameter) + \
            np.outer(np.ones(len(freqs)), parameter)
    raise KeyError(code)


_gauss_max_join = 8


def _join_table(join_ichans, nchan, P):
    """int32 [nchan] join group of each channel (-1: none) from join_ichans, a sequence of channel-index lists
    (one per archive after the first).  Groups must be non-empty, disjoint and in range, at most 8, and P > 0."""
    njoin = len(join_ichans)
    if njoin > _gauss_max_join:
        raise ValueError("at most %d join groups (got %d)" % (_gauss_max_join, njoin))
    if P is None or not float(P) > 0.0:
        raise ValueError("join parameters need the period P > 0 (got %r)" % (P,))
    table = np.full(nchan, -1, dtype=np.int32)
    for j, ich in enumerate(join_ichans):
        ich = np.atleast_1d(np.asarray(ich))
        if not ich.size:
            raise ValueError("join group %d is empty" % j)
        if ich.dtype.kind not in "iu":
            raise ValueError("join group %d: channel indices must be integers" % j)
        if ich.min() < 0 or ich.max() >= nchan:
            raise ValueError("join group %d: channel index out of range [0, %d)" % (j, nchan))
        if (table[ich] >= 0).any() or len(np.unique(ich)) != ich.size:
            raise ValueError("join group %d overlaps another group" % j)
        table[ich] = j
    return table


def gen_gaussian_portrait(model_code, params, scattering_index, phases, freqs,
                          nu_ref, join_ichans=[], P=None):
    """Evolving-Gaussian model portrait (pplib.py:853-930).  params =
    [DC, tau_bin, (loc, m_loc, wid, m_wid, amp, m_amp) * ngauss, (phi_j, DM_j) * len(join_ichans)].

    Join parameters: after scattering, the channels join_ichans[j] are rotated as rotate_data(rows, phi_j, DM_j,
    P, freqs, nu_ref) does, here in float64 numpy: harmonic k times e^{2 pi i k theta_n}, theta_n = phi_j +
    Dconst DM_j / P (nu_n^-2 - nu_ref^-2), the Nyquist term keeping its real part (irfft).  P [s] is required with
    joins; the groups must be disjoint, non-empty and in range (ValueError)."""
    params = np.asarray(params, dtype=np.float64)
    freqs = np.asarray(freqs, dtype=np.float64)
    nbin, nchan = len(phases), len(freqs)
    njoin = len(join_ichans)
    if njoin:
        table = _join_table(join_ichans, nchan, P)
        params, jvals = params[:len(params) - 2 * njoin], params[len(params) - 2 * njoin:]
    locs = evolve_parameter(freqs, nu_ref, params[2::6], params[3::6], model_code[0])
    wids = evolve_parameter(freqs, nu_ref, params[4::6], params[5::6], model_code[1])
    amps = evolve_parameter(freqs, nu_ref, params[6::6], params[7::6], model_code[2])
    gport = np.empty([nchan, nbin])
    for ichan in range(nchan):
        prof = np.zeros(nbin) + params[0]
        for ig in range(locs.shape[1]):
            prof += amps[ichan, ig] * _wrapped_gaussian(nbin, locs[ichan, ig], wids[ichan, ig])
        gport[ichan] = prof
    tau = params[1]
    if tau != 0.0:
        taus = scattering_times(float(tau) / nbin, scattering_index, freqs, nu_ref)
        gport = np.fft.irfft(scattering_portrait_FT(taus, nbin) *
                             np.fft.rfft(gport, axis=-1), axis=-1)
    if njoin:
        rows = np.where(table >= 0)[0]
        j = table[rows]
        theta = jvals[2 * j] + Dconst * jvals[2 * j + 1] / float(P) * (freqs[rows] ** -2.0 - nu_ref ** -2.0)
        ph = np.exp(2j * np.pi * np.outer(theta, np.arange(nbin // 2 + 1)))
        gport[rows] = np.fft.irfft(ph * np.fft.rfft(gport[rows], axis=-1), n=nbin, axis=-1)
    return gport


def gen_gaussian_portrait_device(model_code, params, scattering_index, phases, freqs,
                                 nu_ref, join_ichans=[], P=None):
    """gen_gaussian_portrait (pplib.py:853-930) evaluated by the CUDA kernel
    ``k_gauss_model`` (+ the scattering multiply of ``k_rotate``): the per-archive /
    per-subint model build of pptoas.py:356-379.  ``phases`` must be the bin centres
    of get_bin_centers(nbin).  Returns float64 [nchan, nbin], evaluated in double (a scattered model,
    tau != 0, passes through float32 rows).

    With join_ichans (and P) the joined model of gen_gaussian_portrait is evaluated in FP64 by the model output
    of the fit's kernel (WidebandPlan.gen_gaussian_portrait with join_chan): ngauss >= 1 and nbin a power of
    two."""
    nbin, nchan = len(phases), len(freqs)
    if not np.allclose(phases, get_bin_centers(nbin), rtol=0, atol=1e-12):
        raise ValueError("the device generator works on get_bin_centers(nbin)")
    table = _join_table(join_ichans, nchan, P) if len(join_ichans) else None
    pl = get_plan(nchan, nbin)
    pl.set_freqs(np.asarray(freqs, dtype=np.float64))
    if table is not None:
        return pl.gen_gaussian_portrait(model_code, params, scattering_index, nu_ref, join_chan=table, P=P)
    return pl.gen_gaussian_portrait(model_code, params, scattering_index, nu_ref, dtype=np.float64)


def gen_spline_portrait(mean_prof, freqs, eigvec, tck, nbin=None, device=False):
    """Model portrait from a make_spline_model(...) PCA / B-spline model
    (pplib.py:932-956): mean_prof + splev(freqs, tck).T . eigvec.T.  ``device=True``
    evaluates it with the CUDA kernel ``k_spline_model`` (float32 precision)."""
    mean_prof = np.asarray(mean_prof, dtype=np.float64)
    freqs = np.asarray(freqs, dtype=np.float64)
    eigvec = np.asarray(eigvec, dtype=np.float64).reshape(len(mean_prof), -1)
    shift = 0.0
    if nbin is not None and nbin != len(mean_prof):
        # pplib.py:951-955: Fourier resampling, then the half-bin-difference rotation that undoes
        # the shift ss.resample introduces.  Resampling is linear along the bin axis, so it is
        # applied to the basis (mean profile, eigenvectors) once instead of to every channel.
        import scipy.signal as ss
        shift = 0.5 * (nbin ** -1 - len(mean_prof) ** -1)
        mean_prof = ss.resample(mean_prof, nbin)
        eigvec = ss.resample(eigvec, nbin, axis=0)
    if device:
        pl = get_plan(len(freqs), len(mean_prof))
        pl.set_freqs(freqs)
        port = pl.gen_spline_portrait(mean_prof, eigvec, tck).astype(np.float64)
    elif not eigvec.shape[1]:
        port = np.tile(mean_prof, len(freqs)).reshape(len(freqs), len(mean_prof))
    else:
        import scipy.interpolate as si
        proj_port = np.array(si.splev(freqs, tck, der=0, ext=0)).T
        port = np.dot(proj_port, eigvec.T) + mean_prof
    if shift:
        port = rotate_portrait(port, shift)
    return port


def read_spline_model(modelfile, freqs=None, nbin=None, quiet=False, device=False):
    """Read a make_spline_model(...) pickle (pplib.py:2955-2987): without freqs returns
    (modelname, source, datafile, mean_prof, eigvec, tck), else (modelname, model)."""
    import pickle
    if not quiet:
        print("Reading model from %s..." % modelfile)
    with open(modelfile, "rb") as fh:
        modelname, source, datafile, mean_prof, eigvec, tck = pickle.load(fh, encoding="latin1")
    if freqs is None:
        return (modelname, source, datafile, mean_prof, eigvec, tck)
    return (modelname, gen_spline_portrait(mean_prof, freqs, eigvec, tck, nbin, device=device))


def is_spline_model(modelfile):
    """True if ``modelfile`` is a pickled spline model rather than a text .gmodel file
    (the reference falls back to read_spline_model when read_model fails, pptoas.py:376-379)."""
    import pickle
    try:
        with open(modelfile, "rb") as fh:
            obj = pickle.load(fh, encoding="latin1")
        return isinstance(obj, (list, tuple)) and len(obj) == 6
    except Exception:
        return False


def read_model(modelfile, phases=None, freqs=None, P=None, quiet=False, device=False):
    """Read a ``.gmodel`` file (pplib.py:2867-2953).  Without phases/freqs
    returns (name, code, nu_ref, ngauss, params, fit_flags, alpha, fit_alpha);
    otherwise (name, ngauss, model).  ``device=True`` builds the portrait on the GPU."""
    read_only = phases is None and freqs is None
    comps = []
    modelname, model_code, nu_ref = "", default_model, None
    dc = tau = 0.0
    alpha = scattering_alpha
    fit_dc = fit_tau = fit_alpha = 0
    with open(modelfile, "r") as fh:
        for line in fh:
            info = line.split()
            if not info:
                continue
            try:
                if info[0] == "MODEL":
                    modelname = info[1]
                elif info[0] == "CODE":
                    model_code = info[1]
                elif info[0] == "FREQ":
                    nu_ref = np.float64(info[1])
                elif info[0] == "DC":
                    dc, fit_dc = np.float64(info[1]), int(info[2])
                elif info[0] == "TAU":
                    tau, fit_tau = np.float64(info[1]), int(info[2])
                elif info[0] == "ALPHA":
                    alpha, fit_alpha = np.float64(info[1]), int(info[2])
                elif info[0][:4] == "COMP":
                    comps.append(info)
            except IndexError:
                pass
    ngauss = len(comps)
    params = np.zeros(ngauss * 6 + 2)
    fit_flags = np.zeros(len(params))
    params[0], params[1] = dc, tau
    fit_flags[0], fit_flags[1] = fit_dc, fit_tau
    for ig, info in enumerate(comps):
        params[2 + ig * 6: 8 + ig * 6] = [np.float64(v) for v in info[1::2][:6]]
        fit_flags[2 + ig * 6: 8 + ig * 6] = [int(v) for v in info[2::2][:6]]
    if read_only:
        return (modelname, model_code, nu_ref, ngauss, params, fit_flags, alpha, fit_alpha)
    nbin = len(phases)
    if params[1] != 0:
        if P is None:
            print("Need period P for non-zero scattering value TAU.")
            return 0
        params[1] *= nbin / P
    gen = gen_gaussian_portrait_device if device else gen_gaussian_portrait
    model = gen(model_code, params, alpha, phases, freqs, nu_ref)
    if not quiet:
        print("Model Name: %s" % modelname)
        print("Made %d component model with %d profile bins," % (ngauss, nbin))
    return (modelname, ngauss, model)


# ---- ppgauss: fitting and writing evolving-Gaussian models --------------------------------------
# lower edge of the facade's 0 < wid box: far below one bin of the largest nbin (1/4096 ~ 2.4e-4 rot)
_gauss_wid_min = 1e-6


def _gauss_default_bounds(model_code, ngauss):
    """[P, 2] bounds (NaN = open) in the layout [DC, tau, comps..., alpha]: tau >= 0,
    _gauss_wid_min <= wid <= wid_max, amp >= 0, and loc >= 0 where the loc code is a power law (its
    logarithm is taken)."""
    P = 3 + 6 * ngauss
    b = np.full((P, 2), np.nan)
    b[1, 0] = 0.0
    for ig in range(ngauss):
        o = 2 + 6 * ig
        if model_code[0] == "0":
            b[o, 0] = 0.0
        b[o + 2] = (_gauss_wid_min, wid_max)
        b[o + 4, 0] = 0.0
    return b


def fit_gaussian_portrait(model_code, data, init_params, scattering_index, errs, fit_flags,
                          fit_scattering_index, phases, freqs, nu_ref, join_params=[], P=None,
                          quiet=True):
    """Fit an evolving-Gaussian model portrait to ``data`` [nchan, nbin] (pplib.py:1924-2052), on the GPU.

    init_params = [DC, tau [bin], (loc, m_loc, wid, m_wid, amp, m_amp) * ngauss] as gen_gaussian_portrait
    takes them, scattering_index the start value of alpha, errs [nchan] the per-channel sigma, fit_flags
    one flag per entry of init_params and fit_scattering_index alpha's flag.  ``phases`` must be
    get_bin_centers(nbin); nbin a power of two in [64, 4096].  The objective is the reference's
    chi^2 = sum (data - model)^2 / errs^2 with the model of gen_gaussian_portrait (scattered when tau != 0
    or tau / alpha are free), minimised by a Levenberg-Marquardt solver with analytic derivatives
    (WidebandPlan.fit_gaussian_portraits).

    Bounds, the policy of this facade: tau >= 0, 0 < wid <= wid_max (wid_max = 0.25 in this module's
    settings; the lower edge is wid = 1e-6 rot, far below one bin), amp >= 0, and loc >= 0 when its
    evolution code is a power law.  A free parameter that cannot move the model at the fitted point (alpha
    while tau = 0, for example) gets fit_err 0 and a zero covariance row, MINPACK's convention.

    Join parameters fit one model to the portraits of several archives (receivers or bands) joined along the
    channel axis (join_archives makes such a portrait): join_params = [join_ichans, join_values,
    join_fit_flags] with join_ichans one list of channel indices per archive after the first, join_values
    [phi_1, DM_1, ..., phi_J, DM_J] (start values) and join_fit_flags one flag per value; P [s] is the period
    of the DM term.  The channels join_ichans[j] of the model are rotated by phi_j and DM_j about nu_ref after
    scattering, as gen_gaussian_portrait(..., join_ichans, P) defines it; the other channels are the reference.
    Up to 8 groups, disjoint, non-empty and in range (ValueError otherwise); join_params that is not a
    three-part sequence raises NotImplementedError.  phi_j and DM_j are not bounded.

    Returns a DataBunch with fitted_params (layout of init_params, tau in bins), fit_errs,
    scattering_index, scattering_index_err, join_params and join_param_errs ([phi_1, DM_1, ...]; empty
    without joins), chi2, dof, red_chi2, nfeval, return_code (0 converged, 1 iteration limit, 3 non-finite),
    duration, and the extras covariance ([P, P] in the layout [params..., alpha, phi_1, DM_1, ...], scaled by
    red_chi2 as lmfit's scale_covar) and model (the fitted portrait, float64).  The reference's lm_results
    (the lmfit object) cannot be provided."""
    table, jvals, jflags = None, np.zeros(0), np.zeros(0, bool)
    if len(join_params):
        if isinstance(join_params, (str, bytes)) or len(join_params) != 3:
            raise NotImplementedError("join_params must be [join_ichans, join_values, join_fit_flags]")
        join_ichans, jvals, jflags = join_params
        table = _join_table(join_ichans, np.shape(data)[0], P)
        jvals = np.asarray(jvals, dtype=np.float64).ravel()
        jflags = np.asarray(jflags, dtype=bool).ravel()
        if jvals.size != 2 * len(join_ichans) or jflags.size != jvals.size:
            raise ValueError("join_values and join_fit_flags need 2 entries (phi, DM) per join group")
    start = time.time()
    data = np.asarray(data, dtype=np.float64)
    nchan, nbin = data.shape
    if len(phases) != nbin or not np.allclose(phases, get_bin_centers(nbin), rtol=0, atol=1e-12):
        raise ValueError("the device fit works on get_bin_centers(nbin)")
    init_params = np.asarray(init_params, dtype=np.float64)
    if init_params.ndim != 1 or (init_params.size - 2) % 6 or init_params.size < 8:
        raise ValueError("init_params must have 2 + 6*ngauss entries")
    ngauss = (init_params.size - 2) // 6
    x0 = np.concatenate([init_params, [float(scattering_index)], jvals])
    flags = np.concatenate([np.asarray(fit_flags, dtype=bool), [bool(fit_scattering_index)], jflags])
    bounds = np.concatenate([_gauss_default_bounds(model_code, ngauss), np.full((jvals.size, 2), np.nan)])
    pl = get_plan(nchan, nbin)
    pl.set_freqs(np.asarray(freqs, dtype=np.float64))
    r = pl.fit_gaussian_portraits(data[None], np.asarray(errs, dtype=np.float64).reshape(1, nchan), model_code,
                                  x0[None], flags, nu_ref, bounds=bounds, want_model=True, join_chan=table, P=P)
    params, perrs = r["params"][0], r["param_errs"][0]
    ia = init_params.size
    rc = int(r["return_code"][0])
    if not quiet:
        print("Fit %d-component model: chi2 %.3f, red_chi2 %.5f, %d evaluations (%s)"
              % (ngauss, r["chi2"][0], r["red_chi2"][0], r["nfeval"][0], DEVICE_RCSTRINGS.get(str(rc), rc)))
    return DataBunch(fitted_params=params[:ia].copy(), fit_errs=perrs[:ia].copy(),
                     scattering_index=params[ia], scattering_index_err=perrs[ia],
                     join_params=params[ia + 1:].copy(), join_param_errs=perrs[ia + 1:].copy(),
                     chi2=r["chi2"][0], dof=int(r["dof"][0]), red_chi2=r["red_chi2"][0],
                     nfeval=int(r["nfeval"][0]), return_code=rc, duration=time.time() - start,
                     covariance=r["cov"][0], model=r["model"][0])


def join_archives(archives, ref=0):
    """One portrait of several archives of one pulsar (DataBunches or .npz paths that pptoas.load_data reads, all
    with the same nbin), for a joined fit_gaussian_portrait: each archive is averaged over its subints
    (pptoas.tscrunch_databunch, total intensity), and the usable channels of every archive are concatenated in the
    order given.  Archives are used as stored (dispersed unless stored dedispersed).

    Returns a DataBunch with port [nchan, nbin], freqs [nchan], noise_stds [nchan] (get_noise of each averaged
    channel), P (the period of archive ``ref``), join_ichans (the channel indices of every archive but ``ref``, in
    order: the join_ichans of fit_gaussian_portrait), archive_ichans (those of every archive) and nbin."""
    from .pptoas import load_data, tscrunch_databunch
    if not len(archives):
        raise ValueError("no archives")
    if not 0 <= ref < len(archives):
        raise ValueError("ref must index one of the %d archives" % len(archives))
    ds = [tscrunch_databunch(load_data(a) if isinstance(a, (str, os.PathLike)) else a) for a in archives]
    nbins = {int(d.nbin) for d in ds}
    if len(nbins) != 1:
        raise ValueError("the archives must have one nbin (got %s)" % sorted(nbins))
    ports, freqs, noise, ichans, n0 = [], [], [], [], 0
    for d in ds:
        ok = np.asarray(d.ok_ichans[0], dtype=int)
        ports.append(np.asarray(d.subints, dtype=np.float64)[0, 0, ok])
        freqs.append(np.asarray(d.freqs, dtype=np.float64)[0, ok])
        noise.append(np.asarray(d.noise_stds, dtype=np.float64)[0, 0, ok])
        ichans.append(np.arange(n0, n0 + len(ok)))
        n0 += len(ok)
    return DataBunch(port=np.concatenate(ports), freqs=np.concatenate(freqs), noise_stds=np.concatenate(noise),
                     P=float(np.asarray(ds[ref].Ps)[0]), join_ichans=[ichans[i] for i in range(len(ds)) if i != ref],
                     archive_ichans=ichans, nbin=nbins.pop())


def write_model(filenm, name, model_code, nu_ref, model_params, fit_flags, alpha, fit_alpha,
                append=False, quiet=False):
    """Write a .gmodel file that read_model parses (pplib.py:2830-2865), in the layout of ppgauss's
    output: MODEL, CODE, FREQ, DC, TAU, ALPHA and one COMPnn line per component.

    model_params = [DC, TAU, (loc, m_loc, wid, m_wid, amp, m_amp) * ngauss] with TAU in seconds, the
    file's unit: a tau fitted in bins (fit_gaussian_portrait) is written as tau_bin * P / nbin for a
    period P [s].  Values are printed with 12 decimals (FREQ with 10)."""
    model_params = np.asarray(model_params, dtype=np.float64)
    fit_flags = np.asarray(fit_flags).astype(int)
    ngauss = (len(model_params) - 2) // 6
    lines = ["MODEL   %s" % name,
             "CODE    %s" % model_code,
             "FREQ    %.10f" % nu_ref,
             "DC     % .12f %d" % (model_params[0], fit_flags[0]),
             "TAU    % .12f %d" % (model_params[1], fit_flags[1]),
             "ALPHA  % .12f %d" % (alpha, int(fit_alpha))]
    for ig in range(ngauss):
        o = 2 + 6 * ig
        fields = "".join("  % .12f %d" % (model_params[o + k], fit_flags[o + k]) for k in range(6))
        lines.append("COMP%02d%s" % (ig + 1, fields))
    with open(filenm, "a" if append else "w") as fh:
        fh.write("\n".join(lines) + "\n")
    if not quiet:
        print("%s written." % filenm)


# ---- ppspline: PCA / B-spline models -------------------------------------------------------------
def _sign_convention(vecs):
    """Columns of vecs [nbin, m] with their entry of largest |value| (the first such) made positive."""
    vecs = np.array(vecs, dtype=np.float64)
    if vecs.shape[1]:
        ipk = np.argmax(np.abs(vecs), axis=0)
        vecs *= np.where(vecs[ipk, np.arange(vecs.shape[1])] < 0.0, -1.0, 1.0)
    return vecs


def make_spline_model(port, freqs, weights=None, noise_stds=None, max_ncomp=10, smooth=True, snr_cutoff=150.0, k=3,
                      sfac=1.0, max_nbreak=None, norm="prof", model_name=None, source=None, datafile=None, quiet=True):
    """Build a PCA + B-spline model portrait (ppspline.py make_spline_model, pplib pca / find_significant_eigvec)
    from an aligned portrait port [nchan, nbin] at frequencies freqs [nchan] (MHz), on the device.

    1. Usable channels: weight > 0 and a row not all zero, sorted by frequency (duplicate frequencies raise
       ValueError).  With ``norm`` they are normalised by ppalign.normalize_portrait(norm) and noise_stds scaled by
       the same factors; the default noise_stds are get_noise ("PS") per channel, measured on the device.
    2. PCA: the weighted mean profile mu and the second-moment matrix of sqrt(w_n) (x_n - mu) on the device, on the
       smaller side (the covariance when the usable channels outnumber the bins, else the Gram matrix, whose
       eigenvectors are back-projected); the top max_ncomp eigenpairs on the host, eigenvalues descending.
    3. Significance: with ``smooth`` mu and each eigenvector e_j are low-passed (rfft, harmonics above find_kc's k_c
       zeroed, irfft: WidebandPlan.lowpass_rows); snr_j = ||e~_j|| / sigma(e_j) with sigma the get_noise "PS" noise
       of the unsmoothed e_j, and the e_j with snr_j >= snr_cutoff are kept in eigenvalue order (ieig).  The
       reference smooths with wavelets (pywt), which is not used here, so the S/N of an eigenvector and therefore
       the number kept for a given cutoff can differ from the reference's.
    4. Basis: the kept smoothed vectors orthonormalised (QR, then each with its entry of largest |value| positive),
       eigvec [nbin, ncomp]; the projections proj_port [n_ok, ncomp] of x_n - mu~ on the device.
    5. Spline: scipy.interpolate.splprep(proj_port.T, u=freqs, w=1/noise_stds, k=k, s=sfac ncomp n_ok,
       nest=None or max_nbreak + 2k): s is the expected chi^2 of pure noise under FITPACK's weighted condition.
       ncomp = 0 gives the smoothed mean alone, tck = (zeros(2k + 2), [], k).

    Returns a DataBunch: model_name, source, datafile, mean_prof, eigvec, tck, ncomp, ieig, eigval, snrs, kc (of
    [mean, e_0, ...]; None without smoothing), proj_port, freqs, weights, noise_stds and channel_red_chi2s (all of the
    usable channels in frequency order), fp, ier, msg (splprep's), model (gen_spline_portrait(..., device=True) at the
    input freqs) and duration.  channel_red_chi2s = sum_b ((x_nb - model_nb) / noise_std_n)^2 / nbin of the normalised
    data.  write_spline_model writes the model for read_spline_model / GetTOAs."""
    import scipy.interpolate as si
    import scipy.linalg as sl
    start = time.time()
    port = np.asarray(port, dtype=np.float64)
    if port.ndim != 2:
        raise ValueError("port must be [nchan, nbin]")
    nchan, nbin = port.shape
    freqs = np.asarray(freqs, dtype=np.float64).reshape(-1)
    if len(freqs) != nchan:
        raise ValueError("freqs has %d entries for %d channels" % (len(freqs), nchan))
    weights = np.ones(nchan) if weights is None else np.asarray(weights, dtype=np.float64).reshape(-1)
    if len(weights) != nchan or np.any(weights < 0) or not np.all(np.isfinite(weights)):
        raise ValueError("weights must be [nchan] finite values >= 0")
    k = int(k)
    if not 1 <= k <= 5:
        raise ValueError("the spline degree k must be in [1, 5] (got %d)" % k)
    if int(max_ncomp) < 0:
        raise ValueError("max_ncomp must be >= 0")
    iok = np.nonzero((weights > 0) & port.any(axis=1))[0]
    order = iok[np.argsort(freqs[iok], kind="stable")]
    fok = freqs[order]
    if np.any(np.diff(fok) == 0):
        raise ValueError("duplicate frequencies among the usable channels")
    n_ok = len(order)
    if n_ok <= k:
        raise ValueError("%d usable channels: the spline of degree %d needs more than %d" % (n_ok, k, k))
    X, w = port[order], weights[order]
    norms = np.ones(n_ok)
    if norm is not None:
        from .ppalign import normalize_portrait
        r = normalize_portrait(X, norm, weights=w, return_norms=True)
        if r is None:
            raise ValueError("unknown norm %r" % (norm,))
        X, norms = r
    pl = get_plan(n_ok, nbin)
    if noise_stds is None:
        sig = get_noise_PS(X, chans=True)
    else:
        sig = np.asarray(noise_stds, dtype=np.float64).reshape(-1)
        if len(sig) != nchan:
            raise ValueError("noise_stds has %d entries for %d channels" % (len(sig), nchan))
        sig = sig[order] / norms
    if not np.all(sig > 0):
        raise ValueError("the noise of every usable channel must be positive")

    # PCA.  The eigen decomposition runs on the host (LAPACK's syevr through scipy.linalg.eigh, the top max_ncomp
    # pairs only): the matrix has at most min(n_ok, nbin)^2 entries and the decomposition is a small, latency-bound
    # part of the whole, which a device eigensolver would not shorten enough to be worth writing and pinning.
    gram = n_ok <= nbin
    mu, M = pl.pca_moments(X, w, gram=gram)
    dim = M.shape[0]
    m = min(int(max_ncomp), dim)
    if m:
        eigval, U = sl.eigh(M, subset_by_index=[dim - m, dim - 1])
        eigval, U = eigval[::-1].copy(), np.ascontiguousarray(U[:, ::-1])
        E = pl.pca_backproject(X, w, mu, U) if gram else _sign_convention(U)
    else:
        eigval, E = np.zeros(0), np.zeros((nbin, 0))

    # significance
    rows = np.ascontiguousarray(np.vstack([mu[None], E.T]))
    if smooth:
        srows, kc = get_plan(len(rows), nbin).lowpass_rows(rows)
    else:
        srows, kc = rows, None
    mean_prof = srows[0].copy()
    if m:
        snrs = np.linalg.norm(srows[1:], axis=1) / get_noise_PS(E.T, chans=True)
    else:
        snrs = np.zeros(0)
    ieig = np.nonzero(snrs >= snr_cutoff)[0]
    ncomp = len(ieig)
    if ncomp:
        eigvec = _sign_convention(np.linalg.qr(srows[1:][ieig].T)[0])
        proj = pl.pca_project(X, mean_prof, eigvec)
        nest = None if max_nbreak is None else int(max_nbreak) + 2 * k
        (tck, _), fp, ier, msg = si.splprep(proj.T, u=fok, w=1.0 / sig, k=k, s=float(sfac) * ncomp * n_ok, nest=nest,
                                            full_output=1, quiet=1)
        tck = (np.asarray(tck[0]), [np.asarray(c) for c in tck[1]], int(tck[2]))
    else:
        eigvec, proj = np.zeros((nbin, 0)), np.zeros((n_ok, 0))
        tck, fp, ier, msg = (np.zeros(2 * k + 2), [], k), 0.0, 0, "no significant eigenvector: the model is the mean"
    model = gen_spline_portrait(mean_prof, freqs, eigvec, tck, device=True)
    red_chi2s = (((X - model[order]) / sig[:, None]) ** 2).sum(axis=1) / nbin
    if not quiet:
        print("%d of %d eigenvectors significant (S/N >= %g); splprep: fp = %.4g, ier = %s"
              % (ncomp, m, snr_cutoff, fp, ier))
    return DataBunch(model_name=model_name, source=source, datafile=datafile, mean_prof=mean_prof, eigvec=eigvec,
                     tck=tck, ncomp=ncomp, ieig=ieig, eigval=eigval, snrs=snrs, kc=kc, proj_port=proj, freqs=fok,
                     weights=w, noise_stds=sig, fp=fp, ier=ier, msg=msg, model=model, channel_red_chi2s=red_chi2s,
                     duration=time.time() - start)


def write_spline_model(outfile, model_name, source, datafile, mean_prof, eigvec, tck, quiet=False):
    """Pickle a PCA / B-spline model as the list [model_name, source, datafile, mean_prof, eigvec, tck] (protocol 2),
    the layout of ppspline.py's write_model that read_spline_model, is_spline_model and GetTOAs read."""
    import pickle
    with open(outfile, "wb") as fh:
        pickle.dump([model_name, source, datafile, mean_prof, eigvec, tck], fh, protocol=2)
    if not quiet:
        print("%s written." % outfile)


# ---- simulated archives (pplib.py:3183-3378) --------------------------------------------------
def read_ephemeris(ephemeris):
    """(F0 [Hz], F1 [Hz/s], PEPOCH [MJD], DM, source) from a .par file (F0, optional F1 and PEPOCH, DM, PSRJ / PSR)
    or a spin period in seconds (F1 = 0, DM = 0)."""
    if np.ndim(ephemeris) == 0 and not isinstance(ephemeris, str):
        P = float(ephemeris)
        if not P > 0.0:
            raise ValueError("the period must be positive (got %g)" % P)
        return 1.0 / P, 0.0, 0.0, 0.0, "fake"
    vals, source = {}, "fake"
    with open(ephemeris, "r") as fh:
        for line in fh:
            info = line.split()
            if len(info) < 2:
                continue
            key = info[0].upper()
            if key in ("PSRJ", "PSR", "PSRB"):
                source = info[1]
            elif key in ("F0", "F1", "PEPOCH", "DM"):
                vals[key] = float(info[1].replace("D", "E").replace("d", "e"))
    if not vals.get("F0", 0.0) > 0.0:
        raise ValueError("%s: no positive F0" % ephemeris)
    return vals["F0"], vals.get("F1", 0.0), vals.get("PEPOCH", 0.0), vals.get("DM", 0.0), source


def _per_subint(v, nsub, name):
    a = np.asarray(v, dtype=np.float64)
    if a.ndim > 1 or (a.ndim == 1 and len(a) != nsub):
        raise ValueError("%s must be a scalar or [nsub = %d]" % (name, nsub))
    return np.broadcast_to(a, (nsub,)).copy()


def _per_chan(v, nsub, nchan, name):
    a = np.asarray(v, dtype=np.float64)
    if a.shape not in ((), (nchan,), (nsub, nchan)):
        raise ValueError("%s must be a scalar, [nchan = %d] or [nsub, nchan] = [%d, %d]" % (name, nchan, nsub, nchan))
    return np.broadcast_to(a, (nsub, nchan)).copy()


def make_fake_pulsar(modelfile, ephemeris, outfile=None, nsub=1, npol=1, nchan=512, nbin=2048, nu0=1500.0, bw=800.0,
                     tsub=300.0, phase=0.0, dDM=0.0, start_MJD=None, weights=None, noise_stds=1.0, scales=1.0,
                     dedispersed=False, t_scat=0.0, alpha=scattering_alpha, scint=False, nu_DM=np.inf,
                     state="Intensity", obs="GBT", seed=0, quantize=False, quiet=False):
    """A simulated archive (pplib.py:3183-3378), made on the device (WidebandPlan.simulate_batch) and returned as
    the DataBunch that load_data gives, written with pptoas.save_databunch when ``outfile`` is given (so that
    load_data, GetTOAs, align_archives and tscrunch_databunch take it).  PSRFITS writing is not provided.

    modelfile: a .gmodel file (a TAU != 0 gives one model per distinct period), a spline model, or a [nchan, nbin]
    array.  ephemeris: a .par file (F0, optional F1 and PEPOCH, DM) or a period [s]; subint s is folded with
    P_s = 1/(F0 + F1 (t_s - PEPOCH)) at its mid-epoch t_s = start_MJD + (s + 1/2) tsub (start_MJD default 56000).
    Channels: nchan centre frequencies across bw about nu0 [MHz].  phase [rot], dDM, t_scat [s at nu0] and alpha:
    scalars or [nsub]; noise_stds and scales: scalars, [nchan] or [nsub, nchan].  The subints are dispersed by
    DM_par + dDM about nu_DM, scattered by t_scat, scaled and given Gaussian noise of rms noise_stds drawn from
    ``seed`` (subint s always draws the same numbers).  dedispersed=True stores them with DM_par removed about nu0
    (dmc = 1) by a second device rotation of the simulated rows, which pptoas.restore_dispersion undoes in every
    harmonic but the Nyquist one (a rotation keeps only the real part of that term).  quantize=True also stores them as the int16 samples with
    DAT_SCL / DAT_OFFS a PSRFITS file holds (raw_subints, dat_scl, dat_offs) and ``subints`` holds the decoded
    values.  A scintillation pattern can be given as [nsub, nchan] ``scales`` (scint=True, the reference's own
    pattern, is not provided); npol > 1 is not provided.

    noise_stds in the result are measured from the profiles on the device (get_noise, as load_data does).  SNRs
    are the injected matched-filter S/N per channel, scale ||m_n - mean(m_n)|| / sigma_n; the reference measures
    them from the profiles."""
    from .pptoas import MJD, quantize_subints, save_databunch
    if npol != 1:
        raise ValueError("npol = %d: only total intensity (npol = 1) is simulated" % npol)
    if scint:
        raise NotImplementedError("scint: pass a scintillation pattern as [nsub, nchan] scales")
    nsub, nchan, nbin = int(nsub), int(nchan), int(nbin)
    if nsub < 1:
        raise ValueError("nsub must be >= 1")
    F0, F1, PEPOCH, DM_par, source = read_ephemeris(ephemeris)
    freqs = np.linspace(nu0 - bw / 2.0 + bw / (2.0 * nchan), nu0 + bw / 2.0 - bw / (2.0 * nchan), nchan)
    phases = get_bin_centers(nbin)
    start = MJD(56000, 0.0) if start_MJD is None else (start_MJD if isinstance(start_MJD, MJD) else MJD(start_MJD))
    epochs = [start + (s + 0.5) * tsub / 86400.0 for s in range(nsub)]
    dt = np.array([((e.intday() - PEPOCH) + e.fracday()) * 86400.0 for e in epochs]) if F1 else np.zeros(nsub)
    Ps = 1.0 / (F0 + F1 * dt)
    if not np.all(Ps > 0.0):
        raise ValueError("the ephemeris gives a non-positive period")
    phase = _per_subint(phase, nsub, "phase")
    DMs = DM_par + _per_subint(dDM, nsub, "dDM")
    t_scat = _per_subint(t_scat, nsub, "t_scat")
    alpha = _per_subint(alpha, nsub, "alpha")
    noise = _per_chan(noise_stds, nsub, nchan, "noise_stds")
    scl = _per_chan(scales, nsub, nchan, "scales")
    w = np.ones((nsub, nchan)) if weights is None else _per_chan(weights, nsub, nchan, "weights")
    if np.any(noise < 0):
        raise ValueError("noise_stds must be >= 0")
    # model portraits: one per distinct period when the .gmodel's TAU makes the model depend on it
    if isinstance(modelfile, np.ndarray) or hasattr(modelfile, "shape"):
        models, model_index = np.asarray(modelfile, dtype=np.float64)[None], None
        if models.shape[1:] != (nchan, nbin):
            raise ValueError("the model array must be [nchan, nbin] = [%d, %d]" % (nchan, nbin))
    elif is_spline_model(modelfile):
        m = read_spline_model(modelfile, freqs, nbin, quiet=True, device=True)[1]
        models, model_index = np.asarray(m, dtype=np.float64)[None], None
    else:
        if read_model(modelfile, quiet=True)[4][1] != 0.0:
            uP, model_index = np.unique(Ps, return_inverse=True)
            models = np.stack([read_model(modelfile, phases, freqs, p, quiet=True, device=True)[2] for p in uP])
            model_index = np.asarray(model_index, dtype=np.int32).reshape(-1)
        else:
            models, model_index = read_model(modelfile, phases, freqs, Ps[0], quiet=True, device=True)[2][None], None
        models = np.ascontiguousarray(models, dtype=np.float64)
    scat = t_scat != 0.0
    pl = get_plan(nchan, nbin)
    data = pl.simulate_batch(models, np.tile(freqs, (len(models), 1)), phase, DMs, Ps, nu_DM=nu_DM,
                             tau=t_scat / Ps if scat.any() else None, alpha=alpha if scat.any() else None,
                             nu_tau=nu0 if scat.any() else None, scales=scl, noise_stds=noise, seed=seed,
                             model_index=model_index, device_out=dedispersed)
    if dedispersed:
        # The stored archive, as arch.dedisperse() writes it: the simulated rows rotated by DM_par about nu0, in place
        # on the device.  This is a second pass over the rows rather than DM_par folded into the simulation's phase
        # and DM: folded in, the noise would be drawn in the dedispersed frame, and restore_dispersion could not give
        # back the dedispersed=False archive.  A plan of its own, so that the cached plan's frequency table and FFT
        # precision stay as the caller left them.
        with WidebandPlan(nchan, nbin, device=pl.device) as rp:
            rp.set_freqs(freqs)
            rp.set_fft_precision(64)
            rp.rotate_batch(data, 0.0, DM_par, Ps, nu0, out=data)
        data = data.cpu().numpy()
    raw = dat_scl = dat_offs = None
    if quantize:
        raw, dat_scl, dat_offs, data = quantize_subints(data)
    sig = pl.get_noise_batch(_f32(data))
    mnorm = np.linalg.norm(models - models.mean(axis=-1, keepdims=True), axis=-1)     # [nmodel, nchan]
    mnorm = mnorm[np.zeros(nsub, dtype=int) if model_index is None else model_index]
    with np.errstate(divide="ignore"):
        snrs = np.where(noise > 0, scl * mnorm / np.where(noise > 0, noise, 1.0), np.inf)
    ok_ichans = [np.where(w[s] > 0)[0] for s in range(nsub)]
    d = DataBunch(
        arch=None, backend="fake", backend_delay=0.0, bw=float(bw), doppler_factors=np.ones(nsub),
        DM=float(DM_par), dmc=int(bool(dedispersed)), epochs=epochs, filename=outfile or "fake_pulsar",
        flux_prof=None, freqs=np.tile(freqs, (nsub, 1)), frontend="fake", integration_length=float(nsub * tsub),
        masks=None, nbin=nbin, nchan=nchan, noise_stds=sig[:, None], npol=1, nsub=nsub, nu0=float(nu0),
        ok_ichans=ok_ichans, ok_isubs=np.where((w > 0).any(axis=1))[0], parallactic_angles=np.zeros(nsub),
        phases=phases, prof=None, prof_noise=None, prof_SNR=None, Ps=Ps, SNRs=snrs[:, None], source=source,
        state=state, subints=np.asarray(data, dtype=np.float64)[:, None], subtimes=np.full(nsub, float(tsub)),
        telescope=obs, telescope_code=obs, weights=w, raw_subints=raw, dat_scl=dat_scl, dat_offs=dat_offs)
    if outfile is not None:
        save_databunch(outfile, d)
        if not quiet:
            print("Wrote %s (%d subints, %d channels, %d bins)." % (outfile, nsub, nchan, nbin))
    return d


# ---- TOA output (host text formatting; pplib.py:3380-3503) ----------------------------------
def filter_TOAs(TOAs, flag, cutoff, criterion=">=", pass_unflagged=False, return_culled=False):
    """Keep the TOAs whose attribute ``flag`` satisfies ``<criterion> cutoff`` (pplib.py:3380-3407)."""
    import operator
    ops = {">=": operator.ge, ">": operator.gt, "<=": operator.le, "<": operator.lt,
           "==": operator.eq, "!=": operator.ne}
    test = ops[criterion.strip()]
    kept, culled = [], []
    for toa in TOAs:
        if hasattr(toa, flag):
            (kept if test(getattr(toa, flag), cutoff) else culled).append(toa)
        else:
            (kept if pass_unflagged else culled).append(toa)
    return (kept, culled) if return_culled else kept


def _toa_flag_text(flag, value):
    if hasattr(value, "lower"):
        return " -%s %s" % (flag, value)
    if "int" in str(type(value)):
        return " -%s %d" % (flag, value)
    if "_cov" in flag:
        return " -%s %.1e" % (flag, value)
    if "phs" in flag:
        return " -%s %.8f" % (flag, value)
    if "flux" in flag:
        return " -%s %.5f" % (flag, value)
    return " -%s %.3f" % (flag, value)


def toa_line(toa, inf_is_zero=True):
    """One loosely IPTA-formatted TOA line (pplib.py:3465-3497)."""
    freq = 0.0 if (toa.frequency == np.inf and inf_is_zero) else toa.frequency
    tail = "%.15f   %.3f  %s" % (toa.MJD.fracday(), toa.TOA_error, toa.telescope_code)
    line = "%s %.8f %d" % (toa.archive, freq, toa.MJD.intday()) + tail[1:]
    if toa.DM is not None:
        line += " -pp_dm %.7f" % toa.DM
    if toa.DM_error is not None:
        line += " -pp_dme %.7f" % toa.DM_error
    for flag, value in toa.flags.items():
        if value is not None:
            line += _toa_flag_text(flag, value)
    return line


def write_TOAs(TOAs, inf_is_zero=True, SNR_cutoff=0.0, outfile=None, append=True):
    """Write loosely IPTA-formatted TOAs to ``outfile`` or standard output (pplib.py:3445-3503);
    only TOAs with an ``snr`` flag >= SNR_cutoff are written."""
    toas = TOAs if hasattr(TOAs, "__len__") else [TOAs]
    toas = filter_TOAs(toas, "snr", SNR_cutoff, ">=", pass_unflagged=False)
    lines = [toa_line(t, inf_is_zero) for t in toas]
    if outfile is None:
        for ln in lines:
            print(ln)
        return
    with open(outfile, "a" if append else "w") as fh:
        for ln in lines:
            fh.write(ln + "\n")
