"""The FFTFIT guess of pp_fit_batch and the stand-alone pp_fit_phase_shift_batch against a float64 restatement.

Every fit without `init` starts from the FFTFIT guess (pptoas.py:384-456): k_prep (nu_mean, the weight sum, nu_fit),
the row transform (the weighted, DM_guess-dedispersed profile spectrum as float32 partial rows: k_spectra16 at nbin
2048, k_spectra<N, SpecPlan8<N>> at other powers of two, the FROMSPEC rows after k_fwd_any at any other nbin),
k_model_mean / k_model_mean_masked (the template: the mean model over the used channels) and k_guess (the grid, the
polish, the start vector).  The end-of-fit tests cannot see errors here: Newton reaches the same optimum from a
slightly wrong start.  fit_batch(..., max_iter=-1) returns the start vector itself as `params` (with nu_outs = nu_fits
no frequency transform follows), so phi_guess, lag_index and params are compared here with `reference`, which is
pinned on the CPU to orc.toa_core and orc.fit_phase_shift (polish="exact").

The bound is derived from what the device stores, per harmonic k of the profile-times-template product Y_k:
  * 2^-24 per float32 value a row term passes through (the data harmonic, the weight, and with DM_guess the
    rotated value: cos, sin, two products), and (rows per partial + partials) 2^-24 for the float32 sums of the
    partial rows: (stored + R + P) 2^-24 sum_n w_n |d_nk| / W, plus 1e-14 of the row norms for the double FFTs;
  * 2^-24 |mbar_k| |prof_k| for the float32 template;
  * |Y_k| itself for the harmonics above the model's cut-off (DESIGN section 3), which k_guess does not sum.
A grid value moves by at most sum_k |dY_k|, the phase by sum_k 2 pi k |dY_k| / C''(phi*), plus the residual of the
polish stop: k_guess of a fit stops when the Newton step is below polish_tol = 1e-6 and applies that step, which
leaves |C'''/(2 C'')| polish_tol^2; the stand-alone fit stops at 1e-14 without it.
"""
import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests import synth
from tests.test_cpu_cutoff import cutoff_groups
from tests.test_gpu_pass_sums import (NBINS, _pow2, device_model, expected_keep, matched_data, nu_fits_of, row_slots,
                                      template)

U = 2.0 ** -24
POLISH_TOL = 1e-6
WRONG = ("weights ignored", "unmasked template", "dedispersed about nu_fit", "template not scattered",
         "nu_mean over all channels", "last partial row dropped")


def partials(nchan, nbin):
    """(G, NS): channel rows per k_spectra CTA and row slots per CTA (pp_api.cu rows_per_cta, SpecPlan<N>::kSlots);
    partial q = CTA * NS + slot sums rows CTA * G + step * NS + slot"""
    N = row_slots(nbin)
    ns = max(1, 1024 // N)
    g = max(ns, min(32, nchan // 16))
    return -(-g // ns) * ns, ns


def wrap(x):
    """onto [-0.5, 0.5) (pplib.py:2611-2613)"""
    x = np.float64(x)
    if abs(x) >= 0.5:
        x = x % 1
    if x >= 0.5:
        x -= 1.0
    return x


def dwrap(a, b):
    return (np.asarray(a) - np.asarray(b) + 0.5) % 1.0 - 0.5


def nu_of(freqs, used, snrs=None, nu_fits=None, nu_fit_mode=0, all_channels=False):
    """(nu_mean, nu_fit[3]) as k_prep forms them"""
    fu = freqs[used]
    nu_mean = (freqs if all_channels else fu).mean()
    if nu_fit_mode == 1:
        dflt = orc.guess_fit_freq(fu, None if snrs is None else snrs[used])
    else:
        dflt = nu_mean
    nf = np.full(3, dflt) if nu_fits is None else np.where(np.isnan(nu_fits), dflt, nu_fits)
    return nu_mean, nf


def fftfit(Y, eY, L, Ns=100, bounds=None, NU=None, lag=None):
    """Grid and exact polish of C(phi) = -Re sum_k Y_k e^{2 pi i k phi} over harmonics k = 1..L (Y[k-1]); eY bounds
    |dY_k|.  NU: the device sums harmonics 1..NU only.  Returns grid values, argmin, the minimiser phi* next to grid
    point `lag` (default: the argmin), C, C', C'', C''' there and the bounds of a grid value and of phi*."""
    k = np.arange(1, L + 1, dtype=np.float64)
    w = 2 * np.pi * k
    NU = L if NU is None else min(NU, L)
    cut = k > NU
    dY = np.where(cut, np.abs(Y), eY)                      # the cut harmonics: all of |Y_k| is neglected
    grid = np.mgrid[-0.5:0.5:complex(0, Ns)] if bounds is None else np.mgrid[bounds[0]:bounds[1]:complex(0, Ns)]
    vals = -(Y[None, :] * np.exp(1j * np.outer(grid, w))).real.sum(1)
    if bounds is None:      # -1/2 and +1/2 are one phase: k_guess computes one value for both, the first index wins
        vals[-1] = vals[0]
    tgrid = dY.sum() + 1e-15 * (k * np.abs(Y)).sum()      # + the FP64 phasor recurrences of k_guess
    j = int(np.argmin(vals)) if lag is None else int(lag)
    h = grid[1] - grid[0]

    def derivs(x, Y=Y):
        Z = Y * np.exp(1j * w * x)
        return -Z.real.sum(), (w * Z.imag).sum(), (w ** 2 * Z.real).sum(), -(w ** 3 * Z.imag).sum()

    def polish(Y):                 # k_guess's safeguarded Newton on C' = 0 inside the bracket, run to convergence
        x, lo, hi = grid[j], grid[j] - h, grid[j] + h
        for _ in range(100):
            C0, C1, C2, C3 = derivs(x, Y)
            if C1 < 0:
                lo = x
            else:
                hi = x
            xn = x - C1 / C2 if C2 > 0 else np.nan
            if not lo < xn < hi:
                xn = 0.5 * (lo + hi)
            if abs(xn - x) < 1e-16:
                break
            x = xn
        return x
    x = polish(Y)
    C0, C1, C2, C3 = derivs(x)
    tphi = (w * dY).sum() / C2
    # The bracket (two grid steps) can hold several local minima when the template has power up to high harmonics;
    # which one the polish reaches can then hinge on rounding.  Stable: Y moved by its bound (four draws) gives the
    # same minimum.  Otherwise a device phase passes if it is a minimum of C within the bound (`is_minimum`).
    rng = np.random.RandomState(j)
    alt = [polish(Y + dY * np.exp(2j * np.pi * rng.uniform(size=L))) for _ in range(4)]
    stable = max(abs(a - x) for a in alt) <= tphi

    def is_minimum(xd):
        D0, D1, D2, D3 = derivs(xd)
        return D2 > 0 and abs(D1) <= (w * dY).sum() + abs(D3) * POLISH_TOL ** 2

    def minimum_near(xd):
        """the minimum of C that Newton reaches from xd, C, C', C'', C''' there and its phase bound"""
        for _ in range(50):
            D = derivs(xd)
            step = D[1] / D[2]
            xd -= step
            if abs(step) < 1e-16:
                break
        D = derivs(xd)
        return xd, D, (w * dY).sum() / D[2]
    two = np.sort(vals if bounds is not None else vals[:-1])[:2]
    return dict(vals=vals, grid=grid, lag=int(np.argmin(vals)), phi=x, C=(C0, C1, C2, C3), tgrid=tgrid, tphi=tphi,
                gap=two[1] - two[0], stable=stable, is_minimum=is_minimum, minimum_near=minimum_near)


def reference(data, model, freqs, P, used=None, weights=None, snrs=None, nu_fits=None, nu_fit_mode=0, DMg=0.0,
              scat=None, fit_scat=False, log10_tau=False, Ns=100, keep=None, lag=None, wrong=None):
    """The FFTFIT guess of one subint in float64 (pptoas.py:384-456) with its bounds.

    data, model [nchan, nbin]: the values the device transforms (float32-rounded data, decoded int16, the model as
    the plan holds it); used [nchan]: the channel mask; scat: (tau_guess [rot], alpha_guess) of scat_guess; keep:
    the groups of 16 harmonics the model keeps per channel (None: all).  `wrong` names a deliberately wrong
    reference (WRONG).  Returns the nu's, the fftfit dict, the start vector x [5] and its phase bound."""
    nchan, nbin = data.shape
    L = nbin // 2
    used = np.ones(nchan, bool) if used is None else np.asarray(used, bool)
    w = np.ones(nchan) if weights is None or wrong == "weights ignored" else np.asarray(weights, np.float64)
    nu_mean, nu_fit = nu_of(freqs, used, snrs, nu_fits, nu_fit_mode, wrong == "nu_mean over all channels")
    k = np.arange(1, L + 1, dtype=np.float64)
    d0 = np.fft.rfft(data, axis=1)
    d = d0[:, 1:]
    rows = used & np.isfinite(d).all(1)                    # a non-finite row does not enter the profile
    W = w[used].sum()
    if wrong == "last partial row dropped":
        G, ns = partials(nchan, nbin)
        last = [(nchan - 1) // G * G + st * ns + ns - 1 for st in range(G // ns)]
        rows = rows & ~np.isin(np.arange(nchan), last)
    wr = np.where(rows, w, 0.0)
    nu_rot = nu_fit[0] if wrong == "dedispersed about nu_fit" else nu_mean
    shift = orc.Dconst * DMg / P * (freqs ** -2.0 - nu_rot ** -2.0)
    r = np.where(rows[:, None], d, 0.0) * np.exp(2j * np.pi * np.outer(shift, k))
    r[:, -1] = r[:, -1].real                               # irfft keeps the real part of the Nyquist term
    prof = (wr[:, None] * r).sum(0) / W
    m = np.fft.rfft(model, axis=1)[:, 1:]
    tm = np.ones(nchan, bool) if (wrong == "unmasked template" or not used.any()) else used
    mbar = m[tm].mean(0)
    if fit_scat and scat is not None and scat[0] != 0 and wrong != "template not scattered":
        mbar = mbar / (1.0 + 2j * np.pi * k * scat[0])
        mbar[-1] = mbar[-1].real                           # irfft(B rfft(mprof)): the real part at Nyquist
    Y = prof * np.conj(mbar)
    G, ns = partials(nchan, nbin)
    nround = (2 if DMg == 0 else 5) + G // ns + -(-nchan // G) * ns
    adw = (wr[:, None] * np.where(rows[:, None], np.abs(d), 0.0)).sum(0) / W
    nrm = (wr * np.linalg.norm(np.where(rows[:, None], d0, 0.0), axis=1)).sum() / W
    eY = np.abs(mbar) * (nround * U * adw + 1e-14 * nrm) + U * np.abs(mbar) * np.abs(prof)
    NU = None
    if keep is not None and 16 * int(np.max(keep)) < row_slots(nbin):
        NU = (16 * int(np.max(keep))) & ~1
    g = fftfit(Y, eY, L, Ns, NU=NU, lag=lag)
    C3, C2 = g["C"][3], g["C"][2]
    g["tphi"] += abs(C3 / C2) * POLISH_TOL ** 2           # the applied last Newton step below polish_tol
    x = np.zeros(5)
    x[0] = wrap(g["phi"] + orc.Dconst * DMg / P * (nu_fit[0] ** -2.0 - nu_mean ** -2.0))
    x[1] = DMg
    if scat is not None:
        tg = scat[0]
        if log10_tau:
            tg = np.log10(1.0 / nbin if tg == 0 else tg)
        x[3], x[4] = tg, scat[1]
    return dict(nu_mean=nu_mean, nu_fit=nu_fit, g=g, x=x, Y=Y, prof=prof, mbar=mbar)


def standalone_reference(prof, model, noise=None, Ns=100, bounds=None, fft32=False, lag=None, at=None):
    """pp_fit_phase_shift_batch of one float32 profile in float64: the seven outputs and their bounds (pplib.py
    2054-2100).  The profile spectrum is stored as float32 after an FFT in double (or float, fft32), the model's
    after one in double; err2 = noise^2 nbin/2, or the top-quarter power of the stored profile spectrum.
    lag: polish next to this grid point (default: the argmin).  at: where the polish bracket holds several minima
    that rounding can choose between (not g["stable"]), the outputs are those of the minimum next to `at`."""
    nbin = prof.shape[0]
    L = nbin // 2
    F = np.fft.rfft(prof)
    d, m = F[1:], np.fft.rfft(model)[1:]
    ed = U * np.abs(d) + (7 * U * np.log2(nbin) if fft32 else 1e-14) * np.linalg.norm(F)
    Y = d * np.conj(m)
    eY = ed * np.abs(m) + U * np.abs(d) * np.abs(m)
    g = fftfit(Y, eY, L, Ns, bounds, lag=lag)
    if at is not None and not g["stable"]:
        g["phi"], g["C"], g["tphi"] = g["minimum_near"](at)
    k = np.arange(1, L + 1)
    if noise is None:
        top = k >= (3 * (L + 1)) // 4
        err2 = (np.abs(d[top]) ** 2).sum() / (2.0 * L * (L + 1 - (3 * (L + 1)) // 4)) * L
        rerr2 = (2 * np.abs(d[top]) * ed[top]).sum() / (np.abs(d[top]) ** 2).sum()
    else:
        err2, rerr2 = noise ** 2 * L, 0.0
    C0, C1, C2, C3 = g["C"]
    g["tphi"] += 2e-14
    v0, v1 = (np.abs(d) ** 2).sum(), (np.abs(m) ** 2).sum()
    t0 = g["tgrid"] + 0.5 * C2 * g["tphi"] ** 2
    t2 = (4 * np.pi ** 2 * k ** 2 * eY).sum() + abs(C3) * g["tphi"]
    tv0, tv1 = (2 * np.abs(d) * ed).sum(), 2 * U * v1
    r0, r1, r2 = t0 / abs(C0), tv1 / v1, t2 / abs(C2)
    scale = -C0 / v1
    out = dict(phase=(g["phi"], g["tphi"]),
               scale=(scale, abs(scale) * (r0 + r1)),
               scale_err=((err2 / v1) ** 0.5, (err2 / v1) ** 0.5 * 0.5 * (rerr2 + r1)),
               snr=(abs(C0) / (v1 * err2) ** 0.5, abs(C0) / (v1 * err2) ** 0.5 * (r0 + 0.5 * (r1 + rerr2))),
               phase_err=((scale * C2 / err2) ** -0.5, (scale * C2 / err2) ** -0.5 * 0.5 * (r0 + r1 + r2 + rerr2)))
    rc = (v0 - C0 ** 2 / v1) / err2 / (nbin - 2)
    trc = (tv0 + 2 * abs(C0) * t0 / v1 + C0 ** 2 / v1 ** 2 * tv1) / err2 / (nbin - 2) + abs(rc) * rerr2
    out["red_chi2"] = (rc, trc)
    return out, g


# ---- GPU: the guess of fit_batch --------------------------------------------------------------------------------
class Batch(object):
    """One fit_batch(max_iter=-1) call without init and what each subint's reference needs"""

    def __init__(self, label, dev, subs):
        self.label, self.dev, self.subs = label, dev, subs
        self.stable = None

    def refs(self, wrong=None):
        return [reference(lag=int(self.dev["lag_index"][s]), wrong=wrong, **sub) for s, sub in enumerate(self.subs)]

    def ratio(self, wrong=None):
        """max over subints of |device - reference| / bound for phi_guess and the start phase"""
        if self.stable is None:
            self.stable = [r["g"]["stable"] for r in self.refs()]
        worst = 0.0
        for s, r in enumerate(self.refs(wrong)):
            t = r["g"]["tphi"]
            if not self.stable[s] or not t > 0:    # (a wrong reference whose phase has no minimum there: skipped)
                continue
            worst = max(worst, abs(self.dev["phi_guess"][s] - r["g"]["phi"]) / t,
                        abs(dwrap(self.dev["params"][s, 0], r["x"][0])) / (t + 1e-15))
        return worst

    def check(self, max_ambiguous=1):
        dev, ambiguous = self.dev, 0
        refs = self.refs()
        self.stable = [r["g"]["stable"] for r in refs]
        for s, (sub, r) in enumerate(zip(self.subs, refs)):
            # params is the start vector: phase_transform of phi_guess to nu_fit, DM_guess, 0, and tau / alpha
            nu_mean, nu_fit = r["nu_mean"], r["nu_fit"]
            ph = wrap(dev["phi_guess"][s] + orc.Dconst * sub["DMg"] / sub["P"] * (nu_fit[0] ** -2.0 - nu_mean ** -2.0))
            assert abs(dwrap(dev["params"][s, 0], ph)) < 1e-12, (self.label, s, dev["params"][s, 0], ph)
            assert dev["params"][s, 1] == sub["DMg"] and dev["params"][s, 2] == 0.0
            assert np.allclose(dev["params"][s, 3:], r["x"][3:], rtol=1e-12, atol=1e-14), (dev["params"][s], r["x"])
            g = r["g"]
            if g["gap"] > 2 * g["tgrid"]:
                assert dev["lag_index"][s] == g["lag"], (self.label, s, dev["lag_index"][s], g["lag"])
            else:
                ambiguous += 1
            if not g["stable"]:    # the polish may reach another minimum of the bracket: it must be one
                ambiguous += 1
                assert g["is_minimum"](dev["phi_guess"][s]), (self.label, s, dev["phi_guess"][s], g["phi"])
            elif abs(dev["phi_guess"][s] - g["phi"]) > g["tphi"]:
                print(self.label, "subint", s, "lag", dev["lag_index"][s], g["lag"], "phi", dev["phi_guess"][s], g["phi"],
                      "bound", g["tphi"])
        ratio = self.ratio()
        print("%-48s phase |dev - ref| / bound %.2e  bound %.1e turn  ambiguous lags or minima %d"
              % (self.label, ratio, max(r["g"]["tphi"] for r in refs), ambiguous))
        assert ratio <= 1.0, (self.label, ratio)
        assert ambiguous <= max_ambiguous, (self.label, ambiguous)
        return ratio


def points_for(freqs, P, nsub, span=0.45):
    """(phi, DM_guess) per subint in the nu_mean frame: DM_guess = 0, DM_guess rotating the band edges by up to
    `span` turn either way, and a phase near 0.5 whose transform to nu_fit crosses +-0.5"""
    nm = freqs.mean()
    g = orc.Dconst * (freqs ** -2.0 - nm ** -2.0) / P
    sp = np.abs(g).max() or 1.0
    base = [(0.13, 0.0), (-0.31, span / sp), (0.27, -span / sp), (0.4985, -0.6 * span / sp)]
    return [base[s % 4] for s in range(nsub)]


def guess_data(model, freqs, P, pts, seed, amp=1.0, sigma=1.5):
    """float32 data whose subint s is the model at (phi_s, DM_s) about nu_mean, plus noise"""
    nm = freqs.mean()
    x = np.array([[p, dm, 0.0, 0.0, 0.0] for p, dm in pts])
    return matched_data(model, freqs, P, np.array([nm, nm, nm]), x, seed=seed, amp=amp, sigma=sigma)


def run_batch(pl, data, P, subs, label, **kw):
    """fit_batch(max_iter=-1, nu_outs = nu_fits) and the Batch to check"""
    nsub = len(subs)
    nu_outs = np.stack([nu_of(s["freqs"], np.ones(len(s["freqs"]), bool) if s.get("used") is None else s["used"],
                              s.get("snrs"), s.get("nu_fits"), s.get("nu_fit_mode", 0))[1] for s in subs])
    nu_fits = None if subs[0].get("nu_fits") is None else np.stack([s["nu_fits"] for s in subs])
    DMg = np.array([s["DMg"] for s in subs])
    dev = pl.fit_batch(data, P, nu_fits=nu_fits, nu_outs=nu_outs, DM_guess=DMg, max_iter=-1,
                       nu_fit_mode=subs[0].get("nu_fit_mode", 0), **kw)
    assert (dev["nfeval"] == 1).all()
    assert np.array_equal(dev["nu_out"][:, 0], nu_outs[:, 0])
    return Batch(label, dev, subs)


def sweep_batch(nbin, kind, nchan=37, nsub=4, seed=0):
    from pulseportraiture_b200.engine import WidebandPlan
    freqs, model = template(kind, nchan, nbin)
    P = synth.P_EXAMPLE
    pts = points_for(freqs, P, nsub)
    amp, sigma = (1.0, 1.5) if kind == "analytic" else (0.3, 1.0)
    data = guess_data(model, freqs, P, pts, seed=seed + nbin + nchan, amp=amp, sigma=sigma)
    weights = np.random.RandomState(seed + 3).uniform(0.5, 1.5, (nsub, nchan))
    nf = nu_fits_of(freqs)
    dm = device_model(model, nbin)
    keep = expected_keep(dm, nbin)
    subs = [dict(data=data[s].astype(np.float64), model=dm, freqs=freqs, P=P, weights=weights[s], nu_fits=nf,
                 DMg=pts[s][1], keep=keep) for s in range(nsub)]
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        return run_batch(pl, data, P, subs, "sweep nbin %d nchan %d %s" % (nbin, nchan, kind), weights=weights)


_BATCHES = {}


def cached(key, fn, *a):
    if key not in _BATCHES:
        _BATCHES[key] = fn(*a)
    return _BATCHES[key]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["analytic", "white"])
@pytest.mark.parametrize("nbin", NBINS)
def test_guess_row_plan_sweep(nbin, kind):
    """Every row transform with weights and DM_guess (k_spectra16<0,1,0> at 2048, SpecPlan8<N>, FROMSPEC), the
    template with its cut-off (analytic) or every harmonic and the Nyquist term (white), 37 channels"""
    cached(("sweep", nbin, kind), sweep_batch, nbin, kind).check(max_ambiguous=3 if kind == "white" else 1)


@pytest.mark.gpu
@pytest.mark.parametrize("nchan,nbin", [(1, 2048), (1, 1000), (512, 2048), (4096, 1024)])
def test_guess_channel_counts(nchan, nbin):
    """one channel, and 512 x 2048 / 4096 x 1024: 16 and 256 float32 partial rows"""
    cached(("sweep", nbin, "analytic", nchan), sweep_batch, nbin, "analytic", nchan, 2).check()


@pytest.mark.gpu
@pytest.mark.parametrize("nbin", [512, 2048, 1000])
def test_guess_masks_and_options(nbin):
    """a channel mask (the masked mean template, nu_mean over the used channels), a non-finite row, DM_guess,
    nu_fit_mode 1 with snrs and nu_fit_mode 0 without nu_fits (nu_fit = nu_mean)"""
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 4
    freqs, model = template("analytic", nchan, nbin)
    P = synth.P_EXAMPLE
    pts = points_for(freqs, P, nsub)
    data = guess_data(model, freqs, P, pts, seed=300 + nbin)
    data[2, 5, 17] = np.nan
    mask = np.ones((nsub, nchan), np.uint8)
    mask[1, :9] = 0
    mask[3, 20:] = 0
    rng = np.random.RandomState(4)
    weights, snrs = rng.uniform(0.5, 1.5, (nsub, nchan)), rng.uniform(1.0, 30.0, (nsub, nchan))
    dm = device_model(model, nbin)
    keep = expected_keep(dm, nbin)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        for mode in (0, 1):
            subs = [dict(data=data[s].astype(np.float64), model=dm, freqs=freqs, P=P, used=mask[s] == 1,
                         weights=weights[s], snrs=snrs[s] if mode else None, nu_fit_mode=mode, DMg=pts[s][1],
                         keep=keep) for s in range(nsub)]
            b = run_batch(pl, data, P, subs, "options nbin %d nu_fit_mode %d" % (nbin, mode), chan_mask=mask,
                          weights=weights, snrs=snrs if mode else None)
            assert np.isfinite(b.dev["phi_guess"]).all()
            b.check()
            _BATCHES[("options", nbin, mode)] = b


@pytest.mark.gpu
@pytest.mark.parametrize("log10_tau", [False, True])
@pytest.mark.parametrize("kind", ["analytic", "white"])
@pytest.mark.parametrize("nbin", [64, 512, 2048, 1000])
def test_guess_scattered_template(nbin, kind, log10_tau):
    """fit_flags (1,1,0,1,1) with scat_guess: the template scattered by tau_guess (pptoas.py:444-447), one subint
    with tau_guess = 0 (the start log10 tau is log10(1/nbin))"""
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 4
    freqs, model = template(kind, nchan, nbin)
    P = synth.P_EXAMPLE
    pts = points_for(freqs, P, nsub)
    amp, sigma = (1.0, 1.5) if kind == "analytic" else (0.3, 1.0)
    data = guess_data(model, freqs, P, pts, seed=500 + nbin, amp=amp, sigma=sigma)
    scat = np.array([[0.4 / (2 * np.pi * nbin / 2), -4.0], [0.0, -3.5], [2.0 / (2 * np.pi * nbin / 2), -4.4],
                     [3e-3, -4.0]])
    nf = nu_fits_of(freqs)
    dm = device_model(model, nbin)
    keep = expected_keep(dm, nbin)
    subs = [dict(data=data[s].astype(np.float64), model=dm, freqs=freqs, P=P, nu_fits=nf, DMg=pts[s][1],
                 scat=scat[s], fit_scat=True, log10_tau=log10_tau, keep=keep) for s in range(nsub)]
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        b = run_batch(pl, data, P, subs, "scattered nbin %d %s log10_tau %s" % (nbin, kind, log10_tau),
                      fit_flags=(1, 1, 0, 1, 1), scat_guess=scat, log10_tau=log10_tau)
    b.check(max_ambiguous=3 if kind == "white" else 1)
    _BATCHES[("scat", nbin, kind, log10_tau)] = b


@pytest.mark.gpu
@pytest.mark.parametrize("nbin", [512, 2048])
def test_guess_grid_sizes_and_align(nbin):
    """Ns = 37, 100 and Ns = nbin with align=True (the ppalign path: k_spectra16<0,1,1> at 2048): the grid values
    of a fine grid lie close together, so near-ties are counted"""
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 4
    freqs, model = template("white", nchan, nbin)
    P = synth.P_EXAMPLE
    pts = points_for(freqs, P, nsub)
    data = guess_data(model, freqs, P, pts, seed=600 + nbin, amp=0.3, sigma=1.0)
    nf = nu_fits_of(freqs)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        for Ns, align in ((37, False), (100, False), (nbin, True)):
            subs = [dict(data=data[s].astype(np.float64), model=model, freqs=freqs, P=P, nu_fits=nf, DMg=pts[s][1],
                         Ns=Ns) for s in range(nsub)]
            run_batch(pl, data, P, subs, "Ns %d align %s nbin %d" % (Ns, align, nbin), Ns=Ns, align=align).check(max_ambiguous=3)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "f64", "i16", "torch"])
@pytest.mark.parametrize("nbin", [2048, 1536])
def test_guess_inputs(nbin, dtype):
    """float32, float64 (rounded on the device), int16 (decoded in float32) and CUDA float32 data"""
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 4
    freqs, model = template("analytic", nchan, nbin)
    P = synth.P_EXAMPLE
    pts = points_for(freqs, P, nsub)
    data = guess_data(model, freqs, P, pts, seed=700 + nbin)
    kw, values = {}, data.astype(np.float64)
    if dtype == "f64":
        arg = data.astype(np.float64) + np.random.RandomState(3).normal(0.0, 1e-5, data.shape)
        values = arg.astype(np.float32).astype(np.float64)
    elif dtype == "i16":
        scl = np.full((nsub, nchan), 0.01, np.float32)
        offs = np.full((nsub, nchan), 0.5, np.float32)
        arg = np.clip(np.round((data - offs[..., None]) / scl[..., None]), -32768, 32767).astype(np.int16)
        values = (arg.astype(np.float32) * scl[..., None] + offs[..., None]).astype(np.float64)
        kw = dict(dat_scl=scl, dat_offs=offs)
    elif dtype == "torch":
        arg = torch.from_numpy(data).cuda()
    else:
        arg = data
    nf = nu_fits_of(freqs)
    dm = device_model(model, nbin)
    keep = expected_keep(dm, nbin)
    subs = [dict(data=values[s], model=dm, freqs=freqs, P=P, nu_fits=nf, DMg=pts[s][1], keep=keep)
            for s in range(nsub)]
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        run_batch(pl, arg, P, subs, "inputs nbin %d %s" % (nbin, dtype), **kw).check()


def models_batch(nbin, masked):
    """three models with their own tables, an interleaved model_index (tmpl_by_model, nused_of); with a mask the
    per-subint masked templates of each subint's own model"""
    from pulseportraiture_b200.engine import WidebandPlan
    from tests.test_gpu_multimodel import NCHAN, TABLES, _models
    models, freqs = _models(nbin)
    index = np.array([0, 1, 2, 2, 0, 1, 1, 2, 0], dtype=np.int32)
    nsub = len(index)
    P = np.array([TABLES[m][3] * (1.0 + 1e-7 * s) for s, m in enumerate(index)])
    pts = [points_for(freqs[m], P[s], 4)[s % 4] for s, m in enumerate(index)]
    data = np.concatenate([guess_data(models[m], freqs[m], P[s], [pts[s]], seed=1300 + s)
                           for s, m in enumerate(index)])
    mask = np.ones((nsub, NCHAN), np.uint8)
    if masked:
        mask[1, :12] = 0
        mask[4, 30:] = 0
        mask[7, ::3] = 0
    nf = np.stack([nu_fits_of(freqs[m]) for m in index])
    dms = [device_model(models[m], nbin) for m in range(3)]
    keeps = [expected_keep(dms[m], nbin) for m in range(3)]
    subs = [dict(data=data[s].astype(np.float64), model=dms[m], freqs=freqs[m], P=P[s], used=mask[s] == 1,
                 nu_fits=nf[s], DMg=pts[s][1], keep=keeps[m]) for s, m in enumerate(index)]
    with WidebandPlan(NCHAN, nbin) as pl:
        pl.set_models(models, freqs)
        return run_batch(pl, data, P, subs, "models nbin %d masked %s" % (nbin, masked), model_index=index,
                         chan_mask=mask if masked else None)


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("nbin", [512, 2048, 1536])
def test_guess_per_subint_models(nbin, masked):
    """pp_fit_batch_models: each subint's guess from its own model's (masked) mean template, cut-off and table"""
    cached(("models", nbin, masked), models_batch, nbin, masked).check()


@pytest.mark.gpu
def test_the_guess_bound_rejects_wrong_references():
    """The same device outputs against deliberately wrong references: each must miss by 10 times the bound in at
    least one case, so that a loosened bound shows here"""
    runs = [b for b in _BATCHES.values() if isinstance(b, Batch)]
    if len(runs) < 8:                                        # run alone: compute the cases it needs
        runs = [cached(("sweep", 512, "analytic"), sweep_batch, 512, "analytic"),
                cached(("sweep", 2048, "white"), sweep_batch, 2048, "white"),
                cached(("models", 512, True), models_batch, 512, True),
                cached(("models", 2048, True), models_batch, 2048, True)]
        for nbin in (64, 512):
            test_guess_scattered_template(nbin, "white", False)
        test_guess_masks_and_options(512)
        runs = [b for b in _BATCHES.values() if isinstance(b, Batch)]
    misses = {}
    for wrong in WRONG:
        worst = 0.0
        for b in runs:
            try:
                worst = max(worst, b.ratio(wrong))
            except (ZeroDivisionError, FloatingPointError):
                continue
        misses[wrong] = worst
    print(misses)
    weak = {k: v for k, v in misses.items() if not v >= 10.0}
    assert not weak, weak


# ---- GPU: the stand-alone FFTFIT ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bits", [64, 32])
@pytest.mark.parametrize("nbin", [64, 128, 4096, 66, 1000, 4094])
def test_standalone_fftfit(nbin, bits):
    """pp_fit_phase_shift_batch (k_rfft_rows in double or float, k_guess with polish_tol 1e-14): all seven outputs at
    nbin and FFT precisions the golden tests do not reach, with nmodel = 1, a divisor of n and n, noise given and
    measured, the default grid and general bounds"""
    from pulseportraiture_b200.engine import WidebandPlan
    n = 6
    rng = np.random.RandomState(nbin + bits)
    _, base = template("analytic", 3, nbin)
    white = rng.normal(0.0, 1.0, (3, nbin))
    shifts = np.array([0.21, -0.37, 0.4999, -0.05, 0.33, -0.49])
    cases = []
    for nmodel in (1, 3, n):
        mods = np.concatenate([base[:2], white[:1]])[np.arange(nmodel) % 3].astype(np.float32)
        profs = np.stack([np.fft.irfft(np.fft.rfft(mods[i % nmodel].astype(np.float64)) *
                                       np.exp(-2j * np.pi * shifts[i] * np.arange(nbin // 2 + 1)), n=nbin)
                          for i in range(n)]) * 2.0 + rng.normal(0.0, 1.0, (n, nbin))
        profs = profs.astype(np.float32)
        for noise in (None, rng.uniform(0.8, 1.2, n)):
            for Ns, bounds in ((100, None), (57, (-0.4, 0.55))):
                cases.append((nmodel, mods, profs, noise, Ns, bounds))
    worst, ambiguous = {}, 0
    with WidebandPlan(1, nbin) as pl:
        pl.set_fft_precision(bits)
        for nmodel, mods, profs, noise, Ns, bounds in cases:
            kw = dict(Ns=Ns) if bounds is None else dict(Ns=Ns, bounds=bounds)
            r = pl.fit_phase_shift_batch(profs, mods if nmodel > 1 else mods[0], noise=noise, **kw)
            for i in range(n):
                ref, g = standalone_reference(profs[i].astype(np.float64), mods[i % nmodel].astype(np.float64),
                                              None if noise is None else noise[i], Ns, bounds, fft32=bits == 32,
                                              lag=r["lag_index"][i], at=r["phase"][i])
                if g["gap"] > 2 * g["tgrid"]:
                    assert r["lag_index"][i] == g["lag"], (nbin, bits, nmodel, i)
                else:
                    ambiguous += 1
                if not g["stable"]:       # (white templates at large nbin: several minima in the bracket)
                    ambiguous += 1
                    # the device phase is a minimum of the restated objective inside the polish bracket
                    h = g["grid"][1] - g["grid"][0]
                    assert g["is_minimum"](r["phase"][i]) and abs(g["phi"] - g["grid"][r["lag_index"][i]]) <= h
                for name, (want, tol) in ref.items():
                    worst[name] = max(worst.get(name, 0.0), abs(r[name][i] - want) / tol)
    print("standalone nbin %d fft %d: %s; ambiguous lags or minima %d of %d"
          % (nbin, bits, " ".join("%s %.1e" % kv for kv in worst.items()), ambiguous, n * len(cases)))
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad
    assert ambiguous <= 6, ambiguous


# ---- CPU: the restatement against the oracle ----------------------------------------------------------------------
def _cpu_subint(nchan=8, nbin=128, seed=31, DMg=2e-3, phi=0.2):
    freqs, model = synth.example_model(nchan, nbin, 1500.0, 800.0)
    P = synth.P_EXAMPLE
    nm = freqs.mean()
    x = np.array([[phi, DMg, 0.0, 0.0, 0.0]])
    data = matched_data(model, freqs, P, np.array([nm, nm, nm]), x, seed=seed)[0].astype(np.float64)
    return freqs, model, data, P


@pytest.mark.parametrize("opts", [
    dict(),
    dict(DMg=3e-3, weights=True),
    dict(DMg=-2e-3, nu_fit_mode=1),
    dict(DMg=1e-3, scat=(0.01, -4.0), log10_tau=False),
    dict(DMg=1e-3, scat=(0.0, -4.0), log10_tau=True),
    dict(DMg=-0.3, Ns=37, phi=0.4995),
])
def test_restatement_matches_toa_core(opts):
    """the guess of orc.toa_core (rotate_data, np.average, the mean model, irfft(B rfft(mprof)), fit_phase_shift
    polished exactly, phase_transform with mod) equals the restatement: lag, phi_guess and the start vector"""
    opts = dict(opts)
    DMg, phi = opts.pop("DMg", 0.0), opts.pop("phi", 0.2)
    freqs, model, data, P = _cpu_subint(DMg=DMg, phi=phi)
    nchan = len(freqs)
    rng = np.random.RandomState(8)
    weights = rng.uniform(0.5, 1.5, nchan) if opts.pop("weights", False) else None
    snrs = rng.uniform(1.0, 30.0, nchan)
    mode = opts.pop("nu_fit_mode", 0)
    scat, log10_tau = opts.pop("scat", None), opts.pop("log10_tau", False)
    Ns = opts.pop("Ns", 100)
    nu_fits = None if mode == 1 else nu_fits_of(freqs)
    flags = (1, 1, 0, 1, 1) if scat is not None else (1, 1, 0, 0, 0)
    _, phi_guess, nfs = orc.toa_core(data, model, P, freqs, np.ones(nchan), weights=weights,
                                     SNRs=snrs if mode else None, DM_stored=DMg, fit_flags=flags,
                                     nu_fits=nu_fits, log10_tau=log10_tau,
                                     tau_guess=0.0 if scat is None else scat[0],
                                     alpha_guess=0.0 if scat is None else scat[1], Ns=Ns, polish="exact")
    r = reference(data, model, freqs, P, weights=weights, snrs=snrs if mode else None, nu_fits=nu_fits,
                  nu_fit_mode=mode, DMg=DMg, scat=scat, fit_scat=scat is not None, log10_tau=log10_tau, Ns=Ns)
    assert np.allclose(r["nu_fit"], nfs, rtol=1e-15, atol=0)
    assert abs(dwrap(r["x"][0], phi_guess)) < 1e-9, (r["x"][0], phi_guess)   # (Brent stops at ~1e-11 + 1e-14 |x|)
    rot_prof = np.average(orc.rotate_data(data, 0.0, DMg, P, freqs, freqs.mean()), axis=0, weights=weights)
    lag, _, vals = orc.fit_phase_shift_grid(rot_prof, model.mean(0) if scat is None or scat[0] == 0 else
                                            np.fft.irfft(np.fft.rfft(model.mean(0)) /
                                                         (1 + 2j * np.pi * np.arange(len(rot_prof) // 2 + 1) *
                                                          scat[0])), Ns=Ns)
    assert r["g"]["lag"] == lag
    mine = r["g"]["vals"]
    inv_err2 = (vals * mine).sum() / (mine * mine).sum()
    assert np.allclose(mine * inv_err2, vals, rtol=1e-10, atol=1e-10 * np.abs(vals).max())
    if scat is not None:
        tg = scat[0] if not log10_tau else np.log10(1.0 / data.shape[1] if scat[0] == 0 else scat[0])
        assert r["x"][3] == tg and r["x"][4] == scat[1]
    assert 0 < r["g"]["tphi"] < 1e-5


@pytest.mark.parametrize("noise", [None, 1.1])
@pytest.mark.parametrize("bounds", [None, (-0.3, 0.45)])
@pytest.mark.parametrize("nbin", [64, 1000])
def test_standalone_restatement_matches_fit_phase_shift(nbin, bounds, noise):
    """standalone_reference equals orc.fit_phase_shift(polish="exact") on all seven outputs"""
    rng = np.random.RandomState(nbin)
    _, model = template("analytic", 2, nbin)
    prof = (2.0 * np.roll(model[1], 7) + rng.normal(0.0, 1.0, nbin)).astype(np.float32).astype(np.float64)
    b = (-0.5, 0.5) if bounds is None else bounds
    o = orc.fit_phase_shift(prof, model[1], noise=noise, bounds=b, Ns=57, polish="exact")
    ref, g = standalone_reference(prof, model[1], noise, 57, bounds)
    assert g["lag"] == o.lag_index
    for name, (want, tol) in ref.items():
        # (the oracle's Brent polish stops at ~1e-11 + 1e-14 |x| of the phase)
        # (phase_err is C'' at that phase: |C'''/C''| 1e-9 relative)
        rtol = 1e-9 + abs(g["C"][3] / g["C"][2]) * 1e-9 if name == "phase_err" else 1e-9
        assert np.isclose(want, getattr(o, name), rtol=rtol, atol=1e-9 if name == "phase" else 0), (name, want)
        assert 0 < tol < 1e-4 * abs(want) + 1e-6, (name, tol)


def test_restatement_bound_covers_float32_storage_and_cutoff():
    """Rounding the profile and the template to float32, and dropping the harmonics above the cut-off of an analytic
    float64 model, move the phase by less than the bound"""
    freqs, model, data, P = _cpu_subint(nchan=16, nbin=1024, DMg=3e-3)
    keep = cutoff_groups(model)
    assert keep.max() < 1024 // 32
    r = reference(data, model, freqs, P, DMg=3e-3, keep=keep)
    Y32 = r["prof"].astype(np.complex64).astype(np.complex128) * np.conj(r["mbar"].astype(np.complex64))
    NU = 16 * int(keep.max())
    Y32[NU:] = 0
    g = fftfit(Y32, np.zeros_like(np.abs(Y32)), len(Y32), lag=r["g"]["lag"])
    assert 0 < abs(g["phi"] - r["g"]["phi"]) < r["g"]["tphi"]


def test_wrong_references_differ_on_the_cpu():
    """each wrong reference changes the restated guess of a masked, weighted, dedispersed, scattered case (so the
    GPU test of the bound can see it)"""
    freqs, model, data, P = _cpu_subint(nchan=48, nbin=512, DMg=0.3)
    used = np.ones(48, bool)
    used[:9] = False
    w = np.random.RandomState(2).uniform(0.5, 1.5, 48)
    kw = dict(used=used, weights=w, nu_fits=nu_fits_of(freqs), DMg=0.3, scat=(0.3 / (2 * np.pi * 256), -4.0),
              fit_scat=True)
    r = reference(data, model, freqs, P, **kw)
    for wrong in WRONG:
        rw = reference(data, model, freqs, P, wrong=wrong, **kw)
        miss = max(abs(rw["g"]["phi"] - r["g"]["phi"]), abs(dwrap(rw["x"][0], r["x"][0])))
        assert miss > 10 * r["g"]["tphi"], wrong
