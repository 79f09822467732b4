"""The per-channel sums of the pass kernels, k_pass2 and k_pass5, against a float64 restatement at a chosen point.

Everything a TOA is made of passes through one chain: the row transform stores the cross-spectrum X = d conj(m)
(k_spectra<N, SpecPlan8<N>> for power-of-two nbin, k_spectra16 at nbin 2048, the FROMSPEC rows of k_spectra after
k_fwd_any for any other nbin), then k_pass2 sums C, C', C'', C''', C'''' per channel for the (phi, DM) solver, or k_pass5
the nine sums C, C_th, C_thth, C_t, C_tt, C_tht, S, S_t, S_tt of the general solver (pptoaslib.py:318-523).
fit_batch(..., max_iter=-1) evaluates one pass at `init` and runs the epilogue there, so pp_fit_out_t.chan_sums and the
epilogue outputs can be compared element by element with a plain numpy restatement at exactly that point.  The end-of-fit
parity tests cannot see most errors of these sums: Newton converges to the zero of the gradient wherever the Hessian-side
sums come from.

The bound comes from how X is stored (csrc/kernels.cuh k_spectra, csrc/spectra16.cuh).  Slot k < LoK = min(N, 64)
(slot 0 = the Nyquist term of a power-of-two row) holds a double product as float32 plus its float32 residual: about
2^-48 relative.  Other slots hold a float product of float32 d and float32 conj(m) (N >= 512) or one float32 rounding
of a double product (N < 512): at most 4 float32 roundings, 2^-22 |d||m| per component.  The double FFTs of data and
model add about u log2(nbin) of the row's norm to every harmonic.  Per element

  eps_nk = 2^-22 |d_nk||m_nk| [slot >= LoK] + 1e-12 |d_nk||m_nk| + 1e-14 (||d_n|| |m_nk| + |d_nk| ||m_n||)

and a sum whose terms are f_k X_nk gets sum_k |f_k| eps_nk / sigma_F^2.  The 1e-12 term also covers the phase: theta_n
is rounded to ~1e-15 turn on either side, 2 pi 64 1e-15 < 1e-12 in the low slots.  Sums of the double |m|^2 (S, S_t,
S_tt, the (phi, DM) p_n) and the data power Sd get 1e-12 relative.  The epilogue values at x (chi2, snr, scales,
channel_snrs; for (phi, DM) also the zero-covariance frequency and cov = inv(H/2)) get these bounds carried through
to first order.
"""
import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests import synth
from tests.test_cpu_cutoff import cutoff_groups

LOK = 64
GEN = ("C", "Cth", "Cthth", "Ct", "Ctt", "Ctht", "S", "St", "Stt")
PHIDM = ("C", "C1", "C2", "C3", "C4")
NU0, BW = 1500.0, 800.0


def _pow2(nbin):
    return nbin & (nbin - 1) == 0


def row_slots(nbin):
    """slots per stored row: nbin/2 for powers of two, else the smallest power of two above nbin/2 (k_fwd_any)"""
    if _pow2(nbin):
        return nbin // 2
    n = 1
    while n < nbin // 2 + 1:
        n *= 2
    return n


def kernel_path(nbin):
    if nbin == 2048:
        return "k_spectra16"
    return "SpecPlan8<%d>" % (nbin // 2) if _pow2(nbin) else "FROMSPEC<%d>" % row_slots(nbin)


def reference(data, model, sigma, P, freqs, nu_fits, x, log10_tau=False, keep=None,
              no_xlo=False, drop_nyquist=False, drop_k=None, sf2_npad=False, tau_ref_dm=False, stored=False):
    """One subint's pass sums at x = (phi, DM, GM, tau, alpha), in float64, with their tolerances.

    data, model: [nchan, nbin] float64 holding exactly the values the device transforms; sigma: [nchan] time-domain
    noise (0 = channel unused); nu_fits: (nu_DM, nu_GM, nu_tau); keep: [nchan] leading groups of 16 harmonics the
    harmonic cut-off keeps (None: all; the Nyquist term counts only when all are kept).
    The keyword arguments after `keep` make deliberately wrong references (the tolerance must reject them), except
    `stored`: X as the device stores it (float32 product above LoK), which the tolerance must accept.
    Returns gen [nchan, 9] (k_pass5 layout), phidm [nchan, 5] (k_pass2 layout), S [nchan] (p_n / sigma_F^2 over every
    harmonic, what the (phi, DM) epilogue divides by), Sd [nchan], each with its tolerance t*.
    """
    nchan, nbin = data.shape
    L = nbin // 2
    N = row_slots(nbin)
    d0 = np.fft.rfft(data, axis=1)
    m0 = np.fft.rfft(model, axis=1)
    d, m = d0[:, 1:], m0[:, 1:]                           # harmonics 1..L, DC dropped
    k = np.arange(1, L + 1, dtype=np.float64)
    w = 2.0 * np.pi * k
    # slot of harmonic k: k (< N), the Nyquist term of a power-of-two row sits in slot 0
    lo = (k < min(N, LOK)) | ((k == L) & _pow2(nbin))
    kept = np.ones((nchan, L), dtype=bool)
    if keep is not None:
        for n in range(nchan):
            if keep[n] < L // 16:
                kept[n, 16 * keep[n] - 1:] = False        # harmonics >= 16 keep, the Nyquist term included
    if drop_nyquist:
        kept[:, L - 1] = False
    if drop_k is not None:
        kept[:, drop_k - 1] = False
    X = d * np.conj(m)
    if stored:
        X[:, ~lo] = d[:, ~lo].astype(np.complex64) * np.conj(m[:, ~lo].astype(np.complex64))
    if no_xlo:
        X[:, lo] = X[:, lo].astype(np.complex64)
    used = sigma > 0
    sF2 = np.where(used, sigma ** 2 * (N if sf2_npad else L), 1.0)
    phi, DM, GM, tau, alpha = x
    nD, nG, nT = nu_fits
    gD = orc.Dconst * (freqs ** -2.0 - nD ** -2.0) / P
    gG = orc.Dconst ** 2 * (freqs ** -4.0 - nG ** -4.0) / P
    theta = phi + DM * gD + GM * gG
    theta -= np.rint(theta)
    Z = np.where(kept, X * np.exp(2j * np.pi * np.outer(theta, k)), 0.0)
    taun = (10.0 ** tau if log10_tau else tau) * (freqs / (nD if tau_ref_dm else nT)) ** alpha
    B = 1.0 / (1.0 + 1j * np.outer(taun, w))
    cB = np.conj(B)
    Z1 = Z * cB
    Z2 = Z1 * cB
    Z3 = Z2 * cB
    M = np.where(kept, np.abs(m) ** 2, 0.0)
    q = np.abs(B) ** 2
    tq = taun[:, None] * q
    gen = np.stack([Z1.real.sum(1), -(w * Z1.imag).sum(1), -(w ** 2 * Z1.real).sum(1),
                    -(w * Z2.imag).sum(1), -2.0 * (w ** 2 * Z3.real).sum(1), -(w ** 2 * Z2.real).sum(1),
                    (q * M).sum(1), -2.0 * (w ** 2 * tq * q * M).sum(1), 2.0 * (w ** 2 * q * q * (3 - 4 * q) * M).sum(1)],
                   axis=1)
    phidm = np.stack([Z.real.sum(1), -(w * Z.imag).sum(1), -(w ** 2 * Z.real).sum(1),
                      (w ** 3 * Z.imag).sum(1), (w ** 4 * Z.real).sum(1)], axis=1)
    ad, am = np.abs(d), np.abs(m)
    nd, nm = np.linalg.norm(d0, axis=1), np.linalg.norm(m0, axis=1)     # the FFT error scales with the whole row
    eps = (2.0 ** -22 * ~lo + 1e-12) * ad * am + 1e-14 * (nd[:, None] * am + ad * nm[:, None])
    eps = np.where(kept, eps, 0.0)
    aB = np.abs(B)
    fgen = [aB, w * aB, w ** 2 * aB, w * aB ** 2, 2 * w ** 2 * aB ** 3, w ** 2 * aB ** 2]
    tgen = np.stack([(f * eps).sum(1) for f in fgen] +
                    [1e-12 * (q * M).sum(1), 1e-12 * (2 * w ** 2 * tq * q * M).sum(1),
                     1e-12 * (2 * w ** 2 * q * q * np.abs(3 - 4 * q) * M).sum(1)], axis=1)
    tphidm = np.stack([(w ** p * eps).sum(1) for p in range(5)], axis=1)
    S = (am ** 2).sum(1)
    Sd = (ad ** 2).sum(1)
    out = dict(gen=gen, tgen=tgen, phidm=phidm, tphidm=tphidm, S=S, tS=1e-12 * S, Sd=Sd, tSd=1e-12 * Sd)
    for key, v in out.items():
        v = v / (sF2[:, None] if v.ndim == 2 else sF2)
        out[key] = np.where(used[:, None] if v.ndim == 2 else used, v, 0.0)
    out["used"] = used
    return out


def epilogue(r, solver, freqs, P):
    """The epilogue values at x from the reference sums, each with its first-order tolerance: chi2, snr, scales,
    channel_snrs (k_update5 / k_update2 with max_iter < 0) and, for (phi, DM), nu_zero and cov = inv(H/2)
    (pplib.py:1352-1391, 2187-2190)."""
    u = r["used"]
    if solver == "phidm":
        C, tC = r["phidm"][u, 0], r["tphidm"][u, 0]
        S, tS = r["S"][u], r["tS"][u]
    else:
        C, tC = r["gen"][u, 0], r["tgen"][u, 0]
        S, tS = r["gen"][u, 6], r["tgen"][u, 6]
    a2 = C * C / S
    ta2 = 2 * np.abs(C) * tC / S + a2 * tS / S
    snr = np.sqrt(a2.sum())
    out = dict(chi2=(r["Sd"][u].sum() - a2.sum(), r["tSd"][u].sum() + ta2.sum()),
               snr=(snr, 0.5 * ta2.sum() / snr))
    sc, csn = np.zeros(len(u)), np.zeros(len(u))
    tsc, tcsn = np.zeros(len(u)), np.zeros(len(u))
    sc[u], tsc[u] = C / S, tC / S + np.abs(C) * tS / S ** 2
    csn[u], tcsn[u] = C / np.sqrt(S), tC / np.sqrt(S) + 0.5 * np.abs(C) * tS / S ** 1.5
    out["scales"], out["channel_snrs"] = (sc, tsc), (csn, tcsn)
    if solver == "phidm" and u.sum() > 1:       # (one channel: phi and DM are degenerate, H is singular)
        C1, C2 = r["phidm"][u, 1], r["phidm"][u, 2]
        tC1, tC2 = r["tphidm"][u, 1], r["tphidm"][u, 2]
        W = (C1 * C1 + C * C2) / S
        tW = (2 * np.abs(C1) * tC1 + np.abs(C2) * tC + np.abs(C) * tC2) / S + np.abs(W) * tS / S
        nu2 = freqs[u] ** -2.0
        A, Bs = W.sum(), (W * nu2).sum()
        nz = np.sqrt(A / Bs)
        tnz = 0.5 * nz * (tW.sum() / abs(A) + (tW * nu2).sum() / abs(Bs))
        KP = orc.Dconst / P
        go = KP * (nu2 - nz ** -2.0)
        tgo = KP * 2.0 * nz ** -3.0 * tnz
        H = -2.0 * np.array([[W.sum(), (W * go).sum()], [(W * go).sum(), (W * go * go).sum()]])
        t01 = 2.0 * (tW * np.abs(go) + np.abs(W) * tgo).sum()
        tH = np.array([[2.0 * tW.sum(), t01], [t01, 2.0 * (tW * go * go + 2 * np.abs(W * go) * tgo).sum()]])
        Hi = np.linalg.inv(H)
        out["nu_zero"] = (nz, tnz)
        out["cov"] = (2.0 * Hi, 2.0 * np.abs(Hi) @ tH @ np.abs(Hi))
    return out


def _ratio(got, want, tol):
    """max |got - want| / tol; where the tolerance is 0 (unused channels) the values must be equal"""
    got, want, tol = (np.atleast_1d(np.asarray(v, dtype=np.float64)) for v in (got, want, tol))
    err = np.abs(got - want)
    if not (np.all(np.isfinite(got)) and np.all(np.isfinite(want)) and np.all(np.isfinite(tol))):
        return np.inf
    r = np.where(tol > 0, err / np.where(tol > 0, tol, 1.0), np.where(err == 0, 0.0, np.inf))
    return float(r.max())


class Run(object):
    """One device call (max_iter = -1) and, per subint, what its reference needs."""

    def __init__(self, label, nbin, solver, dev, subs, log10_tau=False):
        self.label, self.nbin, self.solver, self.dev, self.subs, self.log10_tau = label, nbin, solver, dev, subs, log10_tau

    def ratios(self, **perturb):
        """max |device - reference| / tolerance per output over the subints (per-subint models: `model` /
        `table` in perturb replace each subint's model / frequency table)"""
        dev, out = self.dev, {}

        def upd(name, v):
            out[name] = max(out.get(name, 0.0), v)
        rep_model, rep_table = perturb.pop("model", None), perturb.pop("table", None)
        for s, sub in enumerate(self.subs):
            freqs = sub["freqs"] if rep_table is None else rep_table
            model = sub["model"] if rep_model is None else rep_model
            r = reference(sub["data"], model, dev["noise"][s], sub["P"], freqs, sub["nu_fits"], sub["x"],
                          self.log10_tau, sub["keep"], **perturb)
            cs = dev["chan_sums"][s]
            if self.solver == "phidm":
                names, got, want, tol = PHIDM, cs[:, :5], r["phidm"], r["tphidm"]
            else:
                names, got, want, tol = GEN, cs, r["gen"], r["tgen"]
            for j, nm in enumerate(names):
                upd(nm, _ratio(got[:, j], want[:, j], tol[:, j]))
            ep = epilogue(r, self.solver, freqs, sub["P"])
            for nm in ("chi2", "snr", "scales", "channel_snrs"):
                upd(nm, _ratio(dev[nm][s], *ep[nm]))
            if "cov" in ep:
                upd("nu_zero", _ratio(dev["nu_out"][s, 0], *ep["nu_zero"]))
                upd("cov", _ratio(dev["cov"][s][:2, :2], *ep["cov"]))
        return out

    def check(self):
        dev = self.dev
        assert (dev["return_code"] == 0).all() and (dev["nfeval"] == 1).all()
        if self.solver == "phidm":
            assert (dev["chan_sums"][..., 5:] == 0).all()
        # masked channels and channels without a noise level: nine zeros
        for s, sub in enumerate(self.subs):
            assert (dev["chan_sums"][s][dev["noise"][s] == 0] == 0).all()
        r = self.ratios()
        print("%-40s %-16s %-5s %s" % (self.label, kernel_path(self.nbin), self.solver,
                                       " ".join("%s %.1e" % kv for kv in r.items())))
        bad = {k: v for k, v in r.items() if not v <= 1.0}
        assert not bad, "%s: |device - reference| / tolerance > 1: %s" % (self.label, bad)
        return r


# ---- inputs ---------------------------------------------------------------------------------------------------------
def device_model(model, nbin):
    """the model values the device transforms: float64 as given at power-of-two nbin, else rounded to float32"""
    return model if _pow2(nbin) or model.dtype != np.float64 else model.astype(np.float32).astype(np.float64)


def nu_fits_of(freqs):
    """three different fit reference frequencies (nu_tau is not nu_DM, so that the tau_n reference matters)"""
    f0 = freqs.mean()
    return np.array([f0 + 37.0, f0 - 61.0, 0.8 * f0])


def points(freqs, P, nu_fits, nsub, solver, log10_tau=False):
    """init [nsub, 5]: phi near -0.5 and +0.5; a DM whose theta_n spans 1.6 turns over the band; for the general
    solver GM != 0, alpha = -3.2 and tau with w tau_n from 0.01 (k = 1, top of the band) to tens (high harmonics, low
    channels), and one subint with tau = 0 (the analytic limits of the tau-derivatives)"""
    nD, nG, nT = nu_fits
    gD = orc.Dconst * (freqs ** -2.0 - nD ** -2.0) / P
    gG = orc.Dconst ** 2 * (freqs ** -4.0 - nG ** -4.0) / P
    spanD = max(np.ptp(gD), np.abs(gD).max())
    spanG = max(np.ptp(gG), np.abs(gG).max())
    base = [(-0.4999, 2e-4 / spanD), (0.4999, -0.3 / spanD), (0.13, 1.6 / spanD), (-0.21, -0.5 / spanD)]
    x = np.zeros((nsub, 5))
    for s in range(nsub):
        x[s, :2] = base[s % 4]
    if solver == "gen":
        tau_top = 0.01 / (2 * np.pi) / (freqs.max() / nT) ** -3.2        # w tau_n = 0.01 at k = 1, top channel
        for s in range(nsub):
            x[s, 2] = (0.25, -0.1, 0.3, 0.05)[s % 4] / spanG
            x[s, 3] = tau_top * (1.0, 3.0, 0.5, 0.0)[s % 4]
            x[s, 4] = -3.2
        if log10_tau:
            x[:, 3] = np.log10(np.where(x[:, 3] > 0, x[:, 3], 1e-40))
    return x


def template(kind, nchan, nbin, seed=400):
    """(freqs, model [nchan, nbin] float64): the analytic synth.example_model (the harmonic cut-off is active at
    power-of-two nbin >= 256), or a white-noise template (every harmonic and the Nyquist term kept)"""
    if kind == "analytic":
        return synth.example_model(nchan, nbin, NU0, BW)
    return orc.make_freqs(nchan, NU0, BW), np.random.RandomState(seed).normal(0.0, 1.0, (nchan, nbin))


def matched_data(model, freqs, P, nu_fits, x, log10_tau=False, seed=0, amp=1.0, sigma=1.5):
    """float32 data [nsub, nchan, nbin]: subint s is amp * the model rotated by theta_n(x_s) and scattered by
    tau_n(x_s), plus white noise, so that x_s is next to the optimum (where the zero-covariance frequency and the
    covariance exist)"""
    nchan, nbin = model.shape
    rng = np.random.RandomState(seed)
    k = np.arange(nbin // 2 + 1)
    mft = np.fft.rfft(model, axis=1)
    nD, nG, nT = nu_fits
    out = []
    for xs in x:
        phi, DM, GM, tau, alpha = xs
        theta = phi + DM * orc.Dconst * (freqs ** -2.0 - nD ** -2.0) / P + \
            GM * orc.Dconst ** 2 * (freqs ** -4.0 - nG ** -4.0) / P
        taun = (10.0 ** tau if log10_tau else tau) * (freqs / nT) ** alpha
        spec = mft * np.exp(-2j * np.pi * np.outer(theta, k)) / (1.0 + 2j * np.pi * np.outer(taun, k))
        out.append(amp * np.fft.irfft(spec, n=nbin, axis=1) + rng.normal(0.0, sigma, model.shape))
    return np.array(out, dtype=np.float32)


def make_case(kind, nchan, nbin, nsub, solver, seed, log10_tau=False):
    """freqs, model, nu_fits, the points x [nsub, 5] and data matched to them"""
    freqs, model = template(kind, nchan, nbin)
    P = synth.P_EXAMPLE
    nf = nu_fits_of(freqs)
    x = points(freqs, P, nf, nsub, solver, log10_tau)
    amp, sigma = (1.0, 1.5) if kind == "analytic" else (0.3, 1.0)
    return freqs, model, nf, x, matched_data(model, freqs, P, nf, x, log10_tau, seed, amp, sigma)


def expected_keep(model, nbin):
    """the groups of 16 harmonics the device keeps per channel: the restated cut-off of a float64 model at power-of-two
    nbin; at other nbin (float32 model rows of Npad slots) every group holding a harmonic <= nbin/2"""
    if _pow2(nbin):
        return cutoff_groups(model)
    N = row_slots(nbin)
    return np.full(model.shape[0], max(min(N, LOK) // 16, -(-(nbin // 2 + 1) // 16)))


def evaluate(pl, data, P, x, nu_fits, solver, log10_tau=False, **kw):
    """one evaluate-only fit_batch call at x"""
    nsub = x.shape[0]
    flags = (1, 1, 0, 0, 0) if solver == "phidm" else (1, 1, 1, 1, 1)
    return pl.fit_batch(data, P, init=x, nu_fits=np.tile(nu_fits, (nsub, 1)) if np.ndim(nu_fits) == 1 else nu_fits,
                        nu_outs=np.full((nsub, 3), np.nan), fit_flags=flags, log10_tau=log10_tau, max_iter=-1,
                        want_chan_sums=True, **kw)


_RUNS = {}


def sweep_runs(nbin, solver, kind, nchan=37, nsub=4):
    """the row-plan sweep case (cached: the tolerance test below reuses the device outputs)"""
    key = (nbin, solver, kind, nchan)
    if key in _RUNS:
        return _RUNS[key]
    from pulseportraiture_b200.engine import WidebandPlan
    freqs, model, nf, _, data = make_case(kind, nchan, nbin, nsub, solver, seed=nbin + nchan)
    P = synth.P_EXAMPLE
    errs = np.random.RandomState(nbin + nchan).uniform(1.2, 1.8, (nsub, nchan))
    keep = expected_keep(device_model(model, nbin), nbin)
    runs = []
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        NJ = row_slots(nbin) // 16
        assert np.isclose(pl.stats()["x_keep_frac"], keep.mean() / NJ, rtol=1e-12, atol=0)
        if kind == "white":
            assert pl.stats()["x_keep_frac"] == 1.0 or not _pow2(nbin)
        for log10_tau in ((False, True) if solver == "gen" else (False,)):
            x = points(freqs, P, nf, nsub, solver, log10_tau)
            dev = evaluate(pl, data, P, x, nf, solver, log10_tau, errs=errs)
            subs = [dict(data=data[s].astype(np.float64), model=device_model(model, nbin), freqs=freqs, P=P,
                         nu_fits=nf, x=x[s], keep=keep if _pow2(nbin) else None) for s in range(nsub)]
            runs.append(Run("sweep nbin %d nchan %d %s%s" % (nbin, nchan, kind, " log10_tau" if log10_tau else ""),
                            nbin, solver, dev, subs, log10_tau))
    _RUNS[key] = runs
    return runs


NBINS = [64, 128, 256, 512, 1024, 2048, 4096, 66, 1002, 4094, 1000, 1536]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["analytic", "white"])
@pytest.mark.parametrize("solver", ["phidm", "gen"])
@pytest.mark.parametrize("nbin", NBINS)
def test_row_plan_sweep(nbin, solver, kind):
    """Every row transform: k_spectra<N, SpecPlan8<N>> (nbin 64-4096 but 2048), k_spectra16<0,0,0> (2048), and the
    k_fwd_any rows (Bluestein: 66, 1002, 4094; mixed radix: 1000, 1536) into k_spectra<Npad, ..., FROMSPEC> with
    nhalf != Npad; then k_pass2<N> + k_update2 (phidm) or k_pass5<N> + k_update5<128> (gen).  37 channels: the last
    32-channel CTA of the pass kernels is ragged."""
    for run in sweep_runs(nbin, solver, kind):
        run.check()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", ["phidm", "gen"])
@pytest.mark.parametrize("nbin", [2048, 1000])
def test_one_channel(nbin, solver):
    """nchan = 1: k_spectra16 (2048) and FROMSPEC<512> (1000) rows, one live row in a 32-channel pass CTA"""
    for run in sweep_runs(nbin, solver, "analytic", nchan=1):
        run.check()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", ["phidm", "gen"])
@pytest.mark.parametrize("dtype", ["f32", "f64", "i16", "torch"])
@pytest.mark.parametrize("nbin", [2048, 1536])
def test_inputs(nbin, dtype, solver):
    """Host float32, float64 (rounded on the device) and int16 (raw * scl + offs in float32: k_spectra16<1,0,0>,
    FROMSPEC after the int16 k_fwd_any rows) data and CUDA float32 data; errs given and errs=None (the measured
    noise); a chan_mask (masked channels: nine zeros) and an all-zero channel."""
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 3
    freqs, model, nf, x, data = make_case("analytic", nchan, nbin, nsub, solver, seed=700)
    data[2, 11] = 0.0
    P = synth.P_EXAMPLE
    mask = np.ones((nsub, nchan), np.uint8)
    mask[1, 3:10] = 0
    kw, values = {}, data.astype(np.float64)
    if dtype == "f64":
        arg = data.astype(np.float64) + np.random.RandomState(3).normal(0.0, 1e-5, data.shape)
        arg[2, 11] = 0.0
        values = arg.astype(np.float32).astype(np.float64)
    elif dtype == "i16":
        scl = np.full((nsub, nchan), 0.01, np.float32)
        offs = np.full((nsub, nchan), 0.5, np.float32)
        offs[2, 11] = 0.0
        arg = np.clip(np.round((data - offs[..., None]) / scl[..., None]), -32768, 32767).astype(np.int16)
        values = (arg.astype(np.float32) * scl[..., None] + offs[..., None]).astype(np.float64)
        kw = dict(dat_scl=scl, dat_offs=offs)
    elif dtype == "torch":
        arg = torch.from_numpy(data).cuda()
    else:
        arg = data
    assert not values[2, 11].any()
    errs = np.random.RandomState(5).uniform(1.2, 1.8, (nsub, nchan))
    keep = expected_keep(device_model(model, nbin), nbin)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        for e in (errs, None):
            dev = evaluate(pl, arg, P, x, nf, solver, errs=e, chan_mask=mask, **kw)
            assert (dev["noise"][mask == 0] == 0).all()
            if e is not None:
                assert np.array_equal(dev["noise"][mask == 1], errs[mask == 1])
            else:
                assert dev["noise"][2, 11] == 0.0 and (dev["noise"][mask == 1] > 0).sum() == mask.sum() - 1
            subs = [dict(data=values[s], model=device_model(model, nbin), freqs=freqs, P=P, nu_fits=nf, x=x[s],
                         keep=keep if _pow2(nbin) else None) for s in range(nsub)]
            Run("inputs nbin %d %s errs %s" % (nbin, dtype, "given" if e is not None else "None"),
                nbin, solver, dev, subs).check()


@pytest.mark.gpu
@pytest.mark.parametrize("align", [False, True])
@pytest.mark.parametrize("nbin", [2048, 512])
def test_guess_start(nbin, align):
    """No init and no DM_guess: the FFTFIT guess (k_spectra16<0,1,align> at 2048, k_spectra<256> with the guess
    partial sums and, with align, the kept data spectra at 512; k_guess) starts the (phi, DM) solver at
    (wrap(phi_guess), 0) in the nu_fits frame, and the one pass evaluates there."""
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 4
    freqs, model = template("analytic", nchan, nbin)
    P = synth.P_EXAMPLE
    nf = nu_fits_of(freqs)
    x = points(freqs, P, nf, nsub, "phidm")
    x[:, 1] = 0.0                  # the guess starts at DM = 0: data next to it
    data = matched_data(model, freqs, P, nf, x, seed=800)
    errs = np.random.RandomState(9).uniform(1.2, 1.8, (nsub, nchan))
    keep = expected_keep(model, nbin)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        dev = pl.fit_batch(data, P, errs=errs, nu_fits=np.tile(nf, (nsub, 1)), nu_outs=np.full((nsub, 3), np.nan),
                           max_iter=-1, want_chan_sums=True, align=align)
    assert (dev["lag_index"] >= 0).all()
    subs = [dict(data=data[s].astype(np.float64), model=model, freqs=freqs, P=P, nu_fits=nf,
                 x=np.array([dev["phi_guess"][s], 0.0, 0.0, 0.0, 0.0]), keep=keep) for s in range(nsub)]
    Run("guess nbin %d align %s" % (nbin, align), nbin, "phidm", dev, subs).check()


def multimodel_runs(nbin, solver):
    """three models with different tables, an interleaved model_index: host index, device index, chunks of 5"""
    key = ("models", nbin, solver)
    if key in _RUNS:
        return _RUNS[key]
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    from tests.test_gpu_multimodel import NCHAN, TABLES, _models
    models, freqs = _models(nbin)
    index = np.array([0, 0, 1, 2, 2, 0, 1, 1, 2, 0, 2, 1], dtype=np.int32)
    P = np.array([TABLES[m][3] * (1.0 + 1e-7 * s) for s, m in enumerate(index)])
    nf = np.stack([nu_fits_of(freqs[m]) for m in index])
    x = np.stack([points(freqs[m], P[s], nf[s], 4, solver)[s % 4] for s, m in enumerate(index)])
    data = np.concatenate([matched_data(models[m], freqs[m], P[s], nf[s], x[s:s + 1], seed=1200 + s)
                           for s, m in enumerate(index)])
    keeps = [expected_keep(device_model(models[m], nbin), nbin) if _pow2(nbin) else None for m in range(3)]
    runs = []
    with WidebandPlan(NCHAN, nbin) as pl:
        pl.set_models(models, freqs)
        for how, idx in (("host index", index), ("device index", torch.from_numpy(index).cuda()), ("chunk 5", index)):
            if how == "chunk 5":
                pl.set_chunk(5)
            dev = evaluate(pl, data, P, x, nf, solver, model_index=idx)
            subs = [dict(data=data[s].astype(np.float64), model=device_model(models[m], nbin), freqs=freqs[m], P=P[s],
                         nu_fits=nf[s], x=x[s], keep=keeps[m]) for s, m in enumerate(index)]
            runs.append(Run("models nbin %d %s" % (nbin, how), nbin, solver, dev, subs))
    _RUNS[key] = runs, models, freqs
    return _RUNS[key]


@pytest.mark.gpu
@pytest.mark.parametrize("solver", ["phidm", "gen"])
@pytest.mark.parametrize("nbin", [512, 2048, 1536])
def test_per_subint_models(nbin, solver):
    """pp_fit_batch_models: each subint's sums against the reference built from its own model and frequency table
    (the ModelRows reads of k_spectra<256> / k_spectra16 / FROMSPEC<1024> and of the pass and update kernels)"""
    runs, _, _ = multimodel_runs(nbin, solver)
    for run in runs:
        run.check()


@pytest.mark.gpu
@pytest.mark.parametrize("nbin", [512, 1536])
def test_two_kernels_one_sum(nbin):
    """A device-resident init takes the general path (pp_fit_batch_models cannot inspect it): with flags (1,1,0,0,0)
    and tau = 0, k_pass5 evaluates the point k_pass2 evaluates with the same init from the host.  C, C', C'' and chi2
    agree within the two bounds (plus the difference of the two references: k_pass5's S sums the kept harmonics, the
    (phi, DM) epilogue's p_n all of them)."""
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nsub = 37, 4
    freqs, model, nf, x, data = make_case("analytic", nchan, nbin, nsub, "phidm", seed=900)
    P = synth.P_EXAMPLE
    errs = np.random.RandomState(11).uniform(1.2, 1.8, (nsub, nchan))
    keep = expected_keep(device_model(model, nbin), nbin) if _pow2(nbin) else None
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        kw = dict(errs=errs, nu_fits=np.tile(nf, (nsub, 1)), max_iter=-1, want_chan_sums=True)
        two = pl.fit_batch(data, P, init=x, **kw)
        five = pl.fit_batch(data, P, init=torch.from_numpy(x).cuda(), **kw)
    assert (five["chan_sums"][..., 6] > 0).any() and (two["chan_sums"][..., 6] == 0).all()   # k_pass5 wrote S
    for s in range(nsub):
        r = reference(data[s].astype(np.float64), device_model(model, nbin), errs[s], P, freqs, nf, x[s], keep=keep)
        tol = r["tphidm"][:, :3] + r["tgen"][:, :3]
        assert _ratio(five["chan_sums"][s, :, :3], two["chan_sums"][s, :, :3], tol) <= 1.0
        e2, e5 = epilogue(r, "phidm", freqs, P), epilogue(r, "gen", freqs, P)
        tchi2 = e2["chi2"][1] + e5["chi2"][1] + abs(e2["chi2"][0] - e5["chi2"][0])
        assert _ratio(five["chi2"][s], two["chi2"][s], tchi2) <= 1.0


@pytest.mark.gpu
def test_phidm_chan_sums_slots_5_to_8_are_zero():
    """The (phi, DM) layout has no slots 5-8: they must come back as 0, not as what an earlier general-solver call on
    the same plan left in the plan's sums buffer"""
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nbin, nsub = 37, 512, 4
    freqs, model, nf, _, data = make_case("analytic", nchan, nbin, nsub, "gen", seed=1000)
    P = synth.P_EXAMPLE
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        gen = evaluate(pl, data, P, points(freqs, P, nf, nsub, "gen"), nf, "gen")
        assert (gen["chan_sums"][:3, :, 5:9] != 0).all()      # (subint 3 has tau = 0: S_t = 0)
        phidm = evaluate(pl, data, P, points(freqs, P, nf, nsub, "phidm"), nf, "phidm")
    assert (phidm["chan_sums"][..., 5:9] == 0).all()
    assert (phidm["chan_sums"][..., :5] != 0).all()


@pytest.mark.gpu
def test_the_tolerance_rejects_wrong_references():
    """The same comparisons against deliberately wrong references, on device outputs the cases above computed: each
    error must exceed its tolerance 10 times over in at least one case, so that a loosened bound shows here."""
    def worst(runs, **perturb):
        return max(max(run.ratios(**dict(perturb)).values()) for run in runs)
    N512 = 256
    misses = {
        "no Xlo (float32 X in the low slots)": worst(sweep_runs(2048, "phidm", "analytic"), no_xlo=True),
        "Nyquist term dropped": worst(sweep_runs(512, "phidm", "white"), drop_nyquist=True),
        "one mid-row harmonic dropped": worst(sweep_runs(512, "gen", "white"), drop_k=N512 // 2 + 3),
        "sigma_F^2 with Npad": worst(sweep_runs(1000, "phidm", "analytic"), sf2_npad=True),
        "tau_n referenced to nu_DM": worst(sweep_runs(512, "gen", "analytic"), tau_ref_dm=True),
    }
    runs, models, freqs = multimodel_runs(512, "phidm")
    misses["model 0's portrait for every subint"] = worst(runs, model=models[0])
    misses["model 0's table for every subint"] = worst(runs, table=freqs[0])
    print(misses)
    weak = {k: v for k, v in misses.items() if not v >= 10.0}
    assert not weak, weak


# ---- CPU: the restatement against the oracle ------------------------------------------------------------------------
def _cpu_case(nchan=6, nbin=128, seed=21):
    rng = np.random.RandomState(seed)
    freqs = orc.make_freqs(nchan, NU0, BW)
    _, model = synth.example_model(nchan, nbin, NU0, BW)
    data = 0.7 * np.roll(model, 3, axis=1) + rng.normal(0.0, 0.5, model.shape)
    sigma = rng.uniform(0.4, 0.6, nchan)
    return freqs, model, data, sigma


@pytest.mark.parametrize("log10_tau", [False, True])
def test_restatement_matches_the_oracle_primitives(log10_tau):
    """tau > 0: the nine sums are _FullProblem.primitives (pinned to the reference by the golden tests), whose X and M
    carry 1/sigma_F^2; the (phi, DM) slots 0-2 are _chan_sums / sigma_F^2 and slots 3, 4 continue the theta series"""
    freqs, model, data, sigma = _cpu_case()
    nbin = data.shape[1]
    P = synth.P_EXAMPLE
    nf = nu_fits_of(freqs)
    x = points(freqs, P, nf, 4, "gen", log10_tau)[0]
    assert x[3] != 0
    r = reference(data, model, sigma, P, freqs, nf, x, log10_tau)
    dFT, mFT = orc._spectra(data, model)
    prob = orc._FullProblem(dFT, mFT, sigma * np.sqrt(nbin / 2.0), P, freqs, nf[0], nf[1], nf[2], [1] * 5, log10_tau)
    pr = prob.primitives(list(x), order=2)
    for j, nm in enumerate(GEN):
        assert np.allclose(r["gen"][:, j], pr[nm], rtol=1e-10, atol=1e-10 * np.abs(pr[nm]).max()), nm
    x2 = np.array([x[0], x[1], 0.0, 0.0, 0.0])         # _chan_sums has no GM term
    r2 = reference(data, model, sigma, P, freqs, nf, x2)["phidm"]
    C, _, C1, C2 = orc._chan_sums(x[0], x[1], dFT * np.conj(mFT), P, freqs, nf[0])
    sF2 = sigma ** 2 * nbin / 2.0
    for j, v in enumerate((C, C1, C2)):
        assert np.allclose(r2[:, j], v / sF2, rtol=1e-10, atol=1e-10 * np.abs(v / sF2).max())
    # slots 3, 4 are the theta-derivatives of slots 2, 3: central differences in phi (step h: error ~ h^2 C^(5))
    h = 1e-5
    up = reference(data, model, sigma, P, freqs, nf, x + [h, 0, 0, 0, 0], log10_tau)["phidm"]
    dn = reference(data, model, sigma, P, freqs, nf, x - [h, 0, 0, 0, 0], log10_tau)["phidm"]
    for j in (3, 4):
        fd = (up[:, j - 1] - dn[:, j - 1]) / (2 * h)
        assert np.allclose(r["phidm"][:, j], fd, rtol=1e-6, atol=1e-6 * np.abs(fd).max())
    assert np.allclose(r["S"], (np.abs(mFT) ** 2).sum(1) / sF2, rtol=1e-13)


def test_restatement_tau_zero_limits():
    """At tau_n = 0 k_pass5 returns the analytic limits of the tau-derivative sums (the oracle sets them to 0):
    C_t = C_th, C_tht = C_thth, C_tt = 2 C_thth, S_t = 0, S_tt = -2 sum w^2 M; they are the tau -> 0 limits"""
    freqs, model, data, sigma = _cpu_case()
    P = synth.P_EXAMPLE
    nf = nu_fits_of(freqs)
    x = points(freqs, P, nf, 4, "gen")[3]
    assert x[3] == 0
    r = reference(data, model, sigma, P, freqs, nf, x)["gen"]
    g = dict(zip(GEN, r.T))
    assert np.array_equal(g["Ct"], g["Cth"]) and np.array_equal(g["Ctht"], g["Cthth"])
    assert np.allclose(g["Ctt"], 2 * g["Cthth"], rtol=1e-15) and (g["St"] == 0).all()
    m = np.fft.rfft(model, axis=1)[:, 1:]
    w = 2 * np.pi * np.arange(1, m.shape[1] + 1)
    sF2 = sigma ** 2 * data.shape[1] / 2.0
    assert np.allclose(g["Stt"], -2 * (w ** 2 * np.abs(m) ** 2).sum(1) / sF2, rtol=1e-14)
    near = reference(data, model, sigma, P, freqs, nf, x + [0, 0, 0, 1e-13, 0])["gen"]
    scale = np.abs(r).max(0)
    scale[7] = 1e-4 * scale[8]                        # S_t ~ tau_n S_tt (~1e-13 S_tt here): 0 at tau = 0
    assert np.allclose(near, r, rtol=1e-8, atol=1e-8 * scale)


def test_tolerance_of_the_restatement_covers_its_own_float32_storage():
    """The bound is the storage format's: X stored as the device stores it (a float32 product above LoK) moves each sum
    by less than its tolerance, at a shape where most of the model's power sits above LoK"""
    freqs, model, data, sigma = _cpu_case(nbin=1024)
    model = np.roll(model, 5, axis=1) + np.random.RandomState(2).normal(0.0, 0.3, model.shape)
    P = synth.P_EXAMPLE
    nf = nu_fits_of(freqs)
    for solver, x in (("gen", points(freqs, P, nf, 4, "gen")[0]), ("phidm", points(freqs, P, nf, 4, "phidm")[2])):
        r = reference(data, model, sigma, P, freqs, nf, x)
        rs = reference(data, model, sigma, P, freqs, nf, x, stored=True)
        assert 0.0 < _ratio(rs[solver], r[solver], r["t" + solver]) < 1.0
