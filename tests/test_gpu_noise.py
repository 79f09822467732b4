"""Every noise estimate -- sigma_n, from which every channel weight, chi2, S/N, scale error and TOA / DM error bar is
computed -- against a float64 restatement at every row plan.

  get_noise_batch(kc)          pp_get_noise_cut_batch: k_rfft_rows<N, double / float> (power-of-two nbin; float by
                               pp_plan_set_fft_precision(32)), k_fwd_any + k_rows_from_spec (any other nbin)
  fit_batch(errs=None)         the sigma pp_fit_batch measures itself: k_spectra16 (nbin 2048, all eight <I16, GUESS,
                               KEEPD> variants), k_spectra<N, SpecPlan8> (other powers of two), k_spectra<..., FROMSPEC>
  get_noise_fit_batch(fact)    k_noise_fit: the find_kc 20^3 grid search on the rows' float64 spectra
  pplib.get_noise*(chans=False) the whole portrait as one row of any length (float64 rfft, the grid in chunks)

Reference.  sigma^2 = sum_{k >= kc} |X_k|^2 / (nbin (L + 1 - kc)), L = nbin/2, X = rfft(x) in numpy float64, on
exactly the values the device reads: float32 data held in float64, float64 data rounded to float32, int16 data decoded
as fadd_rn(fmul_rn(raw, scl), offs) in float32.  find_kc is restated as scipy.optimize.brute's full grid: np.mgrid
points, chi2 in flat C order, np.argmin (the first NaN wins; otherwise the lowest chi2, the lowest index on ties).

Bound.  Let ||dX|| <= c sqrt(nbin) ||x||_2 be the error of the computed transform, c = u (40 log2 nbin + 40) for the
double rows (u = 2^-53; the constant of test_gpu_rotate.py, covering Bluestein and mixed radix) and
c = 2^-24 (6 log2 nbin + 8) for k_rfft_rows<N, float>.  With T = sqrt(nbin ntop) sigma = ||X_top||,

  |d sigma| / sigma <= e + e^2 / 2 + (ntop + 4) u,     e = ||dX|| / T.

Rows with a pulse 1e4 times the noise make e large; they stay inside this bound, not inside a constant.  For the grid,
the same dX carried into log10 of the powers (|d y_k| <= -2 log10(1 - |dX| / |X_k|)) and the rounding of the residuals
and of the chi2 sums give each point a slack Delta; the device must equal the reference sigma at a grid point whose
chi2 is within Delta of the minimum, and every seeded row has exactly one such point (points with b = 0 have the same
chi2 for every a, bit for bit, so the lowest index among them is the one point), so the argmin is pinned.

Deliberately wrong references, each of which must miss by at least 10x the bound (the rows carry sinusoids at
harmonics kc - 1 and kc, a DC offset and an alternating component so that each of them shows): the cut at kc - 1 and
kc + 1, the Nyquist term dropped, the DC term counted at kc >= 1, ntop off by one, the normalisation by 2 Npad instead
of nbin (any-nbin plans); for the fit estimator the cut at k0 -/+ 1, fact not applied, fact * kc rounded up instead of
truncated, the 0.99 nharm clamp missing (an empty mean) and NaN cells skipped instead of winning (with every cell NaN
the cut-off falls to k = 1).  The CPU tests pin the restatement to the oracle, scipy.optimize.brute and the golden
arrays.
"""
import math
import os

import numpy as np
import pytest
import scipy.optimize as opt

from oracle import pp_oracle as orc
from tests import synth
from tests.test_gpu_rotate import MISS, PLAN_IDS, PLANS, U, _plan, _pow2, c_fft32, c_fft64

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


# ---------------------------------------------------------------------------------------------------------------
# the restatement
# ---------------------------------------------------------------------------------------------------------------
def power(x):
    """|X_k|^2, X = rfft(x) along the last axis"""
    X = np.fft.rfft(x, axis=-1)
    return X.real ** 2 + X.imag ** 2


def sigma_cut(P, nbin, k0, ntop=None, norm=None, extra=0.0):
    """sqrt((sum_{k >= k0} P_k + extra) / (norm ntop)), norm = nbin, ntop = nharm - k0 by default"""
    nt = P.shape[-1] - k0 if ntop is None else ntop
    return np.sqrt((P[..., k0:].sum(-1) + extra) / ((nbin if norm is None else norm) * nt))


def sigma_tol(x, P, nbin, k0, cf):
    """sigma (e + e^2/2 + (ntop + 4) u), e = ||dX|| / ||X_top||, ||dX|| = cf sqrt(nbin) ||x||; where X_top is exactly 0
    (a top that holds only an exactly zero Nyquist term) ||dX|| / sqrt(nbin ntop), the triangle inequality's bound"""
    ntop = P.shape[-1] - k0
    dX = cf * np.sqrt(nbin) * np.linalg.norm(x, axis=-1)
    T = np.sqrt(P[..., k0:].sum(-1))
    with np.errstate(all="ignore"):
        e = dX / T
        return np.where(T > 0, sigma_cut(P, nbin, k0) * (e + 0.5 * e * e + (ntop + 4) * U), dX / np.sqrt(nbin * ntop))


def find_kc_grid(y, dy=None):
    """brute's grid of find_kc for y = log10 pows: (grid [3, 8000], chi2 [8000]) in flat C order (a slowest) and, with
    dy a bound on |d y_k|, the slack of every point's chi2 (the propagated dy and the rounding of both evaluations)"""
    nh = y.size
    k = np.arange(nh)
    c2 = np.empty(8000)
    dl = np.zeros(8000)
    with np.errstate(all="ignore"):
        lo, hi = y.min(), y.max()
        g = np.mgrid[nh ** -1.0:1.0:20j, 0:hi - lo:20j, lo:hi:20j].reshape(3, -1)
        for ia in range(20):
            s = slice(400 * ia, 400 * ia + 400)
            a, b, d = (v[:, None] for v in g[:, s])
            bE = b * np.exp(-a * k)
            r = y - (bE + d)
            c2[s] = np.sum(r ** 2, axis=-1)
            if dy is not None:
                dl[s] = (np.sum((2 * np.abs(r) + dy) * dy + 8 * U * np.abs(r) * (np.abs(y) + np.abs(bE) + np.abs(d)),
                                axis=-1) + 2 * (nh + 8) * U * c2[s])
    return g, c2, dl


def argmin_np(c2):
    """np.argmin: the first NaN if there is one, else the first minimum"""
    nan = np.flatnonzero(np.isnan(c2))
    return int(nan[0]) if nan.size else int(np.argmin(c2))


def kc_at(a, nh):
    hit = np.flatnonzero(np.exp(-a * np.arange(nh)) < 0.005)
    return int(hit[0]) if hit.size else nh - 1


def k0_of(kc, fact, nh, rnd=int):
    """first harmonic of get_noise_fit's mean: fact * kc, clamped to 0.99 nharm when it reaches nharm"""
    kf = fact * kc
    if kf >= nh:
        kf = min(int(0.99 * nh), kf)
    return rnd(kf)


def noise_fit_ref(x, nbin, fact, cf):
    """get_noise_fit of one row: (sigma, tol, {wrong: sigma}, candidate grid points)"""
    P = power(x)
    nh = P.size
    with np.errstate(all="ignore"):
        y = np.log10(P / nbin)
        rel = cf * np.sqrt(nbin) * np.linalg.norm(x) / np.sqrt(P)
        small = rel < 0.5
        dy = np.where(small, -2 * np.log10(1 - np.where(small, rel, 0.0)), np.inf) + 8 * U * (np.abs(y) + 1)
    g, c2, dl = find_kc_grid(y, dy)
    i0 = argmin_np(c2)
    if np.isnan(c2[i0]):
        cands = [i0]
    else:
        near = np.flatnonzero(c2 <= c2[i0] + dl + dl[i0])
        cands = sorted({int(i % 400) if g[1, i] == 0 else int(i) for i in near})
    kc = kc_at(g[0, cands[0]], nh)
    k0 = k0_of(kc, fact, nh)
    ref, tol = sigma_cut(P, nbin, k0), sigma_tol(x, P, nbin, k0, cf)
    wrong = {"k0-1": sigma_cut(P, nbin, k0 - 1)}
    if k0 + 1 < nh:
        wrong["k0+1"] = sigma_cut(P, nbin, k0 + 1)
    for name, k in (("no_fact", k0_of(kc, 1.0, nh)), ("fact_kc_rounded_up", k0_of(kc, fact, nh, math.ceil))):
        if k != k0:
            wrong[name] = sigma_cut(P, nbin, k)
    if fact * kc >= nh:
        wrong["no_clamp"] = np.nan        # pows[int(fact kc):] is empty
    if np.isnan(c2[i0]) and k0_of(1, fact, nh) != k0:
        wrong["nan_skipped"] = sigma_cut(P, nbin, k0_of(1, fact, nh))
    return ref, tol, wrong, cands


def miss(wrong, ref, tol):
    """max over rows of |wrong - ref| / tol; a wrong reference that is not finite misses by inf"""
    d = np.where(np.isfinite(wrong), np.abs(np.asarray(wrong, dtype=np.float64) - ref), np.inf)
    return float(np.max(d / tol))


def check(got, ref, tol, wrongs, label):
    """device within tol of ref; every wrong reference misses ref by >= MISS tol.  Prints the ratios."""
    got = np.asarray(got, dtype=np.float64)
    assert np.all(np.isfinite(got)), label
    r = float(np.max(np.abs(got - ref) / tol))
    m = {k: miss(v, ref, tol) for k, v in wrongs.items()}
    print("RATIO %s err/tol=%.3g %s" % (label, r, " ".join("%s=%.3g" % kv for kv in sorted(m.items()))))
    assert r <= 1.0, (label, r)
    for k, v in m.items():
        assert v >= MISS, (label, k, v)


def ps_wrongs(P, nbin, kc, npad=None):
    """the deliberately wrong references of the cut estimator at kc, for rows with power spectra P"""
    nh = P.shape[-1]
    L, ntop = nh - 1, nh - kc
    w = {"ntop+1": sigma_cut(P, nbin, kc, ntop=ntop + 1)}
    if kc >= 1:
        w["kc-1"] = sigma_cut(P, nbin, kc - 1)
        w["dc_counted"] = sigma_cut(P, nbin, kc, ntop=ntop, extra=P[..., 0])
    if kc < L:
        w["kc+1"] = sigma_cut(P, nbin, kc + 1)
        w["nyquist_dropped"] = sigma_cut(P, nbin, kc, ntop=ntop, extra=-P[..., L])
    if ntop > 1:
        w["ntop-1"] = sigma_cut(P, nbin, kc, ntop=ntop - 1)
    if npad is not None:
        w["norm_2Npad"] = sigma_cut(P, nbin, kc, norm=2 * npad)
    return w


def _npad(nbin):
    """the padded transform length / 2 of an any-nbin plan (None for a power of two)"""
    if _pow2(nbin):
        return None
    n = 1
    while n < nbin // 2 + 1:
        n *= 2
    return n


def _rows(rng, n, nbin, sins=(), hdr=True):
    """float32 rows: white noise, a pulse, a DC offset, an alternating component and sinusoids at the harmonics sins;
    with hdr the last row is a pulse 1e4 times the noise instead"""
    j = np.arange(nbin)
    x = rng.standard_normal((n, nbin))
    d = (j / nbin - rng.uniform(0, 1, (n, 1)) + 0.5) % 1.0 - 0.5
    x += 3.0 * np.exp(-0.5 * (d / 0.02) ** 2) + 0.7 + 0.5 * (-1.0) ** j
    for k in sins:
        if 0 < k < nbin // 2:
            x += 0.8 * np.cos(2 * np.pi * k * j / nbin + rng.uniform(0, 2 * np.pi, (n, 1)))
    if hdr:
        x[-1] = rng.standard_normal(nbin) + 1e4 * np.exp(-0.5 * (d[-1] / (0.8 / nbin)) ** 2)
    return x.astype(np.float32).astype(np.float64)


def _fit_rows(rng, nbin, zero_row):
    """rows for get_noise_fit: a pulse over white noise, white noise only, a steep red spectrum, and (zero_row) small
    integers in equal pairs, whose Nyquist term is exactly 0"""
    j = np.arange(nbin)
    L = nbin // 2
    rows = []
    for _ in range(3):
        d = (j / nbin - rng.uniform() + 0.5) % 1.0 - 0.5
        rows.append(rng.standard_normal(nbin) + 4.0 * np.exp(-0.5 * (d / 0.03) ** 2))
    rows += [rng.standard_normal(nbin) for _ in range(2)]
    k = np.arange(L + 1)
    X = 1e3 * nbin * (k + 1.0) ** -3 * np.exp(2j * np.pi * rng.uniform(size=L + 1))
    X[0] = X[0].real
    X[L] = X[L].real
    rows.append(np.fft.irfft(X, n=nbin) + rng.standard_normal(nbin))
    if zero_row:
        rows.append(np.repeat(rng.randint(-5, 6, L), 2).astype(np.float64))
    else:
        rows.append(np.fft.irfft(X * (k + 1.0) ** -1, n=nbin) + rng.standard_normal(nbin))
    return np.array(rows).astype(np.float32).astype(np.float64)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the restatement against the oracle, scipy.optimize.brute and the golden arrays
# ---------------------------------------------------------------------------------------------------------------
def _zero_row(nbin=512, seed=3):
    return np.repeat(np.random.RandomState(seed).randint(-5, 6, nbin // 2), 2).astype(np.float64)


def test_cut_restatement_matches_oracle_and_golden():
    G = np.load(os.path.join(GOLDEN, "golden_v1.npz"))
    G2 = np.load(os.path.join(GOLDEN, "golden_v2.npz"))
    data = synth.make_case(16, 512, 1500., 800., 701)["data"]
    P = power(data)
    for frac in (1, 2, 4, 8):
        kc = int((1 - frac ** -1) * 257)
        ref = sigma_cut(P, 512, kc)
        assert np.max(np.abs(ref / orc.get_noise_PS(data, frac=frac, chans=True) - 1)) < 1e-13
        assert np.max(np.abs(ref / G2["noise/ps_frac%d" % frac] - 1)) < 1e-12
    x = data[3]
    assert abs(sigma_cut(power(x), 512, int(0.875 * 257)) / G2["noise/ps_prof_frac8"] - 1) < 1e-12
    c = synth.make_case(64, 512, 1500., 800., 0, phi=0.123, dDM=3e-4, legacy_seed=True)
    assert np.max(np.abs(sigma_cut(power(c["data"]), 512, 192) / G["c1/noise"] - 1)) < 1e-12
    xa = c["data"].ravel()
    n = xa.size
    assert abs(sigma_cut(power(xa), n, int(0.75 * (n // 2 + 1))) / G["c1/noise_all"] - 1) < 1e-12
    assert abs(sigma_cut(power(xa), n, int(0.75 * (n // 2 + 1))) / orc.get_noise_PS(c["data"]) - 1) < 1e-13


def test_find_kc_restatement_matches_brute_and_oracle():
    rng = np.random.RandomState(11)
    rows = list(_fit_rows(rng, 256, True)) + [_zero_row()] + list(_rows(rng, 2, 1000, hdr=False))
    for x in rows:
        nbin = x.size
        pows = power(x) / nbin
        with np.errstate(all="ignore"):
            y = np.log10(pows)
        g, c2, _ = find_kc_grid(y)
        i = argmin_np(c2)
        kc = kc_at(g[0, i], pows.size)
        assert kc == orc.find_kc(pows)

        def chi2(p):
            return np.sum((y - (p[1] * np.exp(-p[0] * np.arange(y.size)) + p[2])) ** 2.0)
        with np.errstate(all="ignore"):
            xmin = opt.brute(chi2, [(y.size ** -1.0, 1.0), (0, y.max() - y.min()), (y.min(), y.max())], Ns=20,
                             finish=None)
        assert np.array_equal(xmin, g[:, i], equal_nan=True)


def test_nan_grid_picks_point_zero():
    """A row with an exactly zero harmonic: every chi2 is NaN, np.argmin takes grid point 0 (a = 1/nharm), find_kc
    gives nharm - 1 and the noise comes from the clamped top 1% of the spectrum, far below get_noise_PS."""
    x = _zero_row()
    pows = power(x) / 512
    assert pows[-1] == 0.0
    with np.errstate(all="ignore"):
        g, c2, _ = find_kc_grid(np.log10(pows))
    assert np.isnan(c2).all() and argmin_np(c2) == 0
    assert orc.find_kc(pows) == 256 == kc_at(g[0, 0], 257)
    ref, _, wrong, cands = noise_fit_ref(x, 512, 1.1, c_fft64(512))
    assert cands == [0] and abs(ref / orc.get_noise_fit(x) - 1) < 1e-13
    assert ref < 0.1 * orc.get_noise_PS(x)
    assert "nan_skipped" in wrong and abs(wrong["nan_skipped"] / ref - 1) > 1.0


def test_noise_fit_restatement_matches_oracle_and_golden():
    G2 = np.load(os.path.join(GOLDEN, "golden_v2.npz"))
    data = synth.make_case(16, 512, 1500., 800., 701)["data"]
    for fact, key in ((1.1, "noise/fit_chans"), (2.0, "noise/fit_fact2")):
        ref = np.array([noise_fit_ref(x, 512, fact, c_fft64(512))[0] for x in data])
        assert np.max(np.abs(ref / G2[key] - 1)) < 1e-12
        assert np.max(np.abs(ref / orc.get_noise_fit(data, fact=fact, chans=True) - 1)) < 1e-13
    assert abs(noise_fit_ref(data[3], 512, 1.1, c_fft64(512))[0] / G2["noise/fit_prof"] - 1) < 1e-12
    rng = np.random.RandomState(5)
    for x in _fit_rows(rng, 128, True):
        for fact in (1.1, 2.0, 50.0):
            assert np.isclose(noise_fit_ref(x, 128, fact, c_fft64(128))[0], orc.get_noise_fit(x, fact=fact),
                              rtol=1e-13, atol=0.0)


def test_facade_find_kc_matches_restatement():
    """pplib's whole-portrait grid search (torch, in chunks) on CPU tensors: the same point as brute's"""
    import torch
    from pulseportraiture_b200 import pplib
    rng = np.random.RandomState(8)
    for x in list(_fit_rows(rng, 512, True)) + list(_rows(rng, 2, 1000, hdr=False)):
        pows = power(x) / x.size
        assert pplib._find_kc(torch.from_numpy(pows)) == orc.find_kc(pows)


# ---------------------------------------------------------------------------------------------------------------
# GPU: get_noise_batch at every cut and plan
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_noise_cut_against_float64(nbin, force, monkeypatch):
    L = nbin // 2
    label = PLAN_IDS[PLANS.index((nbin, force))]
    rng = np.random.RandomState(40 + nbin + 17 * force)
    cuts = [("default", -1, (3 * (L + 1)) // 4)] + [("frac%d" % f, int((1 - f ** -1) * (L + 1)),
                                                     int((1 - f ** -1) * (L + 1))) for f in (1, 2, 8)]
    cuts += [("kc1", 1, 1), ("nyquist", L, L)]
    precisions = (0, 64, 32) if _pow2(nbin) else (0, 64)
    nchan = 7                                     # not a multiple of RowGeom<N>::kRows
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        for name, arg, kc in cuts:
            x = _rows(rng, nchan, nbin, sins=(kc - 1, kc))
            P = power(x)
            ref = sigma_cut(P, nbin, kc)
            wrong = ps_wrongs(P, nbin, kc, _npad(nbin))
            for bits in precisions:
                pl.set_fft_precision(bits)
                got = pl.get_noise_batch(x.astype(np.float32)[None], kc=arg)[0]
                f32 = bits == 32
                tol = sigma_tol(x, P, nbin, kc, c_fft32(nbin) if f32 else c_fft64(nbin))
                check(got, ref, tol, wrong, "cut%s-%s-%s" % ("32" if f32 else "64", label, name))


# ---------------------------------------------------------------------------------------------------------------
# GPU: the sigma pp_fit_batch measures (errs = None)
# ---------------------------------------------------------------------------------------------------------------
FIT = [(37, "float32", False, False), (1, "float64", True, False), (300, "int16", False, True),
       (37, "cuda", True, True)]
FIT2048 = FIT + [(37, dt, init, align) for dt in ("float32", "int16") for init in (False, True)
                 for align in (False, True) if (37, dt, init, align) not in FIT]


@pytest.mark.gpu
@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_fit_batch_noise_against_float64(nbin, force, monkeypatch):
    import torch
    L, nsub = nbin // 2, 3
    kc = (3 * (L + 1)) // 4
    label = PLAN_IDS[PLANS.index((nbin, force))]
    rng = np.random.RandomState(80 + nbin + 17 * force)
    for nchan, dtype, init, align in (FIT2048 if nbin == 2048 else FIT):
        x = _rows(rng, nsub * nchan, nbin, sins=(kc - 1, kc)).reshape(nsub, nchan, nbin)
        mask = np.ones((nsub, nchan), dtype=np.uint8)
        zeros = []
        if nchan > 1:
            mask[0, 1] = 0                       # masked
            x[2, 3] = 0.0                        # all zero
            zeros += [(0, 1), (2, 3)]
            if dtype != "int16":
                x[1, 2, 5] = np.nan              # a NaN sample
                zeros.append((1, 2))
        kw = {}
        if dtype == "float32":
            dev = x.astype(np.float32)
        elif dtype == "cuda":
            dev = torch.from_numpy(x.astype(np.float32)).cuda()
        elif dtype == "float64":
            dev = x + 1e-9 * rng.standard_normal(x.shape)     # rounded to float32 on the device
            x = dev.astype(np.float32).astype(np.float64)
        else:
            from pulseportraiture_b200 import pptoas
            raw, scl, offs, _ = pptoas.quantize_subints(x)
            dev = raw
            kw = dict(dat_scl=scl, dat_offs=offs)
            # fadd_rn(fmul_rn(raw, scl), offs) in float32, as the device decodes
            x = ((raw.astype(np.float32) * scl[..., None]).astype(np.float32) + offs[..., None]).astype(np.float32)
            x = x.astype(np.float64)
        freqs, model = synth.example_model(nchan, nbin, 1500., 800.)
        flags = (1, 0, 0, 0, 0) if nchan == 1 else (1, 1, 0, 0, 0)
        with _plan(nchan, nbin, force, monkeypatch) as pl:
            pl.set_model(model.astype(np.float32), freqs)
            r = pl.fit_batch(dev, synth.P_EXAMPLE, chan_mask=mask, init=np.zeros((nsub, 5)) if init else None,
                             fit_flags=flags, align=align, **kw)
        got = r["noise"]
        for z in zeros:
            assert got[z] == 0.0, (z, got[z])
        ok = np.ones((nsub, nchan), dtype=bool)
        for z in zeros:
            ok[z] = False
        P = power(np.where(ok[..., None], x, 1.0))
        ref = sigma_cut(P, nbin, kc)[ok]
        tol = sigma_tol(x[ok], P[ok], nbin, kc, c_fft64(nbin))
        wrong = {k: v[ok] for k, v in ps_wrongs(P, nbin, kc, _npad(nbin)).items()}
        check(got[ok], ref, tol, wrong, "fit_batch-%s-nchan%d-%s%s%s" % (label, nchan, dtype, "-init" if init else "",
                                                                          "-align" if align else ""))


# ---------------------------------------------------------------------------------------------------------------
# GPU: get_noise_fit_batch (k_noise_fit)
# ---------------------------------------------------------------------------------------------------------------
def _check_fit(got, rows, nbin, fact, cf, label):
    refs, tols, cands = [], [], []
    wl = []
    for x in rows:
        ref, tol, wrong, cand = noise_fit_ref(x, nbin, fact, cf)
        refs.append(ref)
        tols.append(tol)
        cands.append(cand)
        wl.append(wrong)
    assert all(len(c) == 1 for c in cands), (label, cands)     # the argmin is pinned
    refs, tols = np.array(refs), np.array(tols)
    keys = sorted({k for w in wl for k in w})
    wrong = {k: np.array([w.get(k, r) for w, r in zip(wl, refs)]) for k in keys}
    check(got, refs, tols, wrong, label)


@pytest.mark.gpu
@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_noise_fit_against_float64(nbin, force, monkeypatch):
    label = PLAN_IDS[PLANS.index((nbin, force))]
    rng = np.random.RandomState(120 + nbin + 17 * force)
    zero_row = _pow2(nbin)
    rows = _fit_rows(rng, nbin, zero_row)
    if zero_row:
        assert power(rows[-1])[-1] == 0.0
    with _plan(len(rows), nbin, force, monkeypatch) as pl:
        for fact in (1.1, 2.0, 50.0):
            got = pl.get_noise_fit_batch(rows.astype(np.float32)[None], fact)[0]
            _check_fit(got, rows, nbin, fact, c_fft64(nbin), "fit-%s-fact%g" % (label, fact))


# ---------------------------------------------------------------------------------------------------------------
# GPU: the whole portrait as one row (chans=False), at any length
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_whole_portrait_noise_any_length():
    from pulseportraiture_b200 import pplib
    G = np.load(os.path.join(GOLDEN, "golden_v1.npz"))
    c1 = synth.make_case(64, 512, 1500., 800., 0, phi=0.123, dDM=3e-4, legacy_seed=True)["data"]
    rng = np.random.RandomState(9)
    c2 = synth.make_case(16, 1000, 1500., 800., 702)["data"]
    prof = _rows(rng, 1, 32, sins=(11, 12), hdr=False)[0]
    for name, data in (("64x512", c1), ("16x1000", c2), ("prof32", prof)):
        x = data.ravel()
        n = x.size
        P = power(x)
        for frac in (4, 2):
            kc = int((1 - frac ** -1) * (n // 2 + 1))
            got = pplib.get_noise_PS(data, frac=frac)
            ref, tol = sigma_cut(P, n, kc), sigma_tol(x, P, n, kc, c_fft64(n))
            check(got, ref, tol, ps_wrongs(P, n, kc), "whole-PS-frac%d-%s" % (frac, name))
            if name == "64x512" and frac == 4:
                assert pplib.get_noise(data) == got
                assert abs(got - G["c1/noise_all"]) <= 2 * tol      # the reference's own value, its own rfft
        for fact in (1.1, 2.0):
            got = pplib.get_noise_fit(data, fact=fact)
            _check_fit(np.array([got]), [x], n, fact, c_fft64(n), "whole-fit-fact%g-%s" % (fact, name))
