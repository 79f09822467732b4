"""PCA / B-spline model building on the device (pp_pca_moments, pp_pca_project, pp_lowpass_rows and
pplib.make_spline_model) against the float64 restatement of tests/test_cpu_spline_build.py, and the recovery of an
injected truth model through make_fake_pulsar, make_spline_model and GetTOAs.

Error model of the device sums (u = 2^-53): the mean adds nchan products in order, |mu - mu_ref| <=
4 (nchan + 2) u sum_n w_n |x_n| / W; a moment adds K products of rows formed with one rounding each, so
|M - M_ref| <= 4 (K + 8) u S with S = sum_n w_n (|x_n| + |mu|)(|x_n| + |mu|)^T / W on the same side (the reference's
own BLAS sum is inside the same bound).  Low-passed rows are a forward and an inverse FP64 transform of the same
truncated spectrum, within the transform bound of test_gpu_rotate.py, u (40 log2 nbin + 40) ||x||."""
import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests.test_cpu_spline_build import basis, lowpass, moments, moments_scale, sign_convention, smooth_portrait

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
# (nchan, nbin, gram): both sides, power-of-two and other nbin (mixed radix 1000, Bluestein 1002), nbin 64 and 4096
CASES = [(96, 64, False), (96, 64, True), (40, 1000, True), (1100, 1000, False), (48, 1002, True), (64, 4096, True),
         (600, 512, False)]
IDS = ["%dx%d-%s" % (c, b, "gram" if g else "cov") for c, b, g in CASES]


def _plan(nchan, nbin):
    from pulseportraiture_b200.engine import WidebandPlan
    return WidebandPlan(nchan, nbin)


def c_fft64(nbin):
    return U * (40.0 * np.log2(nbin) + 40.0)


@pytest.mark.parametrize("nchan,nbin,gram", CASES, ids=IDS)
def test_moments_basis_and_projection_vs_restatement(nchan, nbin, gram):
    port, w = smooth_portrait(nchan, nbin, 3, 3 * nchan + nbin, zero=(0, 7, nchan - 1))
    pl = _plan(nchan, nbin)
    mu, M = pl.pca_moments(port, w, gram=gram)
    mu_ref, M_ref = moments(port, w, gram)
    W = w.sum()
    tol_mu = 4 * (nchan + 2) * U * (w[:, None] * np.abs(port)).sum(0) / W
    assert np.all(np.abs(mu - mu_ref) <= tol_mu)
    K = nbin if gram else nchan
    tol = 4 * (K + 8) * U * moments_scale(port, w, gram)
    err = np.abs(M - M_ref)
    print("RATIO moments %.3g" % np.max(err[tol > 0] / tol[tol > 0]))
    assert np.all(err <= tol)      # (rows and columns of zero-weight channels of G are exactly 0)
    assert np.array_equal(M, M.T)
    mu2, M2 = pl.pca_moments(port, w, gram=gram)
    assert np.array_equal(mu, mu2) and np.array_equal(M, M2)

    # basis: the top 3 eigenvectors (host eigh of the device matrix, back-projected on the device on the Gram side)
    import scipy.linalg as sl
    dim = M.shape[0]
    vals, Uv = sl.eigh(M, subset_by_index=[dim - 3, dim - 1])
    Uv = np.ascontiguousarray(Uv[:, ::-1])
    E = pl.pca_backproject(port, w, mu, Uv) if gram else sign_convention(Uv)
    if gram:
        assert np.array_equal(E, pl.pca_backproject(port, w, mu, Uv))
    # the reference: numpy.linalg.eigh of the restated covariance (the Gram route for nbin 4096, which
    # test_gram_and_covariance_routes_give_one_basis ties to it)
    _, E_ref = basis(port, w, 3, gram=nbin > 2048)
    dots = np.sum(E * E_ref, axis=0)
    print("DOTS", 1 - dots)
    assert np.all(dots >= 1 - 1e-12)
    assert np.allclose(np.linalg.norm(E, axis=0), 1.0, rtol=0, atol=1e-14)

    # projections of x_n - mu~ onto E
    mus = mu + 0.01
    P = pl.pca_project(port, mus, E)
    P_ref = (port - mus) @ E
    tolp = 4 * (nbin + 2) * U * ((np.abs(port) + np.abs(mus)) @ np.abs(E))
    assert np.all(np.abs(P - P_ref) <= tolp)
    assert np.array_equal(P, pl.pca_project(port, mus, E))


@pytest.mark.parametrize("nbin", [64, 512, 1000, 1002, 4096])
def test_lowpass_rows_vs_restatement(nbin):
    rng = np.random.RandomState(nbin)
    x = orc.get_bin_centers(nbin)
    rows = []
    for i, (wid, lvl) in enumerate([(0.02, 1e-3), (0.05, 1e-2), (0.01, 1e-4), (0.03, 0.1), (0.2, 1e-6)]):
        rows.append(np.exp(-0.5 * ((x - 0.3 - 0.1 * i) / wid) ** 2) + lvl * rng.standard_normal(nbin))
    rows.append(rng.standard_normal(nbin))                 # white noise
    rows = np.array(rows)
    pl = _plan(1, nbin)
    out, kc = pl.lowpass_rows(rows)
    ref, kc_ref = lowpass(rows)
    print("KC", kc, kc_ref)
    assert np.array_equal(kc, kc_ref)
    tol = c_fft64(nbin) * np.linalg.norm(rows, axis=1)[:, None]
    r = np.abs(out - ref) / tol
    print("RATIO lowpass %.3g" % r.max())
    assert r.max() <= 1.0
    # a wrong reference (the Nyquist term kept regardless, or k_c itself dropped) misses by far more
    X = np.fft.rfft(rows, axis=1)
    for i, k in enumerate(kc_ref):
        if k + 1 <= nbin // 2:
            Xw = X[i].copy()
            Xw[k:] = 0.0
            assert np.max(np.abs(np.fft.irfft(Xw, nbin) - ref[i]) / tol[i]) > 10.0
    out2, kc2 = pl.lowpass_rows(rows)
    assert np.array_equal(out, out2) and np.array_equal(kc, kc2)


# ---- injected truth -------------------------------------------------------------------------------
NCHAN, NBIN, NSUB, SIGMA, P0 = 128, 1024, 64, 0.05, 0.0042


def _truth(ncomp):
    """a mean profile, ncomp band-limited orthonormal evolution vectors and smooth spline curves over 1100-1900 MHz"""
    import scipy.interpolate as si
    x = orc.get_bin_centers(NBIN)
    g = lambda c, s: np.exp(-0.5 * ((x - c) / s) ** 2)          # noqa: E731
    mean_prof = g(0.4, 0.03) + 0.4 * g(0.47, 0.05)
    if not ncomp:
        return mean_prof, np.zeros((NBIN, 0)), (np.zeros(8), [], 3)
    raw = np.array([g(0.42, 0.03) * np.cos(2 * np.pi * 3 * (x - 0.42)), g(0.38, 0.04) * np.sin(2 * np.pi * 2 * (x - 0.38))])
    eigvec = sign_convention(np.linalg.qr(raw[:ncomp].T)[0])
    f = np.linspace(1080., 1920., 12)
    curves = np.array([0.3 * np.sin(f / 150.), 0.3 * np.sin(f / 120. + 1.0)])[:ncomp]   # both vary across the band
    tck, _ = si.splprep(curves, u=f, k=3, s=0)
    return mean_prof, eigvec, tck


def _write_truth(tmp_path, ncomp):
    from pulseportraiture_b200 import pplib
    path = str(tmp_path / ("truth%d.spl" % ncomp))
    pplib.write_spline_model(path, "truth", "fake", "none", *_truth(ncomp), quiet=True)
    return path


def _averaged(path, sigma, nsub, seed):
    from pulseportraiture_b200 import pplib
    d = pplib.make_fake_pulsar(path, P0, nsub=nsub, nchan=NCHAN, nbin=NBIN, nu0=1500., bw=800., noise_stds=sigma,
                               seed=seed, quiet=True)
    return d.subints[:, 0].mean(0), d.freqs[0]


@pytest.fixture(scope="module")
def truth2(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("spline_truth")
    path = _write_truth(tmp, 2)
    port, freqs = _averaged(path, SIGMA, NSUB, 5)
    return tmp, path, port, freqs


def test_injected_truth_recovered(truth2):
    from pulseportraiture_b200 import pplib, pptoas
    tmp, tpath, port, freqs = truth2
    r = pplib.make_spline_model(port, freqs, norm=None, model_name="built", source="fake", datafile="avg")
    print("SNRS", r.snrs, "KC", r.kc, "ncomp", r.ncomp, "fp", r.fp, "ier", r.ier)
    assert r.ncomp == 2 and list(r.ieig) == [0, 1]
    assert np.all(np.diff(r.eigval) <= 0)
    assert np.allclose(r.eigvec.T @ r.eigvec, np.eye(2), rtol=0, atol=1e-12)
    mp, ev, tk = _truth(2)
    truth = pplib.gen_spline_portrait(mp, freqs, ev, tk)
    # bound: the noise of the averaged portrait, sigma / sqrt(nsub), in the (ncomp + 1) (2 kc + 1) Fourier
    # coefficients a channel's model can carry at most, plus the truth's own power above the lowest kc, plus the
    # float32 evaluation of the model
    s_avg = SIGMA / np.sqrt(NSUB)
    kmax, kmin = int(np.max(r.kc)), int(np.min(r.kc))
    T = np.fft.rfft(truth, axis=1)
    T[:, :kmin + 1] = 0.0
    above = np.sqrt(np.mean(np.fft.irfft(T, NBIN, axis=1) ** 2, axis=1))
    bound = 4 * s_avg * np.sqrt((r.ncomp + 1) * (2 * kmax + 1) / NBIN) + above + 2e-7 * np.abs(truth).max()
    rms = np.sqrt(np.mean((r.model - truth) ** 2, axis=1))
    print("RMS/BOUND max %.3f median %.3f" % (np.max(rms / bound), np.median(rms / bound)))
    assert np.all(rms <= bound)
    assert np.all(np.isfinite(r.channel_red_chi2s))

    # TOAs of fresh subints with the built model and with the truth
    bpath = str(tmp / "built.spl")
    pplib.write_spline_model(bpath, r.model_name, r.source, r.datafile, r.mean_prof, r.eigvec, r.tck, quiet=True)
    rng = np.random.RandomState(9)
    nsub = 16
    fresh = str(tmp / "fresh.npz")
    pplib.make_fake_pulsar(tpath, P0, outfile=fresh, nsub=nsub, nchan=NCHAN, nbin=NBIN, nu0=1500., bw=800.,
                           noise_stds=SIGMA, phase=rng.uniform(-0.3, 0.3, nsub), dDM=rng.normal(0, 2e-4, nsub),
                           seed=77, quiet=True)
    res = {}
    for name, mpath in (("built", bpath), ("truth", tpath)):
        gt = pptoas.GetTOAs(fresh, mpath, quiet=True)
        gt.get_TOAs(quiet=True)
        res[name] = (np.asarray(gt.phis[0]), np.asarray(gt.phi_errs[0]), np.asarray(gt.DMs[0]),
                     np.asarray(gt.DM_errs[0]), np.array([v[0] for v in gt.nu_refs[0]]), np.asarray(gt.Ps[0]))
    pb, _, db, _, nub, Ps = res["built"]
    pt, et, dt, edt, nut, _ = res["truth"]
    ddm = np.abs(db - dt) / np.median(edt)
    pb_at_t = pplib.phase_transform(pb, db, nub, nut, Ps, mod=False)
    dphi = (pb_at_t - pt + 0.5) % 1.0 - 0.5
    spread = np.abs(dphi - np.median(dphi)) / np.median(et)
    print("DDM/err max %.3f  phase spread/err max %.3f  offset %.3g" % (ddm.max(), spread.max(), np.median(dphi)))
    assert ddm.max() < 0.3
    assert spread.max() < 0.1


def test_low_snr_keeps_no_spurious_components(tmp_path):
    from pulseportraiture_b200 import pplib
    path0 = _write_truth(tmp_path, 0)
    port, freqs = _averaged(path0, SIGMA, NSUB, 6)
    r = pplib.make_spline_model(port, freqs, norm=None)
    print("SNRS ncomp=0 truth", r.snrs)
    assert r.ncomp == 0 and r.eigvec.shape == (NBIN, 0)
    assert r.model.shape == (NCHAN, NBIN) and np.allclose(r.model, r.mean_prof[None], rtol=0, atol=1e-6)
    # the two-component truth under 20x the noise: fewer components survive
    port, freqs = _averaged(_write_truth(tmp_path, 2), 20 * SIGMA, 4, 7)
    r = pplib.make_spline_model(port, freqs, norm=None)
    print("SNRS low S/N", r.snrs)
    assert r.ncomp < 2


def test_channel_order_and_smoothing_invariance(truth2):
    from pulseportraiture_b200 import pplib
    _, _, port, freqs = truth2
    w = np.ones(NCHAN)
    w[[3, 50]] = 0.0
    a = pplib.make_spline_model(port, freqs, weights=w)
    for perm in (np.random.RandomState(1).permutation(NCHAN), np.arange(NCHAN)[::-1]):
        b = pplib.make_spline_model(port[perm], freqs[perm], weights=w[perm])
        assert np.array_equal(a.mean_prof, b.mean_prof) and np.array_equal(a.eigvec, b.eigvec)
        assert np.array_equal(a.tck[0], b.tck[0]) and all(np.array_equal(c, d) for c, d in zip(a.tck[1], b.tck[1]))
        assert np.array_equal(a.model[perm], b.model) and np.array_equal(a.freqs, b.freqs)
    c = pplib.make_spline_model(port, freqs, weights=w, smooth=False)
    assert c.kc is None and c.ncomp >= 1 and np.all(np.isfinite(c.model))
    # unsmoothed, the mean profile is the weighted mean of the normalised channels: it carries their noise, which
    # the smoothed one does not
    assert not np.array_equal(c.mean_prof, a.mean_prof)
    hi = np.abs(np.fft.rfft(c.mean_prof)[NBIN // 4:]).max()
    assert np.abs(np.fft.rfft(a.mean_prof)[NBIN // 4:]).max() < 1e-9 * hi
    d = pplib.make_spline_model(port, freqs, weights=w, smooth=False)
    assert np.array_equal(c.mean_prof, d.mean_prof) and np.array_equal(c.eigvec, d.eigvec)
