"""GPU tests of the evolving-Gaussian portrait fit (pp_fit_gaussian_portraits, WidebandPlan.
fit_gaussian_portraits, pplib.fit_gaussian_portrait): the device sums at a point against the float64
restatement of tests/test_cpu_gaussfit.py, the optimum against scipy.optimize.least_squares on the
restated residual, the error bars by recovery, batch invariance, the facade through write_model /
read_model / GetTOAs, and argument errors."""
import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests import synth
from tests.test_cpu_gaussfit import make_problem, model_time, restate

pytestmark = pytest.mark.gpu

# Bound on the device sums relative to their natural scales: chi2 relative, J^T r over
# sqrt(jtj_ii chi2) and J^T J over sqrt(jtj_ii jtj_jj) (Cauchy-Schwarz).  The rows are double FFTs
# (1e-15 of the row norm per harmonic) summed in a different order than numpy's.
SUM_TOL = 3e-13


def _plan(nchan, nbin, freqs):
    from pulseportraiture_b200.engine import WidebandPlan
    pl = WidebandPlan(nchan, nbin)
    pl.set_freqs(freqs)
    return pl


def _sum_errors(dev, ref, free, scale=None):
    """Largest normalised deviation of chi2, jtr, jtj (free entries) from the reference.  Entries are scaled
    by the diagonal of ``scale`` (default ``ref``); where that diagonal is 0 (alpha while tau = 0) the
    device's entries must be exactly 0."""
    scale = ref if scale is None else scale
    f = np.where(free)[0]
    d = np.sqrt(np.diag(scale["jtj"])[f])
    z = d == 0
    assert not dev["jtr"][0][f][z].any() and not dev["jtj"][0][np.ix_(f, f)][z].any()
    f, d = f[~z], d[~z]
    e_chi = abs(dev["chi2"][0] / ref["chi2"] - 1.0)
    e_jtr = np.max(np.abs(dev["jtr"][0][f] - ref["jtr"][f]) / (d * np.sqrt(scale["chi2"])))
    e_jtj = np.max(np.abs(dev["jtj"][0][np.ix_(f, f)] - ref["jtj"][np.ix_(f, f)]) / np.outer(d, d))
    return max(e_chi, e_jtr, e_jtj)


def _evaluate(code, p, freqs, nu_ref, nbin, data, errs, free):
    with _plan(len(freqs), nbin, freqs) as pl:
        return pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref, max_iter=-1,
                                         want_sums=True)


SUM_CASES = [   # code, nchan, nbin, tau, free tau, free alpha, flags off (indices)
    ("000", 1, 64, 0.0, 0, 0, ()),
    ("110", 37, 512, 1.3, 0, 0, ()),
    ("011", 16, 2048, 0.0, 1, 1, (5,)),
    ("000", 512, 512, 0.8, 1, 1, (3, 9)),
    ("110", 6, 4096, 2.0, 1, 1, ()),
    ("011", 3, 1024, 0.5, 1, 0, (7, 8)),
]


@pytest.mark.parametrize("code,nchan,nbin,tau,ftau,falpha,off", SUM_CASES)
def test_sums_at_a_point_match_the_restatement(code, nchan, nbin, tau, ftau, falpha, off):
    p, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, tau=tau, seed=nchan + nbin)
    p = p * (1 + 0.01 * np.random.RandomState(1).randn(len(p)))   # away from the truth
    free = np.ones(len(p), bool)
    free[1], free[-1] = bool(ftau), bool(falpha)
    free[list(off)] = False
    dev = _evaluate(code, p, freqs, nu_ref, nbin, data, errs, free)
    ref = restate(code, p, freqs, nu_ref, nbin, data, errs)
    assert dev["return_code"][0] == 0 and dev["nfeval"][0] == 1
    assert np.array_equal(dev["params"][0], p)
    err = _sum_errors(dev, ref, free)
    assert err < SUM_TOL, err
    fixed = ~free
    assert not dev["jtr"][0][fixed].any() and not dev["jtj"][0][fixed].any() and not dev["jtj"][0][:, fixed].any()


def test_wrong_references_miss_by_ten_times_the_bound():
    """Nyquist taken as B_N G_N, the DC harmonic dropped, the alpha chain without the log: each misses the
    device sums by more than 10 x SUM_TOL (narrow components at nbin 64 so that G_N is not negligible)."""
    code, nchan, nbin = "000", 8, 64
    p, freqs, nu_ref, _, _ = make_problem(code, nchan, nbin, tau=1.1, seed=4)
    p[4:-1:6] = 0.022                                 # wid of every component: about 1.4 bins
    rng = np.random.RandomState(8)
    data = model_time(code, p, freqs, nu_ref, nbin) + 0.05 * rng.randn(nchan, nbin)
    errs = np.full(nchan, 0.05)
    free = np.ones(len(p), bool)
    dev = _evaluate(code, p, freqs, nu_ref, nbin, data, errs, free)
    ref = restate(code, p, freqs, nu_ref, nbin, data, errs)
    assert _sum_errors(dev, ref, free) < SUM_TOL
    for wrong in ("nyquist", "nodc", "alpha_nolog"):
        miss = _sum_errors(dev, restate(code, p, freqs, nu_ref, nbin, data, errs, wrong=wrong), free, scale=ref)
        assert miss > 10 * SUM_TOL, (wrong, miss)


# ---- optimum vs scipy ---------------------------------------------------------------------------------
def _scipy_fit(code, p0, freqs, nu_ref, nbin, data, errs, free, bounds):
    from scipy.optimize import least_squares
    f = np.where(free)[0]

    def full(q):
        p = p0.copy()
        p[f] = q
        return p

    def fun(q):
        r = restate(code, full(q), freqs, nu_ref, nbin, data, errs)
        sw = np.sqrt(r["w"])
        return np.concatenate([(sw * r["R"].real).ravel(), (sw * r["R"].imag).ravel()])

    def jac(q):
        r = restate(code, full(q), freqs, nu_ref, nbin, data, errs)
        sw = np.sqrt(r["w"])[:, None, :]
        J = r["J"][:, f]
        return -np.concatenate([(sw * J.real).transpose(0, 2, 1).reshape(-1, len(f)),
                                (sw * J.imag).transpose(0, 2, 1).reshape(-1, len(f))])
    if bounds is None:
        res = least_squares(fun, p0[f], jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    else:
        lo = np.where(np.isnan(bounds[f, 0]), -np.inf, bounds[f, 0])
        hi = np.where(np.isnan(bounds[f, 1]), np.inf, bounds[f, 1])
        res = least_squares(fun, np.clip(p0[f], lo, hi), jac=jac, bounds=(lo, hi), method="trf",
                            xtol=1e-15, ftol=1e-15, gtol=1e-15)
    p = full(res.x)
    r = restate(code, p, freqs, nu_ref, nbin, data, errs)
    dof = len(freqs) * nbin - len(f)
    cov = np.linalg.inv(r["jtj"][np.ix_(f, f)]) * r["chi2"] / dof
    errs_out = np.zeros(len(p))
    errs_out[f] = np.sqrt(np.diag(cov))
    return p, r["chi2"], errs_out


PARITY_CASES = [   # code, nchan, nbin, true tau, free tau, free alpha, bound
    ("000", 16, 256, 0.0, 0, 0, None),
    ("110", 16, 256, 1.5, 1, 1, None),
    ("011", 12, 128, 0.0, 0, 0, "wid_max"),
    ("000", 16, 256, -0.4, 1, 0, "tau"),
]


@pytest.mark.parametrize("code,nchan,nbin,tau,ftau,falpha,bound", PARITY_CASES)
def test_optimum_matches_scipy(code, nchan, nbin, tau, ftau, falpha, bound):
    p_true, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, tau=tau, seed=11 + nchan)
    P = len(p_true)
    free = np.ones(P, bool)
    free[1], free[-1] = bool(ftau), bool(falpha)
    bounds = None
    if bound == "wid_max":
        bounds = np.full((P, 2), np.nan)
        bounds[4, 1] = p_true[4] * 0.9                 # the first component's width is held at its maximum
    elif bound == "tau":
        bounds = np.full((P, 2), np.nan)
        bounds[1, 0] = 0.0
    rng = np.random.RandomState(5)
    p0 = p_true.copy()
    ng = (P - 3) // 6
    p0[2:-1:6] += 0.002 * rng.randn(ng)
    p0[4:-1:6] *= 1 + 0.03 * rng.randn(ng)
    p0[6:-1:6] *= 1 + 0.05 * rng.randn(ng)
    if ftau:
        p0[1] = max(p0[1], 0.0) + 0.3
    with _plan(nchan, nbin, freqs) as pl:
        dev = pl.fit_gaussian_portraits(data[None], errs[None], code, p0[None], free, nu_ref, bounds=bounds)
    assert dev["return_code"][0] == 0
    p_ref, chi2_ref, errs_ref = _scipy_fit(code, p0, freqs, nu_ref, nbin, data, errs, free, bounds)
    f = np.where(free)[0]
    sig = dev["param_errs"][0][f]
    assert np.max(np.abs(dev["params"][0][f] - p_ref[f]) / sig) < 1e-3
    assert abs(dev["chi2"][0] / chi2_ref - 1.0) < 1e-8
    assert np.max(np.abs(dev["param_errs"][0][f] / errs_ref[f] - 1.0)) < 1e-4
    assert dev["red_chi2"][0] == pytest.approx(dev["chi2"][0] / (nchan * nbin - len(f)), rel=1e-15)
    if bound == "wid_max":
        assert dev["params"][0][4] == bounds[4, 1]
    if bound == "tau":
        assert dev["params"][0][1] == 0.0


# ---- zero Jacobian columns -------------------------------------------------------------------------
def test_tau_and_alpha_free_from_an_unscattered_start():
    """tau and alpha free from tau = 0: alpha's column is exactly zero at the start point (tau_n = 0).  The
    fit leaves alpha out of that step, moves tau off 0 and converges to scipy's optimum with finite errors
    for every parameter."""
    code, nchan, nbin = "000", 16, 256
    p_true, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, tau=1.2, seed=31)
    free = np.ones(len(p_true), bool)
    p0 = p_true.copy()
    p0[1] = 0.0
    p0[2:-1:6] += 0.002
    with _plan(nchan, nbin, freqs) as pl:
        dev = pl.fit_gaussian_portraits(data[None], errs[None], code, p0[None], free, nu_ref)
    assert dev["return_code"][0] == 0
    sig = dev["param_errs"][0]
    assert np.all(np.isfinite(sig)) and np.all(sig > 0)
    p_ref, chi2_ref, errs_ref = _scipy_fit(code, p0, freqs, nu_ref, nbin, data, errs, free, None)
    assert np.max(np.abs(dev["params"][0] - p_ref) / sig) < 1e-3
    assert abs(dev["chi2"][0] / chi2_ref - 1.0) < 1e-8
    assert np.max(np.abs(sig / errs_ref - 1.0)) < 1e-4


def test_tau_on_its_lower_bound_with_alpha_free():
    """tau and alpha free with tau >= 0 and data whose best tau is negative: tau ends on the bound, where
    alpha cannot move the model.  The fit converges; alpha gets error 0 and a zero covariance row (MINPACK's
    convention for a zero column); every other parameter matches scipy's bounded fit of the same problem
    (alpha has no effect at tau = 0) with finite errors."""
    code, nchan, nbin = "000", 16, 256
    p_true, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, tau=-0.4, seed=32)
    P = len(p_true)
    free = np.ones(P, bool)
    bounds = np.full((P, 2), np.nan)
    bounds[1, 0] = 0.0
    p0 = p_true.copy()
    p0[1] = 0.3
    with _plan(nchan, nbin, freqs) as pl:
        dev = pl.fit_gaussian_portraits(data[None], errs[None], code, p0[None], free, nu_ref, bounds=bounds)
    assert dev["return_code"][0] == 0
    assert dev["params"][0][1] == 0.0
    assert dev["param_errs"][0][-1] == 0.0 and not dev["cov"][0][-1].any() and not dev["cov"][0][:, -1].any()
    f = np.where(free)[0][:-1]                                # all but alpha
    sig = dev["param_errs"][0][f]
    assert np.all(np.isfinite(sig)) and np.all(sig > 0)
    free_ref = free.copy()
    free_ref[-1] = False
    p0_ref = p0.copy()
    p0_ref[-1] = dev["params"][0][-1]
    p_ref, chi2_ref, errs_ref = _scipy_fit(code, p0_ref, freqs, nu_ref, nbin, data, errs, free_ref, bounds)
    assert np.max(np.abs(dev["params"][0][f] - p_ref[f]) / sig) < 1e-3
    assert abs(dev["chi2"][0] / chi2_ref - 1.0) < 1e-8
    # the device's dof counts alpha as free, scipy's does not: compare the unscaled errors
    dof_dev, dof_ref = nchan * nbin - P, nchan * nbin - (P - 1)
    unscaled = sig / np.sqrt(dev["chi2"][0] / dof_dev)
    assert np.max(np.abs(unscaled / (errs_ref[f] / np.sqrt(chi2_ref / dof_ref)) - 1.0)) < 1e-4


def test_more_portraits_than_one_launch_holds():
    """A batch of more small portraits than one chunk may hold (the chunk's portraits are a grid dimension,
    at most 65535): evaluated in two chunks, each portrait as when it is evaluated alone."""
    code, nchan, nbin, nport = "000", 1, 64, 66000
    p, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, seed=41, ngauss=1)
    rng = np.random.RandomState(42)
    datas = data[None] + 0.05 * rng.randn(nport, nchan, nbin)
    free = np.ones(len(p), bool)
    free[1] = free[-1] = False
    with _plan(nchan, nbin, freqs) as pl:
        r = pl.fit_gaussian_portraits(datas, np.tile(errs, (nport, 1)), code, np.tile(p, (nport, 1)), free,
                                      nu_ref, max_iter=-1, want_sums=True)
        for s in (0, 65534, 65535, nport - 1):
            one = pl.fit_gaussian_portraits(datas[s:s + 1], errs[None], code, p[None], free, nu_ref, max_iter=-1,
                                            want_sums=True)
            for k in ("chi2", "jtr", "jtj"):
                assert np.array_equal(r[k][s], one[k][0]), (s, k)
    assert (r["return_code"] == 0).all()


# ---- error bars by recovery -----------------------------------------------------------------------
def test_recovery_pulls_of_200_portraits():
    code, nchan, nbin, nport, sigma = "000", 64, 512, 200, 0.05
    p_true, freqs, nu_ref, _, _ = make_problem(code, nchan, nbin, tau=1.5, seed=21, ngauss=3, sigma=sigma)
    clean = model_time(code, p_true, freqs, nu_ref, nbin)
    rng = np.random.RandomState(22)
    data = clean[None] + sigma * rng.randn(nport, nchan, nbin)
    errs = np.full((nport, nchan), sigma)
    free = np.ones(len(p_true), bool)
    with _plan(nchan, nbin, freqs) as pl:
        r = pl.fit_gaussian_portraits(data, errs, code, np.tile(p_true, (nport, 1)), free, nu_ref)
    assert (r["return_code"] == 0).all()
    pulls = (r["params"] - p_true[None]) / r["param_errs"]
    assert np.all(np.abs(pulls.mean(axis=0)) < 0.2), pulls.mean(axis=0)
    rms = np.sqrt((pulls ** 2).mean(axis=0))
    assert np.all((rms > 0.85) & (rms < 1.15)), rms


# ---- batch invariance -----------------------------------------------------------------------------
def test_batch_equals_single_fits_bit_for_bit():
    code, nchan, nbin = "110", 24, 256
    probs = [make_problem(code, nchan, nbin, tau=0.9, seed=40 + s) for s in range(8)]
    freqs, nu_ref = probs[0][1], probs[0][2]
    data = np.stack([q[3] for q in probs])
    errs = np.stack([q[4] for q in probs])
    init = np.stack([q[0] * (1 + 0.01 * np.random.RandomState(s).randn(len(q[0]))) for s, q in enumerate(probs)])
    free = np.ones(init.shape[1], bool)
    keys = ("params", "param_errs", "cov", "chi2", "red_chi2", "nfeval", "return_code", "model")
    with _plan(nchan, nbin, freqs) as pl:
        batch = pl.fit_gaussian_portraits(data, errs, code, init, free, nu_ref, want_model=True)
        singles = [pl.fit_gaussian_portraits(data[s:s + 1], errs[s:s + 1], code, init[s:s + 1], free, nu_ref,
                                             want_model=True) for s in range(8)]
        pl.set_chunk(3)
        chunked = pl.fit_gaussian_portraits(data, errs, code, init, free, nu_ref, want_model=True)
    for k in keys:
        one = np.concatenate([s[k] for s in singles])
        assert np.array_equal(batch[k], one), k
        assert np.array_equal(chunked[k], one), k
    # the model output is the portrait at the fitted parameters
    for s in (0, 5):
        want = model_time(code, batch["params"][s], freqs, nu_ref, nbin)
        assert np.max(np.abs(batch["model"][s] - want)) < 1e-12 * np.max(np.abs(want))


def test_cuda_tensor_inputs_give_the_same_fit():
    torch = pytest.importorskip("torch")
    code, nchan, nbin = "011", 8, 128
    p, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, seed=60)
    free = np.ones(len(p), bool)
    free[1] = free[-1] = False
    with _plan(nchan, nbin, freqs) as pl:
        a = pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref)
        dev = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda")
        b = pl.fit_gaussian_portraits(dev(data[None]), dev(errs[None]), code, dev(p[None]), free, nu_ref)
    assert np.array_equal(a["params"], b["params"]) and np.array_equal(a["chi2"], b["chi2"])


# ---- facade: align -> fit -> write_model -> read_model -> GetTOAs ------------------------------------
def test_facade_from_aligned_portrait_to_toas(tmp_path):
    from pulseportraiture_b200 import pplib, ppalign, pptoas
    from tests.test_gpu_parity import _fake_archive
    nchan, nbin = 32, 512
    archive, cases = _fake_archive(8, nchan, nbin, 7100, sigma=0.5)
    aligned = ppalign.align_archives([archive], cases[0]["model"], fit_dm=True, niter=1, quiet=True).port
    freqs = cases[0]["freqs"]
    name, code, nu_ref, ngauss, params, flags, alpha, _ = pplib.read_model(synth.GMODEL)
    flags = flags.copy()
    flags[1] = 0                                              # unscattered data: tau stays 0
    init = params.copy()
    init[2::6] += 0.003
    errs = orc.get_noise(aligned, chans=True)
    fit = pplib.fit_gaussian_portrait(code, aligned, init, alpha, errs, flags, 0, pplib.get_bin_centers(nbin),
                                      freqs, nu_ref)
    assert fit.return_code == 0 and fit.model.shape == (nchan, nbin)
    assert fit.dof == nchan * nbin - int(flags.sum()) and 0.5 < fit.red_chi2 < 2.0
    assert fit.covariance.shape == (len(params) + 1,) * 2
    out = np.array(fit.fitted_params)
    out[1] = out[1] * cases[0]["P"] / nbin                    # TAU in seconds
    path = str(tmp_path / "fit.gmodel")
    pplib.write_model(path, name, code, nu_ref, out, flags, fit.scattering_index, 0, quiet=True)
    _, _, rebuilt = pplib.read_model(path, pplib.get_bin_centers(nbin), freqs, cases[0]["P"], quiet=True,
                                     device=True)
    assert np.max(np.abs(rebuilt - fit.model)) < 1e-9 * np.max(np.abs(fit.model))
    # TOAs of fresh subints with the fitted model recover the injected phase and DM
    fresh, fcases = _fake_archive(4, nchan, nbin, 7300, sigma=1.0)
    gt = pptoas.GetTOAs([fresh], path, quiet=True)
    gt.get_TOAs()
    for s, c in enumerate(fcases):
        nu = gt.nu_refs[0][s][0]
        phi_true = pplib.phase_transform(c["phi"], c["dDM"], c["nu0"], nu, c["P"], mod=True)
        dphi = (gt.phis[0][s] - phi_true + 0.5) % 1.0 - 0.5
        assert abs(dphi) < 3 * gt.phi_errs[0][s]
        assert abs(gt.DMs[0][s] / fresh.doppler_factors[s] - c["dDM"]) < 3 * gt.DM_errs[0][s]


# ---- errors ---------------------------------------------------------------------------------------
def test_argument_errors_raise():
    from pulseportraiture_b200 import _ffi, pplib
    from pulseportraiture_b200.engine import WidebandPlan
    code, nchan, nbin = "000", 4, 64
    p, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, seed=1)
    free = np.ones(len(p), bool)
    with _plan(nchan, nbin, freqs) as pl:
        with pytest.raises(ValueError):                       # ngauss 0
            pl.fit_gaussian_portraits(data[None], errs[None], code, p[None, :3], free[:3], nu_ref)
        p17 = np.concatenate([p[:2], np.tile(p[2:8], 17), p[-1:]])
        with pytest.raises(_ffi.PPError, match="ngauss"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p17[None], np.ones(len(p17), bool), nu_ref)
        with pytest.raises(_ffi.PPError, match="model_code"):
            pl.fit_gaussian_portraits(data[None], errs[None], "020", p[None], free, nu_ref)
        bad = errs.copy()
        bad[2] = 0.0
        with pytest.raises(_ffi.PPError, match="errs"):
            pl.fit_gaussian_portraits(data[None], bad[None], code, p[None], free, nu_ref)
        with pytest.raises(_ffi.PPError, match="nu_ref"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, -1.0)
    with WidebandPlan(nchan, 1000) as pl:
        pl.set_freqs(freqs)
        with pytest.raises(_ffi.PPError, match="power of two"):
            pl.fit_gaussian_portraits(np.zeros((1, nchan, 1000)), errs[None], code, p[None], free, nu_ref)
    with WidebandPlan(nchan, nbin) as pl:
        with pytest.raises(_ffi.PPError, match="pp_set_freqs"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref)
    with pytest.raises(NotImplementedError):
        pplib.fit_gaussian_portrait(code, data, p[:-1], p[-1], errs, free[:-1], 0, pplib.get_bin_centers(nbin),
                                    freqs, nu_ref, join_params=[0.1])
