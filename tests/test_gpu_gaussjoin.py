"""GPU tests of join parameters in the evolving-Gaussian portrait fit (pp_fit_gaussian_portraits_join,
WidebandPlan.fit_gaussian_portraits(join_chan=...), pplib.fit_gaussian_portrait(join_params=...),
pplib.gen_gaussian_portrait_device(join_ichans=...)): the device sums at a point against the float64 restatement
of tests/test_cpu_gaussjoin.py, the optimum against scipy.optimize.least_squares, the joined model, recovery of
injected offsets from simulated archives, batch invariance and the facade through write_model and GetTOAs."""
import numpy as np
import pytest

from tests import synth
from tests.test_cpu_gaussjoin import PSPIN, join_groups, make_join_problem, model_time_join, restate_join
from tests.test_gpu_gaussfit import SUM_TOL, _sum_errors

pytestmark = pytest.mark.gpu


def _plan(nchan, nbin, freqs):
    from pulseportraiture_b200.engine import WidebandPlan
    pl = WidebandPlan(nchan, nbin)
    pl.set_freqs(freqs)
    return pl


def _evaluate(code, p, freqs, nu_ref, nbin, data, errs, free, jc):
    with _plan(len(freqs), nbin, freqs) as pl:
        return pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref, max_iter=-1,
                                         want_sums=True, join_chan=jc, P=PSPIN)


# ---- sums at a point ---------------------------------------------------------------------------------
@pytest.mark.parametrize("code", ["000", "111"])
@pytest.mark.parametrize("ftau", [0, 1])
@pytest.mark.parametrize("njoin", [1, 3])
@pytest.mark.parametrize("nbin", [64, 128, 256, 512, 1024, 2048, 4096])
def test_join_sums_at_a_point_match_the_restatement(code, ftau, njoin, nbin):
    nchan = 8
    p, freqs, nu_ref, data, errs, jc = make_join_problem(code, nchan, nbin, njoin, tau=0.8 if ftau else 0.0,
                                                         seed=nbin + njoin)
    p = p * (1 + 0.01 * np.random.RandomState(1).randn(len(p)))   # away from the truth
    free = np.ones(len(p), bool)
    ia = len(p) - 2 * njoin - 1
    free[1], free[ia] = bool(ftau), bool(ftau)
    dev = _evaluate(code, p, freqs, nu_ref, nbin, data, errs, free, jc)
    ref = restate_join(code, p, freqs, nu_ref, nbin, data, errs, jc, PSPIN)
    assert dev["return_code"][0] == 0 and dev["nfeval"][0] == 1
    assert np.array_equal(dev["params"][0], p)
    err = _sum_errors(dev, ref, free)
    assert err < SUM_TOL, err


def test_wrong_join_references_miss_by_ten_times_the_bound():
    """The phasor's sign flipped, the DM_j chain term dropped, the full complex phasor at the Nyquist term: each
    misses the device sums by more than 10 x SUM_TOL (narrow components at nbin 64, so that G_N is not
    negligible)."""
    code, nchan, nbin, njoin = "000", 8, 64, 3
    p, freqs, nu_ref, _, errs, jc = make_join_problem(code, nchan, nbin, njoin, tau=1.1, seed=4)
    ia = len(p) - 2 * njoin - 1
    p[4:ia:6] = 0.022                                 # wid of every component: about 1.4 bins
    p[ia + 1::2] = [0.11, -0.07, 0.23]                # phases large enough for sin(2 pi N theta) to matter
    rng = np.random.RandomState(8)
    data = model_time_join(code, p, freqs, nu_ref, nbin, jc, PSPIN) + 0.05 * rng.randn(nchan, nbin)
    errs = np.full(nchan, 0.05)
    free = np.ones(len(p), bool)
    dev = _evaluate(code, p, freqs, nu_ref, nbin, data, errs, free, jc)
    ref = restate_join(code, p, freqs, nu_ref, nbin, data, errs, jc, PSPIN)
    assert _sum_errors(dev, ref, free) < SUM_TOL
    for wrong in ("sign", "nodm", "nyquist"):
        miss = _sum_errors(dev, restate_join(code, p, freqs, nu_ref, nbin, data, errs, jc, PSPIN, wrong=wrong),
                           free, scale=ref)
        print("WRONG %s miss %.3g (bound %.3g)" % (wrong, miss, SUM_TOL))
        assert miss > 10 * SUM_TOL, (wrong, miss)


def test_no_groups_through_the_join_entry_is_the_plain_fit_bit_for_bit():
    code, nchan, nbin = "110", 16, 256
    from tests.test_cpu_gaussfit import make_problem
    probs = [make_problem(code, nchan, nbin, tau=0.9, seed=70 + s) for s in range(3)]
    freqs, nu_ref = probs[0][1], probs[0][2]
    data = np.stack([q[3] for q in probs])
    errs = np.stack([q[4] for q in probs])
    init = np.stack([q[0] * (1 + 0.01 * np.random.RandomState(s).randn(len(q[0]))) for s, q in enumerate(probs)])
    free = np.ones(init.shape[1], bool)
    with _plan(nchan, nbin, freqs) as pl:
        a = pl.fit_gaussian_portraits(data, errs, code, init, free, nu_ref, want_model=True, want_sums=True)
        b = pl.fit_gaussian_portraits(data, errs, code, init, free, nu_ref, want_model=True, want_sums=True,
                                      join_chan=np.full(nchan, -1), P=PSPIN)
    assert set(a) == set(b)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


# ---- optimum vs scipy ------------------------------------------------------------------------------------
def _scipy_fit(code, p0, freqs, nu_ref, nbin, data, errs, free, jc):
    from scipy.optimize import least_squares
    f = np.where(free)[0]

    def full(q):
        p = p0.copy()
        p[f] = q
        return p

    def fun(q):
        r = restate_join(code, full(q), freqs, nu_ref, nbin, data, errs, jc, PSPIN)
        sw = np.sqrt(r["w"])
        return np.concatenate([(sw * r["R"].real).ravel(), (sw * r["R"].imag).ravel()])

    def jac(q):
        r = restate_join(code, full(q), freqs, nu_ref, nbin, data, errs, jc, PSPIN)
        sw = np.sqrt(r["w"])[:, None, :]
        J = r["J"][:, f]
        return -np.concatenate([(sw * J.real).transpose(0, 2, 1).reshape(-1, len(f)),
                                (sw * J.imag).transpose(0, 2, 1).reshape(-1, len(f))])
    res = least_squares(fun, p0[f], jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    p = full(res.x)
    r = restate_join(code, p, freqs, nu_ref, nbin, data, errs, jc, PSPIN)
    cov = np.linalg.inv(r["jtj"][np.ix_(f, f)]) * r["chi2"] / (len(freqs) * nbin - len(f))
    errs_out = np.zeros(len(p))
    errs_out[f] = np.sqrt(np.diag(cov))
    return p, r["chi2"], errs_out


@pytest.mark.parametrize("code,njoin,tau,ftau", [("000", 1, 0.0, 0), ("110", 2, 1.5, 1), ("011", 3, 0.0, 0)])
def test_joined_optimum_matches_scipy(code, njoin, tau, ftau):
    nchan, nbin = 16, 256
    p_true, freqs, nu_ref, data, errs, jc = make_join_problem(code, nchan, nbin, njoin, tau=tau, seed=11 + njoin)
    P = len(p_true)
    ia = P - 2 * njoin - 1
    free = np.ones(P, bool)
    free[1], free[ia] = bool(ftau), bool(ftau)
    rng = np.random.RandomState(5)
    p0 = p_true.copy()
    ng = (ia - 2) // 6
    p0[2:ia:6] += 0.002 * rng.randn(ng)
    p0[4:ia:6] *= 1 + 0.03 * rng.randn(ng)
    p0[ia + 1::2] += 0.003 * rng.randn(njoin)
    p0[ia + 2::2] += 0.02 * rng.randn(njoin)
    if ftau:
        p0[1] += 0.3
    with _plan(nchan, nbin, freqs) as pl:
        dev = pl.fit_gaussian_portraits(data[None], errs[None], code, p0[None], free, nu_ref, join_chan=jc, P=PSPIN)
    assert dev["return_code"][0] == 0
    p_ref, chi2_ref, errs_ref = _scipy_fit(code, p0, freqs, nu_ref, nbin, data, errs, free, jc)
    f = np.where(free)[0]
    sig = dev["param_errs"][0][f]
    assert np.max(np.abs(dev["params"][0][f] - p_ref[f]) / sig) < 1e-3
    assert abs(dev["chi2"][0] / chi2_ref - 1.0) < 1e-8
    assert np.max(np.abs(dev["param_errs"][0][f] / errs_ref[f] - 1.0)) < 1e-4
    assert dev["cov"][0].shape == (P, P)


# ---- joined model ------------------------------------------------------------------------------------
@pytest.mark.parametrize("code,nbin,tau", [("000", 64, 0.0), ("011", 1024, 1.2), ("111", 4096, 0.4)])
def test_device_joined_model_matches_the_host_generator(code, nbin, tau):
    from pulseportraiture_b200 import pplib
    nchan, njoin = 12, 3
    p, freqs, nu_ref, _, _, jc = make_join_problem(code, nchan, nbin, njoin, tau=tau, seed=nbin)
    ia = len(p) - 2 * njoin - 1
    params = np.concatenate([p[:ia], p[ia + 1:]])
    ichans = [np.where(jc == j)[0] for j in range(njoin)]
    phases = pplib.get_bin_centers(nbin)
    dev = pplib.gen_gaussian_portrait_device(code, params, p[ia], phases, freqs, nu_ref, join_ichans=ichans, P=PSPIN)
    host = pplib.gen_gaussian_portrait(code, params, p[ia], phases, freqs, nu_ref, join_ichans=ichans, P=PSPIN)
    assert dev.dtype == np.float64 and dev.shape == (nchan, nbin)
    assert np.max(np.abs(dev - host)) < 1e-12 * np.max(np.abs(host))


# ---- recovery from simulated archives -------------------------------------------------------------------
BANDS = [(1300.0, 200.0), (820.0, 200.0), (1900.0, 300.0)]   # the reference archive first (the .gmodel's FREQ)
OFFSETS = [(0.0, 0.0), (0.031, -2.0e-3), (-0.017, 1.5e-3)]   # injected (phase, dDM) of each archive


def _joined_fit(seed, nchan=128, nbin=1024):
    from pulseportraiture_b200 import pplib
    Pspin = synth.P_EXAMPLE
    arch = [pplib.make_fake_pulsar(synth.GMODEL, Pspin, nchan=nchan, nbin=nbin, nu0=nu0, bw=bw, phase=ph, dDM=dm,
                                   nu_DM=1300.0, noise_stds=1.0, seed=seed * 10 + a, quiet=True)
            for a, ((nu0, bw), (ph, dm)) in enumerate(zip(BANDS, OFFSETS))]
    j = pplib.join_archives(arch)
    name, code, nu_ref, ngauss, params, flags, alpha, _ = pplib.read_model(synth.GMODEL)
    # the offsets and DC free, the components held at the .gmodel's values: the offsets' errors are then those of a
    # known profile, and their pulls test the join columns alone
    flags = np.zeros_like(flags)
    flags[0] = 1
    init = params.copy()
    jp = [j.join_ichans, np.zeros(2 * len(j.join_ichans)), np.ones(2 * len(j.join_ichans))]
    fit = pplib.fit_gaussian_portrait(code, j.port, init, alpha, j.noise_stds, flags, 0, pplib.get_bin_centers(nbin),
                                      j.freqs, nu_ref, join_params=jp, P=j.P)
    # make_fake_pulsar rotates the model by -(phase, dDM): the joined model's offsets are minus the injected ones
    # relative to the reference archive
    truth = -np.ravel([[ph - OFFSETS[0][0], dm - OFFSETS[0][1]] for ph, dm in OFFSETS[1:]])
    return fit, truth, (name, code, nu_ref, flags, j)


def test_injected_offsets_are_recovered():
    fit, truth, _ = _joined_fit(0)
    assert fit.return_code == 0, (fit.return_code, fit.nfeval)
    assert fit.join_params.shape == (4,) and fit.join_param_errs.shape == (4,)
    assert fit.covariance.shape == (len(fit.fitted_params) + 5,) * 2
    pulls = (fit.join_params - truth) / fit.join_param_errs
    print("JOIN pulls", pulls)
    assert np.all(np.abs(pulls) < 3.0), pulls


def test_offset_pulls_over_many_seeds():
    pulls = []
    for seed in range(1, 101):
        fit, truth, _ = _joined_fit(seed)
        assert fit.return_code == 0, (seed, fit.return_code, fit.nfeval)
        pulls.append((fit.join_params - truth) / fit.join_param_errs)
    pulls = np.array(pulls)
    print("JOIN pull mean", pulls.mean(axis=0), "std", pulls.std(axis=0))
    assert np.all(np.abs(pulls.mean(axis=0)) < 0.3)
    assert np.all((pulls.std(axis=0) > 0.8) & (pulls.std(axis=0) < 1.25))


# ---- batch invariance ---------------------------------------------------------------------------------
def test_joined_batch_equals_single_fits_bit_for_bit():
    code, nchan, nbin, njoin = "110", 24, 256, 2
    probs = [make_join_problem(code, nchan, nbin, njoin, tau=0.9, seed=40 + s) for s in range(6)]
    freqs, nu_ref, jc = probs[0][1], probs[0][2], probs[0][5]
    data = np.stack([q[3] for q in probs])
    errs = np.stack([q[4] for q in probs])
    init = np.stack([q[0] * (1 + 0.01 * np.random.RandomState(s).randn(len(q[0]))) for s, q in enumerate(probs)])
    free = np.ones(init.shape[1], bool)
    kw = dict(want_model=True, join_chan=jc, P=PSPIN)
    keys = ("params", "param_errs", "cov", "chi2", "red_chi2", "nfeval", "return_code", "model")
    with _plan(nchan, nbin, freqs) as pl:
        batch = pl.fit_gaussian_portraits(data, errs, code, init, free, nu_ref, **kw)
        singles = [pl.fit_gaussian_portraits(data[s:s + 1], errs[s:s + 1], code, init[s:s + 1], free, nu_ref, **kw)
                   for s in range(len(probs))]
        pl.set_chunk(4)
        chunked = pl.fit_gaussian_portraits(data, errs, code, init, free, nu_ref, **kw)
    assert (batch["return_code"] == 0).all()
    for k in keys:
        one = np.concatenate([s[k] for s in singles])
        assert np.array_equal(batch[k], one), k
        assert np.array_equal(chunked[k], one), k
    for s in (0, 4):
        want = model_time_join(code, batch["params"][s], freqs, nu_ref, nbin, jc, PSPIN)
        assert np.max(np.abs(batch["model"][s] - want)) < 1e-12 * np.max(np.abs(want))


# ---- facade: joined fit -> write_model -> GetTOAs ----------------------------------------------------------
def test_joined_model_times_the_reference_archive(tmp_path):
    from pulseportraiture_b200 import pplib, pptoas
    fit, _, (name, code, nu_ref, flags, j) = _joined_fit(500)
    assert fit.return_code == 0
    nbin = 1024
    out = np.array(fit.fitted_params)
    out[1] = out[1] * j.P / nbin                               # TAU in seconds
    path = str(tmp_path / "joined.gmodel")
    pplib.write_model(path, name, code, nu_ref, out, flags, fit.scattering_index, 0, quiet=True)
    nu0, bw = BANDS[0]
    dDM, phase = 3e-3, 0.21
    arch = pplib.make_fake_pulsar(synth.GMODEL, synth.P_EXAMPLE, nsub=4, nchan=128, nbin=nbin, nu0=nu0, bw=bw,
                                  phase=phase, dDM=dDM, noise_stds=1.0, seed=4242, quiet=True)
    gt = pptoas.GetTOAs([arch], path, quiet=True)
    gt.get_TOAs(quiet=True)
    for s in range(4):
        assert abs(gt.DMs[0][s] - dDM) < 3 * gt.DM_errs[0][s], (s, gt.DMs[0][s], gt.DM_errs[0][s])


# ---- errors ---------------------------------------------------------------------------------------------
def test_join_argument_errors_raise():
    from pulseportraiture_b200 import _ffi
    code, nchan, nbin, njoin = "000", 8, 64, 2
    p, freqs, nu_ref, data, errs, jc = make_join_problem(code, nchan, nbin, njoin, seed=1)
    free = np.ones(len(p), bool)
    with _plan(nchan, nbin, freqs) as pl:
        with pytest.raises(_ffi.PPError, match="period"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref, join_chan=jc, P=-1.0)
        bad = jc.copy()
        bad[jc == 0] = -1                                      # group 0 empty, group 1 in use
        with pytest.raises(_ffi.PPError, match="no channel"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref, join_chan=bad, P=PSPIN)
        bad = jc.copy()
        bad[0] = -2
        with pytest.raises(_ffi.PPError, match="not a group"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p[None], free, nu_ref, join_chan=bad, P=PSPIN)
        nine = np.arange(nchan, dtype=np.int32) % 9
        nine[-1] = 8
        p9 = np.concatenate([p[:len(p) - 2 * njoin], np.zeros(18)])
        with pytest.raises(_ffi.PPError, match="njoin"):
            pl.fit_gaussian_portraits(data[None], errs[None], code, p9[None], np.ones(len(p9), bool), nu_ref,
                                      join_chan=nine, P=PSPIN)
