"""CPU checks of join parameters in the evolving-Gaussian portrait fit.

This module holds the float64 numpy restatement of the joined model that pp_fit_gaussian_portraits_join,
WidebandPlan.fit_gaussian_portraits(join_chan=...) and pplib.gen_gaussian_portrait(join_ichans=...) follow
(tests/test_gpu_gaussjoin.py uses it as the reference):

    gport[join_ichans[j]] = rotate_data(gport[join_ichans[j]], phi_j, DM_j, P, freqs[join_ichans[j]], nu_ref)

applied to the unjoined (scattered) portrait of gen_gaussian_portrait.  Harmonic k of channel n of group j is
multiplied by e^{2 pi i k theta_n}, theta_n = phi_j + Dconst DM_j / P (nu_n^-2 - nu_ref^-2); the Nyquist term, which
irfft keeps real, by cos(2 pi N theta_n).  Channels in no group are not rotated.  The parameter vector is
[DC, tau, comps..., alpha, phi_1, DM_1, ..., phi_J, DM_J]."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests.test_cpu_gaussfit import make_problem, model_time, restate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DCONST = 0.000241 ** -1
PSPIN = 0.0047


# ---- restatement ------------------------------------------------------------------------------
def join_theta(pj, freqs, nu_ref, join_chan, Pspin, no_dm=False):
    """theta_n [nchan] of the join values pj = [phi_1, DM_1, ...]; 0 on channels in no group."""
    jc = np.asarray(join_chan)
    theta = np.zeros(len(freqs))
    on = jc >= 0
    dm = 0.0 if no_dm else pj[2 * jc[on] + 1] * DCONST / Pspin * (freqs[on] ** -2.0 - nu_ref ** -2.0)
    theta[on] = pj[2 * jc[on]] + dm
    return theta


def rotate_rows(port, theta):
    """irfft(e^{2 pi i k theta_n} rfft(port_n)) of every row, numpy float64 (irfft keeps Re of the Nyquist term)."""
    nbin = port.shape[-1]
    ph = np.exp(2j * np.pi * np.outer(theta, np.arange(nbin // 2 + 1)))
    return np.fft.irfft(ph * np.fft.rfft(port, axis=-1), n=nbin, axis=-1)


def model_time_join(code, p, freqs, nu_ref, nbin, join_chan, Pspin):
    """The joined portrait at p = [DC, tau, comps..., alpha, (phi_j, DM_j) x njoin]."""
    njoin = int(np.max(join_chan)) + 1
    ia = len(p) - 2 * njoin - 1
    g = model_time(code, p[:ia + 1], freqs, nu_ref, nbin)
    return rotate_rows(g, join_theta(p[ia + 1:], freqs, nu_ref, join_chan, Pspin))


def restate_join(code, p, freqs, nu_ref, nbin, data, errs, join_chan, Pspin, wrong=None):
    """Weighted Fourier-domain residual and Jacobian of the joined fit at p (as restate of test_cpu_gaussfit).

    ``wrong`` picks a deliberately wrong variant: 'sign' (e^{-2 pi i k theta}), 'nodm' (the DM_j chain term
    dropped), 'nyquist' (the full complex phasor at the Nyquist term)."""
    p = np.asarray(p, dtype=np.float64)
    freqs = np.asarray(freqs, dtype=np.float64)
    jc = np.asarray(join_chan)
    njoin = int(jc.max()) + 1
    ia = len(p) - 2 * njoin - 1
    base = restate(code, p[:ia + 1], freqs, nu_ref, nbin, data, errs)
    N = nbin // 2
    k = np.arange(N + 1)
    D = np.fft.rfft(data, axis=-1)
    M0 = D - base["R"]                                       # unjoined model spectra; M0[:, N] is real
    theta = join_theta(p[ia + 1:], freqs, nu_ref, jc, Pspin)
    sgn = -1.0 if wrong == "sign" else 1.0
    E = np.exp(sgn * 2j * np.pi * np.outer(theta, k))
    dE = sgn * 2j * np.pi * k[None, :] * E                   # dE/dtheta
    if wrong != "nyquist":
        dE[:, N] = -2 * np.pi * N * np.sin(2 * np.pi * N * theta) * sgn
        E[:, N] = np.cos(2 * np.pi * N * theta)
    M = E * M0
    J = np.concatenate([E[:, None, :] * base["J"], np.zeros((len(freqs), 2 * njoin, N + 1), complex)], axis=1)
    Jth = dE * M0
    kdm = DCONST / Pspin * (freqs ** -2.0 - nu_ref ** -2.0)
    for j in range(njoin):
        on = (jc == j)[:, None]
        J[:, ia + 1 + 2 * j] = on * Jth
        J[:, ia + 2 + 2 * j] = 0.0 if wrong == "nodm" else on * kdm[:, None] * Jth
    R = D - M
    w = base["w"]
    chi2 = np.sum(w * np.abs(R) ** 2)
    jtr = np.einsum("nk,nik->i", w, (np.conj(J) * R[:, None, :]).real)
    jtj = np.einsum("nk,nik,njk->ij", w, J.real, J.real) + np.einsum("nk,nik,njk->ij", w, J.imag, J.imag)
    return dict(R=R, J=J, w=w, chi2=chi2, jtr=jtr, jtj=jtj)


def join_groups(nchan, njoin):
    """join_chan [nchan]: the band in njoin + 1 contiguous parts, the first the reference (-1)."""
    jc = np.full(nchan, -1, dtype=np.int32)
    edges = np.linspace(0, nchan, njoin + 2).astype(int)
    for j in range(njoin):
        jc[edges[j + 1]:edges[j + 2]] = j
    return jc


def make_join_problem(code, nchan, nbin, njoin, tau=0.0, seed=0, sigma=0.05, ngauss=2, Pspin=PSPIN):
    """make_problem's parity-safe portrait with njoin groups rotated by small phase and DM offsets.
    Returns (p_true, freqs, nu_ref, data, errs, join_chan)."""
    p, freqs, nu_ref, _, errs = make_problem(code, nchan, nbin, tau=tau, seed=seed, sigma=sigma, ngauss=ngauss)
    rng = np.random.RandomState(seed + 1000)
    pj = np.ravel([[0.01 * rng.randn(), 0.05 * rng.randn()] for _ in range(njoin)])
    p = np.concatenate([p, pj])
    jc = join_groups(nchan, njoin)
    data = model_time_join(code, p, freqs, nu_ref, nbin, jc, Pspin) + sigma * rng.randn(nchan, nbin)
    return p, freqs, nu_ref, data, errs, jc


# ---- the restatement against itself ------------------------------------------------------------------
@pytest.mark.parametrize("code,tau,njoin", [("000", 0.0, 1), ("110", 1.3, 3), ("011", 0.7, 2)])
def test_restated_join_jacobian_equals_finite_differences(code, tau, njoin):
    nchan, nbin = 8, 128
    p, freqs, nu_ref, data, errs, jc = make_join_problem(code, nchan, nbin, njoin, tau=tau, seed=3)
    r = restate_join(code, p, freqs, nu_ref, nbin, data, errs, jc, PSPIN)
    Jt = np.fft.irfft(r["J"], n=nbin, axis=-1)
    for i in range(len(p)):
        if i == len(p) - 2 * njoin - 1 and tau == 0.0:
            assert np.max(np.abs(Jt[:, i])) == 0.0          # alpha moves nothing while tau = 0
            continue
        h = 1e-6 * max(abs(p[i]), 1e-2)
        pp, pm = p.copy(), p.copy()
        pp[i] += h
        pm[i] -= h
        fd = (model_time_join(code, pp, freqs, nu_ref, nbin, jc, PSPIN) -
              model_time_join(code, pm, freqs, nu_ref, nbin, jc, PSPIN)) / (2 * h)
        scale = np.max(np.abs(fd)) + 1e-300
        assert np.max(np.abs(Jt[:, i] - fd)) < 2e-6 * scale, i


@pytest.mark.parametrize("nbin", [64, 128, 256, 512, 1024, 2048, 4096])
@pytest.mark.parametrize("tau", [0.0, 1.7])
def test_fourier_chi2_equals_time_domain_chi2(nbin, tau):
    code, njoin = "000", 3
    p, freqs, nu_ref, data, errs, jc = make_join_problem(code, 6, nbin, njoin, tau=tau, seed=nbin)
    p[-2 * njoin:] += 0.003                                      # away from the truth
    r = restate_join(code, p, freqs, nu_ref, nbin, data, errs, jc, PSPIN)
    res = (data - model_time_join(code, p, freqs, nu_ref, nbin, jc, PSPIN)) / errs[:, None]
    want = np.sum(res * res)
    assert abs(r["chi2"] / want - 1.0) < 1e-12


def test_nyquist_rule_is_numpys_irfft():
    """The restated rotation, cos(2 pi N theta) at the Nyquist term, is irfft(e^{2 pi i k theta} rfft(x))."""
    rng = np.random.RandomState(2)
    nbin = 64
    x = rng.randn(5, nbin)
    theta = np.array([0.0, 0.013, -0.29, 0.5, 0.77])
    k = np.arange(nbin // 2 + 1)
    want = np.fft.irfft(np.exp(2j * np.pi * np.outer(theta, k)) * np.fft.rfft(x, axis=-1), n=nbin, axis=-1)
    X = np.fft.rfft(x, axis=-1)
    E = np.exp(2j * np.pi * np.outer(theta, k))
    E[:, -1] = np.cos(2 * np.pi * (nbin // 2) * theta)
    got = np.fft.irfft(E * X, n=nbin, axis=-1)
    assert np.max(np.abs(got - want)) < 1e-14 * np.max(np.abs(x))
    assert np.max(np.abs(rotate_rows(x, theta) - want)) < 1e-14 * np.max(np.abs(x))
    # a real Nyquist term, so that the real row it gives is exactly what the restatement's spectrum says
    assert np.allclose(np.fft.rfft(got, axis=-1)[:, -1].imag, 0.0, atol=1e-12)


def test_host_generator_is_the_restatement():
    from pulseportraiture_b200 import pplib
    code, nchan, nbin, njoin = "011", 9, 256, 2
    p, freqs, nu_ref, _, _, jc = make_join_problem(code, nchan, nbin, njoin, tau=0.9, seed=6)
    ia = len(p) - 2 * njoin - 1
    ichans = [np.where(jc == j)[0] for j in range(njoin)]
    got = pplib.gen_gaussian_portrait(code, np.concatenate([p[:ia], p[ia + 1:]]), p[ia], pplib.get_bin_centers(nbin),
                                      freqs, nu_ref, join_ichans=ichans, P=PSPIN)
    want = model_time_join(code, p, freqs, nu_ref, nbin, jc, PSPIN)
    assert np.max(np.abs(got - want)) < 1e-12 * np.max(np.abs(want))
    # the reference channels are the unjoined model
    unj = pplib.gen_gaussian_portrait(code, p[:ia], p[ia], pplib.get_bin_centers(nbin), freqs, nu_ref)
    assert np.array_equal(got[jc < 0], unj[jc < 0])


# ---- C struct ----------------------------------------------------------------------------------------
def test_join_struct_layout_matches_the_header(tmp_path):
    from pulseportraiture_b200 import _ffi
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ppb200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu\\n", sizeof(pp_gfit_join_t),'
                   'offsetof(pp_gfit_join_t, njoin), offsetof(pp_gfit_join_t, join_chan),'
                   'offsetof(pp_gfit_join_t, P));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    J = _ffi.GfitJoin
    assert got == [C.sizeof(J), J.njoin.offset, J.join_chan.offset, J.P.offset]
    assert "pp_fit_gaussian_portraits_join" in _ffi.SYMBOLS


# ---- facade argument checks ---------------------------------------------------------------------------
def test_facade_join_argument_checks_need_no_gpu():
    from pulseportraiture_b200 import pplib
    nchan, nbin = 8, 64
    args = ("000", np.zeros((nchan, nbin)), np.zeros(8), -4.0, np.ones(nchan), np.ones(8), 0,
            pplib.get_bin_centers(nbin), np.linspace(1e3, 2e3, nchan), 1500.)
    for bad in ([1], [0.1], [[1], [0.0, 0.0]]):                   # not a three-part sequence
        with pytest.raises(NotImplementedError):
            pplib.fit_gaussian_portrait(*args, join_params=bad, P=PSPIN)
    good = [[np.arange(4, 8)], [0.0, 0.0], [1, 1]]
    with pytest.raises(ValueError, match="period"):               # P missing
        pplib.fit_gaussian_portrait(*args, join_params=good)
    with pytest.raises(ValueError, match="overlaps"):
        pplib.fit_gaussian_portrait(*args, join_params=[[[2, 3], [3, 4]], [0.0] * 4, [1] * 4], P=PSPIN)
    with pytest.raises(ValueError, match="out of range"):
        pplib.fit_gaussian_portrait(*args, join_params=[[[6, 8]], [0.0, 0.0], [1, 1]], P=PSPIN)
    with pytest.raises(ValueError, match="out of range"):
        pplib.fit_gaussian_portrait(*args, join_params=[[[-1]], [0.0, 0.0], [1, 1]], P=PSPIN)
    with pytest.raises(ValueError, match="empty"):
        pplib.fit_gaussian_portrait(*args, join_params=[[[]], [0.0, 0.0], [1, 1]], P=PSPIN)
    with pytest.raises(ValueError, match="at most 8"):
        pplib.fit_gaussian_portrait("000", np.zeros((9, nbin)), np.zeros(8), -4.0, np.ones(9), np.ones(8), 0,
                                    pplib.get_bin_centers(nbin), np.linspace(1e3, 2e3, 9), 1500.,
                                    join_params=[[[i] for i in range(9)], [0.0] * 18, [1] * 18], P=PSPIN)
    with pytest.raises(ValueError, match="2 entries"):
        pplib.fit_gaussian_portrait(*args, join_params=[[np.arange(4, 8)], [0.0], [1]], P=PSPIN)
    with pytest.raises(ValueError, match="period"):
        pplib.gen_gaussian_portrait("000", np.zeros(10), -4.0, pplib.get_bin_centers(nbin),
                                    np.linspace(1e3, 2e3, nchan), 1500., join_ichans=[[1]], P=0.0)
    doc = pplib.fit_gaussian_portrait.__doc__
    assert "not supported" not in doc and "join_params" in doc


# ---- join_archives --------------------------------------------------------------------------------------
def _npz_archive(path, nsub, freqs, nbin, P, zap, seed):
    from pulseportraiture_b200 import pplib, pptoas
    rng = np.random.RandomState(seed)
    nchan = len(freqs)
    w = np.ones((nsub, nchan))
    w[:, zap] = 0.0
    d = pplib.DataBunch(
        arch=None, backend="fake", backend_delay=0.0, bw=float(np.ptp(freqs)), doppler_factors=np.ones(nsub), DM=0.0,
        dmc=0, epochs=[pptoas.MJD(56000, 0.1 * s) for s in range(nsub)], filename=str(path), flux_prof=None,
        freqs=np.tile(freqs, (nsub, 1)), frontend="fake", integration_length=60.0 * nsub, masks=None, nbin=nbin,
        nchan=nchan, noise_stds=np.ones((nsub, 1, nchan)), npol=1, nsub=nsub, nu0=float(np.mean(freqs)),
        ok_ichans=[np.where(w[s] > 0)[0] for s in range(nsub)], ok_isubs=np.arange(nsub),
        parallactic_angles=np.zeros(nsub), phases=orc.get_bin_centers(nbin), prof=None, prof_noise=None,
        prof_SNR=None, Ps=np.full(nsub, P), SNRs=np.ones((nsub, 1, nchan)), source="J0000+0000",
        state="Intensity", subints=rng.randn(nsub, 1, nchan, nbin), subtimes=np.full(nsub, 60.0),
        telescope="GBT", telescope_code="GBT", weights=w, raw_subints=None, dat_scl=None, dat_offs=None)
    pptoas.save_databunch(str(path), d)
    return d


def test_join_archives_concatenates_the_usable_channels(tmp_path, monkeypatch):
    from pulseportraiture_b200 import pplib

    class _NoisePlan(object):   # tscrunch_databunch's get_noise, in numpy
        def get_noise_batch(self, x):
            return np.stack([orc.get_noise(np.asarray(r, dtype=np.float64), chans=True) for r in x])
    monkeypatch.setattr(pplib, "get_plan", lambda nchan, nbin, device=None: _NoisePlan())
    nbin = 64
    specs = [(np.linspace(700., 900., 6), [1], 0.0051), (np.linspace(1200., 1600., 8), [0, 5, 7], 0.0052),
             (np.linspace(2000., 2400., 4), [], 0.0053)]
    paths, ds = [], []
    for a, (f, zap, P) in enumerate(specs):
        path = tmp_path / ("a%d.npz" % a)
        ds.append(_npz_archive(path, 3, f, nbin, P, zap, seed=a))
        paths.append(str(path))
    j = pplib.join_archives([paths[0], ds[1], paths[2]], ref=1)
    oks = [np.setdiff1d(np.arange(len(f)), zap) for f, zap, _ in specs]
    n = [len(o) for o in oks]
    assert j.port.shape == (sum(n), nbin) and j.freqs.shape == (sum(n),) and j.noise_stds.shape == (sum(n),)
    assert j.P == specs[1][2] and j.nbin == nbin
    assert [list(a) for a in j.archive_ichans] == [list(range(0, n[0])), list(range(n[0], n[0] + n[1])),
                                                   list(range(n[0] + n[1], sum(n)))]
    assert [list(a) for a in j.join_ichans] == [list(j.archive_ichans[0]), list(j.archive_ichans[2])]
    for a, (f, _, _) in enumerate(specs):
        ich = j.archive_ichans[a]
        assert np.array_equal(j.freqs[ich], f[oks[a]])
        want = np.asarray(ds[a].subints)[:, 0][:, oks[a]].mean(axis=0)     # equal weights: the subint mean
        assert np.allclose(j.port[ich], want, rtol=0, atol=1e-12)
    with pytest.raises(ValueError, match="nbin"):
        other = tmp_path / "b.npz"
        _npz_archive(other, 1, np.linspace(700., 900., 6), 128, 0.005, [], seed=9)
        pplib.join_archives([paths[0], str(other)])
