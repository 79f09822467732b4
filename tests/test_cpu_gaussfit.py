"""CPU checks of the evolving-Gaussian portrait fit: the float64 numpy restatement of its Fourier-domain
objective, local columns and chain rule (used by tests/test_gpu_gaussfit.py as the reference), the
.gmodel writer, and the layout of the new C structs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import pp_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- restatement ------------------------------------------------------------------------------
def model_time(code, p, freqs, nu_ref, nbin):
    """gen_gaussian_portrait (pplib.py:853-930) at p = [DC, tau_bin, comps..., alpha], via the oracle."""
    ng = (len(p) - 3) // 6
    gm = dict(code=code, nu_ref=nu_ref, dc=p[0], tau=p[1] / nbin, alpha=p[-1],
              comps=np.asarray(p[2:-1], dtype=np.float64).reshape(ng, 6))
    return orc.gen_gaussian_portrait(gm, orc.get_bin_centers(nbin), freqs, P=1.0)


def local_of(i, P, L):
    if i == 0:
        return 0
    if i in (1, P - 1):
        return L - 1
    j = i - 2
    return 1 + 3 * (j // 6) + (j % 6) // 2


def restate(code, p, freqs, nu_ref, nbin, data, errs, wrong=None):
    """Weighted Fourier-domain residual and Jacobian of the fit at p.

    Returns dict(R [nchan, N+1] residual spectra, J [nchan, P, N+1] model derivative spectra, w
    [nchan, N+1] Parseval weights 1/(nbin sigma^2) x (1 or 2), chi2, jtr, jtj).  ``wrong`` picks a
    deliberately wrong variant: 'nyquist' (M_N = B_N G_N), 'nodc' (harmonic 0 dropped), 'alpha_nolog'
    (the alpha chain without ln(nu/nu_ref))."""
    p = np.asarray(p, dtype=np.float64)
    freqs = np.asarray(freqs, dtype=np.float64)
    P = len(p)
    ng = (P - 3) // 6
    L = 2 + 3 * ng
    nchan, N = len(freqs), nbin // 2
    x = orc.get_bin_centers(nbin)
    lr = np.log(freqs) - np.log(nu_ref)
    comps = p[2:-1].reshape(ng, 6)

    def ev(base, m, c):
        if c == "0":
            return np.exp(np.outer(lr, m) + np.log(base)[None, :])
        return np.outer(freqs - nu_ref, m) + base[None, :]
    vals = [ev(comps[:, 2 * q], comps[:, 2 * q + 1], code[q]) for q in range(3)]   # loc, wid, amp [nchan, ng]
    g = np.full((nchan, nbin), p[0])
    cols = np.zeros((nchan, L, nbin))
    cols[:, 0] = 1.0
    for n in range(nchan):
        for ig in range(ng):
            loc, wid, amp = vals[0][n, ig], vals[1][n, ig], vals[2][n, ig]
            if not wid > 0:
                continue
            sig = wid / (2 * np.sqrt(2 * np.log(2)))
            mean = loc % 1.0
            xw = np.where(x > mean + 0.5, x - 1.0, x) if mean < 0.5 else np.where(x < mean - 0.5, x + 1.0, x)
            z = (xw - mean) / sig
            near = np.abs(z) < 20.0
            e = np.where(near, np.exp(-0.5 * np.where(near, z, 0.0) ** 2), 0.0)
            if e.max() == 0.0:
                continue
            ipk = e.argmax()
            ratio = np.exp(-0.5 * ((xw[ipk] - loc) / sig) ** 2) / e[ipk]
            scale = amp * ratio
            g[n] += scale * e
            cols[n, 1 + 3 * ig] = scale * e * z / sig
            cols[n, 2 + 3 * ig] = scale * e * z * z / wid
            cols[n, 3 + 3 * ig] = ratio * e
    G = np.fft.rfft(g, axis=-1)
    Cf = np.fft.rfft(cols, axis=-1)
    k = np.arange(N + 1)
    tau_n = p[1] / nbin * (freqs / nu_ref) ** p[-1]
    B = 1.0 / (1.0 + 2j * np.pi * np.outer(tau_n, k))
    T = -2j * np.pi * k[None, :] * B ** 2
    if wrong != "nyquist":
        B[:, N] = B[:, N].real
        T[:, N] = T[:, N].real
    M = B * G
    Jl = B[:, None, :] * Cf
    Jl[:, L - 1] = T * G
    R = np.fft.rfft(data, axis=-1) - M
    w = np.full((nchan, N + 1), 2.0)
    w[:, 0] = w[:, N] = 1.0
    if wrong == "nodc":
        w[:, 0] = 0.0
    w /= nbin * np.asarray(errs, dtype=np.float64)[:, None] ** 2
    c = np.zeros((nchan, P))
    c[:, 0] = 1.0
    c[:, 1] = (freqs / nu_ref) ** p[-1] / nbin
    c[:, P - 1] = tau_n * (1.0 if wrong == "alpha_nolog" else lr)
    for ig in range(ng):
        for q in range(3):
            i = 2 + 6 * ig + 2 * q
            if code[q] == "1":
                c[:, i], c[:, i + 1] = 1.0, freqs - nu_ref
            else:
                c[:, i], c[:, i + 1] = np.exp(lr * p[i + 1]), vals[q][:, ig] * lr
    J = np.stack([c[:, i, None] * Jl[:, local_of(i, P, L)] for i in range(P)], axis=1)
    chi2 = np.sum(w * np.abs(R) ** 2)
    jtr = np.einsum("nk,nik->i", w, (np.conj(J) * R[:, None, :]).real)
    jtj = np.einsum("nk,nik,njk->ij", w, J.real, J.real) + np.einsum("nk,nik,njk->ij", w, J.imag, J.imag)
    return dict(R=R, J=J, w=w, chi2=chi2, jtr=jtr, jtj=jtj)


def chi2_time(code, p, freqs, nu_ref, nbin, data, errs):
    r = (data - model_time(code, p, freqs, nu_ref, nbin)) / np.asarray(errs)[:, None]
    return np.sum(r * r)


def make_problem(code, nchan, nbin, tau=0.0, alpha=-4.0, seed=0, sigma=0.05, ngauss=2, nu0=1500., bw=400.):
    """A parity-safe problem: every loc_n in (0.05, 0.95) and every component negligible half a turn from
    its centre across the band.  Returns (p_true, freqs, nu_ref, data, errs)."""
    rng = np.random.RandomState(seed)
    freqs = orc.make_freqs(nchan, nu0, bw)
    nu_ref = nu0 + 17.0
    comps = []
    for ig in range(ngauss):
        loc = 0.3 + 0.35 * ig / max(1, ngauss - 1) + 0.01 * rng.randn()
        wid, amp = 0.04 + 0.01 * rng.rand(), 1.0 + rng.rand()
        m = [0.0, 0.0, 0.0]
        for q, (lin, pl) in enumerate(((2e-5, 0.02), (1e-5, -0.3), (1e-4, -0.8))):
            m[q] = (lin if code[q] == "1" else pl) * (1 + 0.3 * rng.randn())
        comps += [loc, m[0], wid, m[1], amp, m[2]]
    p = np.array([0.05, tau] + comps + [alpha])
    clean = model_time(code, p, freqs, nu_ref, nbin)
    data = clean + sigma * rng.randn(nchan, nbin)
    errs = sigma * (1.0 + 0.2 * rng.rand(nchan))
    return p, freqs, nu_ref, data, errs


def _fd_jacobian(code, p, freqs, nu_ref, nbin, free):
    cols = []
    for i in np.where(free)[0]:
        h = 1e-6 * max(abs(p[i]), 1e-2)
        pp, pm = p.copy(), p.copy()
        pp[i] += h
        pm[i] -= h
        cols.append((model_time(code, pp, freqs, nu_ref, nbin) - model_time(code, pm, freqs, nu_ref, nbin)) / (2 * h))
    return np.stack(cols, axis=-1)


@pytest.mark.parametrize("code", ["000", "110", "011"])
@pytest.mark.parametrize("tau", [0.0, 1.3])
def test_restated_jacobian_equals_finite_differences(code, tau):
    nchan, nbin = 6, 128
    p, freqs, nu_ref, data, errs = make_problem(code, nchan, nbin, tau=tau, seed=3)
    free = np.ones(len(p), bool)
    r = restate(code, p, freqs, nu_ref, nbin, data, errs)
    Jt = np.fft.irfft(r["J"], n=nbin, axis=-1)           # time-domain columns [nchan, P, nbin]
    fd = _fd_jacobian(code, p, freqs, nu_ref, nbin, free)  # [nchan, nbin, P]
    for i in range(len(p)):
        scale = np.max(np.abs(fd[:, :, i])) + 1e-300
        if i == len(p) - 1 and tau == 0.0:
            assert np.max(np.abs(Jt[:, i])) == 0.0          # alpha moves nothing while tau = 0
            continue
        assert np.max(np.abs(Jt[:, i] - fd[:, :, i])) < 2e-6 * scale, i


@pytest.mark.parametrize("code,tau,nbin", [("000", 0.0, 64), ("110", 2.5, 64), ("011", 0.7, 256)])
def test_fourier_chi2_equals_time_domain_chi2(code, tau, nbin):
    p, freqs, nu_ref, data, errs = make_problem(code, 5, nbin, tau=tau, seed=5)
    r = restate(code, p, freqs, nu_ref, nbin, data, errs)
    want = chi2_time(code, p, freqs, nu_ref, nbin, data, errs)
    assert abs(r["chi2"] / want - 1.0) < 1e-13
    # the Nyquist and DC terms matter: the wrong variants miss (the Nyquist term only where G_N is not tiny)
    if tau and nbin == 64:
        assert abs(restate(code, p, freqs, nu_ref, nbin, data, errs, wrong="nyquist")["chi2"] / want - 1) > 1e-12
    assert abs(restate(code, p, freqs, nu_ref, nbin, data, errs, wrong="nodc")["chi2"] / want - 1) > 1e-6


def test_tau_zero_with_free_tau_has_the_tau_column():
    """At tau = 0 the tau column is -2 pi i k G_k (B = 1): d chi^2 / d tau agrees with a one-sided
    difference into tau > 0 (the model is smooth through tau = 0)."""
    code, nbin = "000", 128
    p, freqs, nu_ref, data, errs = make_problem(code, 4, nbin, tau=0.0, seed=9)
    r = restate(code, p, freqs, nu_ref, nbin, data, errs)
    h = 1e-6
    ph, pm = p.copy(), p.copy()
    ph[1], pm[1] = h, -h
    fd = (model_time(code, ph, freqs, nu_ref, nbin) - model_time(code, pm, freqs, nu_ref, nbin)) / (2 * h)
    Jt = np.fft.irfft(r["J"][:, 1], n=nbin, axis=-1)
    assert np.max(np.abs(Jt - fd)) < 1e-6 * np.max(np.abs(fd))
    assert abs(r["chi2"] / chi2_time(code, p, freqs, nu_ref, nbin, data, errs) - 1) < 1e-13


# ---- write_model / read_model -------------------------------------------------------------------
def test_write_model_round_trip(tmp_path):
    from pulseportraiture_b200 import pplib
    code, nbin = "011", 256
    p, freqs, nu_ref, _, _ = make_problem(code, 16, nbin, tau=1.7, alpha=-3.7, seed=2, ngauss=3)
    Pspin = 0.00289
    params = p[:-1].copy()
    params[1] = p[1] * Pspin / nbin                        # TAU in seconds: tau_bin * P / nbin
    flags = np.array([1, 1] + [1, 0, 1, 1, 0, 1] * 3)
    path = str(tmp_path / "fit.gmodel")
    pplib.write_model(path, "J0000+0000", code, nu_ref, params, flags, p[-1], 1, quiet=True)
    name, code2, nu2, ng, params2, flags2, alpha2, fit_alpha2 = pplib.read_model(path)
    assert (name, code2, ng, fit_alpha2) == ("J0000+0000", code, 3, 1)
    assert nu2 == pytest.approx(nu_ref, abs=5e-11) and alpha2 == pytest.approx(p[-1], abs=5e-13)
    assert np.max(np.abs(params2 - params)) <= 5e-13
    assert np.array_equal(flags2, flags)
    _, _, port = pplib.read_model(path, pplib.get_bin_centers(nbin), freqs, Pspin, quiet=True)
    want = model_time(code, p, freqs, nu_ref, nbin)
    assert np.max(np.abs(port - want)) < 1e-8 * np.max(np.abs(want))
    # append=True adds a second model to the file
    pplib.write_model(path, "second", code, nu_ref, params, flags, p[-1], 1, append=True, quiet=True)
    assert open(path).read().count("MODEL") == 2


# ---- C structs --------------------------------------------------------------------------------
def test_gfit_struct_layouts_match_the_header(tmp_path):
    from pulseportraiture_b200 import _ffi
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ppb200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(pp_gfit_args_t), offsetof(pp_gfit_args_t, model_code), offsetof(pp_gfit_args_t, ngauss),'
                   'offsetof(pp_gfit_args_t, nu_ref), offsetof(pp_gfit_args_t, fit_flags),'
                   'offsetof(pp_gfit_args_t, max_iter), offsetof(pp_gfit_args_t, tol),'
                   'sizeof(pp_gfit_out_t), offsetof(pp_gfit_out_t, model));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    A, O = _ffi.GfitArgs, _ffi.GfitOut
    want = [C.sizeof(A), A.model_code.offset, A.ngauss.offset, A.nu_ref.offset, A.fit_flags.offset,
            A.max_iter.offset, A.tol.offset, C.sizeof(O), O.model.offset]
    assert got == want


def test_facade_argument_checks_need_no_gpu():
    from pulseportraiture_b200 import pplib
    with pytest.raises(NotImplementedError):
        pplib.fit_gaussian_portrait("000", np.zeros((4, 64)), np.zeros(8), -4.0, np.ones(4), np.ones(8), 0,
                                    pplib.get_bin_centers(64), np.linspace(1e3, 2e3, 4), 1500., join_params=[1])
    b = pplib._gauss_default_bounds("011", 2)
    assert b.shape == (15, 2) and b[1, 0] == 0.0 and np.isnan(b[0]).all()
    assert list(b[4]) == [pplib._gauss_wid_min, pplib.wid_max] and 0.0 < pplib._gauss_wid_min   # 0 < wid
    assert b[6, 0] == 0.0 and b[2, 0] == 0.0                                            # power-law loc: >= 0
    assert np.isnan(pplib._gauss_default_bounds("100", 1)[2]).all()                    # linear loc: open
    # the docstring carries the bounds policy and says that lm_results cannot be provided
    doc = pplib.fit_gaussian_portrait.__doc__
    assert doc and "0 < wid <= wid_max" in doc and "lm_results" in doc
