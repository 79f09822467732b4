"""The Fourier-domain row kernels -- rotation, response, scattering and both ppalign sums -- against a float64
restatement at every row plan.

Every entry point here computes y = irfft(H * rfft(x)) per row, or a weighted sum of such rows, with
H_nk = e^{2 pi i k theta_n} for a rotation (theta_n = phi + Dconst DM (nu_n^-2 - nu_ref^-2)/P
+ Dconst^2 GM (nu_n^-4 - nu_GM^-4)/P), times 1/(1 + 2 pi i k tau_n) for scattering and times resp[n, k] for a
response; irfft keeps the real part of the Nyquist term.  Power-of-two nbin runs k_rotate<N, float> (fft_precision
0/32), k_rotate<N, double> (64, response, scattering) and k_align_accum; any other even nbin runs k_fwd_any, k_rot_mul
and k_inv_any (Bluestein or mixed radix, always double), and pp_align_accumulate adds the rotated spectra in double
(k_wsum_spec) before one inverse transform per channel.  The fused sum of pp_fit_batch(align) adds the float2 data
spectra the fit keeps (k_align_spec) and finishes with k_align_finish / k_align_reduce_any + k_inv_any.

The references are numpy float64 on exactly the values the device reads (float32 data held in float64); the phase
k theta is formed in long double and reduced to one turn before the phasor, so the reference's own phase error is
below the device's wherever long double is wider than double.  Error model, per output sample j of row n
(u = 2^-53, L = nbin/2, ||x|| the row's 2-norm, |y_j| the reference value):

  output rounding     2^-24 |y_j| for float32 output (0 for the float64 ppalign sums);
  phase               theta_n is formed with relative rounding u on terms of total size A_n = |theta_n|
                      + 4 |Dconst DM/P| (nu^-2 + nu_ref^-2) + 4 |Dconst^2 GM/P| (nu^-4 + nu_GM^-4) (the difference of
                      the nu^-2 terms cancels), k theta costs u k/2 after the reduction, cis2pi u: a phasor error of
                      at most 2 pi u (L (2 A_n + 1/2) + 2) radians at every harmonic, which reaches a sample as at most
                      that times ||x|| (Parseval, |H| <= 1);
  double transforms   u (40 log2 nbin + 40) ||x||: forward and inverse radix-4/8 FFTs, the real-FFT split, and the
                      three length-M transforms and chirp products of Bluestein;
  float transform     2^-24 (6 log2 nbin + 8) ||x|| instead (k_rotate<N, float>: float twiddles, the float phasor);
  response            the transform terms times max_k |resp_nk|.

A sum over subints gets sum_s |w_sn| ||x_sn|| in place of ||x|| (plus nsub u for the double accumulation).  The fused
sum adds the storage of the data spectra as float2: eps_k = 2^-24 sum_s |w_sn| (|Re d_snk| + |Im d_snk|) at every
harmonic 1..L (the DC term is kept in double), which reaches a sample as at most (2/nbin) sum_k eps_k.

Each case also builds deliberately wrong references (Nyquist or DC term dropped, the response or scattering factor
missing at the Nyquist term or resp[N] applied at DC, the GM term about nu_DM, subint 0's nu_ref and P for every
subint, |w| for negative weights, rotated rows rounded to float32 before the double sum, the fused theta about nu_fit
instead of nu_out); each must miss the correct reference by at least 10x its tolerance, so the tolerance could not
let that mistake through.
"""
import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests import synth

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
U32 = 2.0 ** -24
UL = float(np.finfo(np.longdouble).eps) / 2        # unit roundoff of the reference's phase arithmetic
LD = np.longdouble
# (nbin, force Bluestein): every k_rotate N = 32..2048, Bluestein (66, 1002, 4094), mixed radix (1000, 1536) and a
# mixed-radix size kept on the chirp-z path
PLANS = [(n, False) for n in (64, 128, 256, 512, 1024, 2048, 4096, 66, 1002, 4094, 1000, 1536)] + [(1000, True)]
PLAN_IDS = ["%d%s" % (n, "-bluestein" if f else "") for n, f in PLANS]
MISS = 10.0


def _pow2(nbin):
    return nbin & (nbin - 1) == 0


def _plan(nchan, nbin, force, monkeypatch):
    from pulseportraiture_b200.engine import WidebandPlan
    if force:
        monkeypatch.setenv("PP_FORCE_BLUESTEIN", "1")
    else:
        monkeypatch.delenv("PP_FORCE_BLUESTEIN", raising=False)
    return WidebandPlan(nchan, nbin)


def c_fft64(nbin):
    return U * (40.0 * np.log2(nbin) + 40.0)


def c_fft32(nbin):
    return U32 * (6.0 * np.log2(nbin) + 8.0)


def theta_rows(freqs, phase, DM, P, nu_ref, GM=None, nu_GM=None):
    """theta [nsub, nchan] in long double and the size A [nsub, nchan] of the terms the device rounds"""
    col = lambda v: np.asarray(v, dtype=np.float64).astype(LD)[:, None]     # noqa: E731
    f = np.asarray(freqs, dtype=np.float64).astype(LD)[None, :]
    D = LD(orc.Dconst)
    kd = D * col(DM) / col(P)
    th = col(phase) + kd * (f ** -2 - col(nu_ref) ** -2)
    A = np.abs(th) + 4 * np.abs(kd) * (f ** -2 + col(nu_ref) ** -2)
    if GM is not None:
        kg = D * D * col(GM) / col(P)
        th = th + kg * (f ** -4 - col(nu_GM) ** -4)
        A = A + 4 * np.abs(kg) * (f ** -4 + col(nu_GM) ** -4)
    return th, A.astype(np.float64)


def phasors(theta, L):
    """e^{2 pi i k theta} for k = 0..L ([..., L + 1]), k theta reduced to one turn in long double"""
    a = theta[..., None] * np.arange(L + 1, dtype=LD)
    a -= np.rint(a)
    return np.exp(2j * np.pi * a.astype(np.float64))


def c_phase(A, L):
    """phasor error [rad] of the device plus the reference's, per row of size A"""
    return 2 * np.pi * (U * (L * (2 * A + 0.5) + 2) + UL * (L * (2 * A + 1) + 2))


def irfft_rows(X, nbin):
    return np.fft.irfft(X, n=nbin, axis=-1)


def miss(wrong, ref, tol):
    """min over what a wrong reference gets wrong: max_j |wrong - ref| / tol"""
    return float(np.max(np.abs(wrong - ref) / tol))


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


def _rows(rng, nsub, nchan, nbin, noise=1.0, amp=3.0, wid=0.02, dc=0.7, alt=0.5):
    """float32 rows: noise, a pulse at a random phase, a DC offset and a Nyquist-frequency component"""
    j = np.arange(nbin)
    x = noise * rng.standard_normal((nsub, nchan, nbin))
    loc = rng.uniform(0, 1, (nsub, nchan, 1))
    d = (j / nbin - loc + 0.5) % 1.0 - 0.5
    x += amp * np.exp(-0.5 * (d / wid) ** 2) + dc + alt * (-1.0) ** j
    return x.astype(np.float32).astype(np.float64)


# ---------------------------------------------------------------------------------------------------------------
# rotation: pp_rotate_batch / pp_rotate_full_batch
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_rotate_rows_against_float64(nbin, force, monkeypatch):
    import torch
    nsub, nchan, L = 3, 7, nbin // 2         # 21 rows: not a multiple of RowGeom<N>::kRows
    rng = np.random.RandomState(nbin + 17 * force)
    freqs = orc.make_freqs(nchan, 1500., 800.)
    x = _rows(rng, nsub, nchan, nbin)
    phase = np.array([0.4999, -0.4999, 0.123])
    DM = np.array([2.0, 0.0, -1.3])            # theta spans > 1 turn across the band; DM = 0 skips the DM term
    P = np.array([0.0031, 0.0029, 0.0045])
    nu_ref = np.array([1400., 1700., 1250.])
    GM = np.array([2.0, 0.0, -1.5])
    nu_GM = np.array([900., 1000., 1800.])
    X = np.fft.rfft(x, axis=-1)
    nx = np.linalg.norm(x, axis=-1)[..., None]
    any_n = not _pow2(nbin)

    def ref_of(th):
        return irfft_rows(X * phasors(th, L), nbin)

    def drop_nyq(th):
        H = phasors(th, L)
        H[..., L] = 0.0
        return irfft_rows(X * H, nbin)

    th, A = theta_rows(freqs, phase, DM, P, nu_ref)
    thg, Ag = theta_rows(freqs, phase, DM, P, nu_ref, GM, nu_GM)
    th_gdm, _ = theta_rows(freqs, phase, DM, P, nu_ref, GM, nu_ref)                  # GM about nu_DM
    th_s0, _ = theta_rows(freqs, phase, DM, np.full(nsub, P[0]), np.full(nsub, nu_ref[0]))   # subint 0's P, nu_ref
    ref, refg = ref_of(th), ref_of(thg)
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        pl.set_freqs(freqs)
        out = {}
        for bits in (0, 64):
            pl.set_fft_precision(bits)
            out[bits] = np.asarray(pl.rotate_batch(x.astype(np.float32), phase, DM, P, nu_ref), dtype=np.float64)
            out["g%d" % bits] = np.asarray(pl.rotate_batch(x.astype(np.float32), phase, DM, P, nu_ref, GM=GM, nu_GM=nu_GM),
                                           dtype=np.float64)
        # a CUDA tensor, out of place and in place (in/out may alias): the same bits
        pl.set_fft_precision(0)
        xt = torch.from_numpy(x.astype(np.float32)).cuda()
        dev = pl.rotate_batch(xt, phase, DM, P, nu_ref, GM=GM, nu_GM=nu_GM).cpu().numpy()
        pl.rotate_batch(xt, phase, DM, P, nu_ref, out=xt, GM=GM, nu_GM=nu_GM)
        torch.cuda.synchronize()
        inplace = xt.cpu().numpy()
    assert np.array_equal(dev, inplace)
    assert np.array_equal(dev.astype(np.float64), out["g0"])
    for bits in (0, 64):
        double = bits == 64 or any_n
        cf = c_fft64(nbin) if double else c_fft32(nbin)
        tol = U32 * np.abs(ref) + (cf + c_phase(A, L)[..., None]) * nx
        tolg = U32 * np.abs(refg) + (cf + c_phase(Ag, L)[..., None]) * nx
        kind = "rotate%s-%s" % ("64" if double else "32", PLAN_IDS[PLANS.index((nbin, force))])
        check(out[bits], ref, tol, {"nyquist": drop_nyq(th), "subint0_P_nuref": ref_of(th_s0)}, kind)
        check(out["g%d" % bits], refg, tolg, {"nyquist": drop_nyq(thg), "GM_about_nuDM": ref_of(th_gdm)}, kind + "-GM")


# ---------------------------------------------------------------------------------------------------------------
# response: pp_apply_response_batch
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_apply_response_against_float64(nbin, force, monkeypatch):
    from pulseportraiture_b200 import pptoaslib
    nsub, nchan, L = 3, 7, nbin // 2
    rng = np.random.RandomState(100 + nbin + 17 * force)
    freqs = orc.make_freqs(nchan, 1500., 800.)
    x = _rows(rng, nsub, nchan, nbin)
    X = np.fft.rfft(x, axis=-1)
    nx = np.linalg.norm(x, axis=-1)[..., None]
    resp = rng.uniform(-1.5, 1.5, (nchan, L + 1))
    resp[:, 0] = 0.8                           # resp[0] != 1
    resp[:, L] = -0.7                          # a distinct Nyquist value
    resp[:, 3] = 0.0
    resp[2, 5:9] = 0.0
    # a smearing-rectangle table as the facade builds it (real for a response centred at phase 0)
    irf = pptoaslib.instrumental_response_port_FT(nbin, freqs, DM=30.0, P=0.002, wids=[0.4 / nbin],
                                                  irf_types=["rect"]).real
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        pl.set_freqs(freqs)
        outs = [np.asarray(pl.apply_response_batch(x.astype(np.float32), r), dtype=np.float64) for r in (resp, irf)]
    for name, r, out in (("random", resp, outs[0]), ("irf", irf, outs[1])):
        ref = irfft_rows(X * r[None], nbin)
        tol = U32 * np.abs(ref) + (c_fft64(nbin) * np.abs(r).max(axis=1)[None, :, None]) * nx
        no_nyq = r.copy()
        no_nyq[:, L] = 1.0
        nyq_dc = r.copy()
        nyq_dc[:, 0] = r[:, L]
        wrong = {"nyquist_unscaled": irfft_rows(X * no_nyq[None], nbin)}
        if np.abs(r[:, 0] - r[:, L]).max() > 0:
            wrong["resp_N_at_DC"] = irfft_rows(X * nyq_dc[None], nbin)
        check(out, ref, tol, wrong, "response-%s-%s" % (name, PLAN_IDS[PLANS.index((nbin, force))]))


# ---------------------------------------------------------------------------------------------------------------
# scattering: pp_gen_gaussian_portrait with tau != 0 (k_gauss_model rows, then the scattering multiply)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_scattered_model_against_float64(nbin, force, monkeypatch):
    nchan, L = 11, nbin // 2
    gm = dict(orc.read_gmodel(synth.GMODEL))
    comps = np.array(gm["comps"], dtype=np.float64)
    # a component half a bin wide centred on a bin: a large Nyquist term, so that the factor there is seen (centred
    # between two bins, its two equal samples would cancel at the Nyquist frequency)
    loc = (np.floor(0.3 * nbin) + 0.5) / nbin
    comps = np.vstack([comps, [loc, 0.0, 0.5 / nbin, 0.0, 2.0, 0.0]])
    alpha, nu_ref, tau_bin = -3.7, gm["nu_ref"], 0.8
    params = np.concatenate([[gm["dc"], 0.0], comps.ravel()])
    freqs = orc.make_freqs(nchan, 1500., 800.)
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        pl.set_freqs(freqs)
        plain64 = pl.gen_gaussian_portrait("000", params, alpha, nu_ref, dtype=np.float64)
        params[1] = tau_bin
        out = np.asarray(pl.gen_gaussian_portrait("000", params, alpha, nu_ref), dtype=np.float64)
        out64 = pl.gen_gaussian_portrait("000", params, alpha, nu_ref, dtype=np.float64)
    assert np.array_equal(out, out64)              # the float64 generator returns the float32 scattered rows
    # the rows the scattering multiply reads: the float64 generator's values rounded to float32 (k_gauss_model)
    x = plain64.astype(np.float32).astype(np.float64)
    X = np.fft.rfft(x, axis=-1)
    taus = orc.scattering_times(tau_bin / nbin, alpha, freqs, nu_ref)
    B = orc.scattering_portrait_FT(taus, nbin)
    ref = irfft_rows(X * B, nbin)
    nx = np.linalg.norm(x, axis=-1)[:, None]
    tol = U32 * np.abs(ref) + (c_fft64(nbin) + 2 * np.pi * U * (L + 4)) * nx
    Bn = B.copy()
    Bn[:, L] = 1.0
    check(out, ref, tol, {"nyquist_unscattered": irfft_rows(X * Bn, nbin)},
          "scatter-%s" % PLAN_IDS[PLANS.index((nbin, force))])


# ---------------------------------------------------------------------------------------------------------------
# pp_align_accumulate
# ---------------------------------------------------------------------------------------------------------------
def _lr_sum(w):
    """left-to-right sum over subints of the weights the accumulation uses"""
    t = np.zeros(w.shape[1])
    for s in range(w.shape[0]):
        use = (w[s] != 0) & (np.abs(w[s]) < 1e300)
        t = np.where(use, t + w[s], t)
    return t


def _align_case(rng, nsub, nchan, nbin):
    # narrow pulses over little noise: the rounding of a rotated row to float32 is visible at the pulse peak
    x = _rows(rng, nsub, nchan, nbin, noise=0.05, amp=10.0, wid=0.6 / nbin, dc=0.4, alt=0.2)
    phase = rng.uniform(-0.5, 0.5, nsub)
    phase[0] = 0.4999
    DM = rng.normal(0.0, 2e-3, nsub)
    DM[nsub // 2] = 0.0
    P = rng.uniform(0.002, 0.006, nsub)
    nu_ref = rng.uniform(1200., 1800., nsub)
    w = rng.uniform(0.5, 2.0, (nsub, nchan))
    mid = w[1:-1]                                       # (subint 0 and the last one keep every channel)
    mid[rng.uniform(size=mid.shape) < 0.1] = 0.0
    mid[rng.uniform(size=mid.shape) < 0.1] *= -0.5      # negative fitted amplitudes weigh in with their sign
    if nchan > 4:
        w[:, 4] = 0.0                                   # a channel no subint contributes to
    if nsub > 2:
        w[1, 0] = -1.0
    return x, phase, DM, P, nu_ref, w


def _align_ref(x, freqs, phase, DM, P, nu_ref, w, nbin, absw=False, f32=False, dropk=None):
    nsub, nchan, _ = x.shape
    L = nbin // 2
    th, A = theta_rows(freqs, phase, DM, P, nu_ref)
    H = phasors(th, L)
    if dropk is not None:
        H[..., dropk] = 0.0
    y = irfft_rows(np.fft.rfft(x, axis=-1) * H, nbin)
    if f32:
        y = y.astype(np.float32).astype(np.float64)
    ww = np.abs(w) if absw else w
    use = (w != 0) & (np.abs(w) < 1e300)
    acc = np.einsum("sn,snj->nj", np.where(use, ww, 0.0), y)
    scale = np.einsum("sn,sn->n", np.where(use, np.abs(w), 0.0),
                      np.linalg.norm(x, axis=-1) * (c_fft64(nbin) + nsub * U + c_phase(A, L)))
    return acc, scale[:, None]


@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_align_accumulate_against_float64(nbin, force, monkeypatch):
    rng = np.random.RandomState(300 + nbin + 17 * force)
    label = PLAN_IDS[PLANS.index((nbin, force))]
    for nchan, calls in ((37, (70, 1)), (1, (3,))):     # 70 > the 64-subint block of the any-nbin path
        freqs = orc.make_freqs(nchan, 1500., 800.)
        with _plan(nchan, nbin, force, monkeypatch) as pl:
            pl.set_freqs(freqs)
            for nsub in calls:                          # one plan, several calls: no stale accumulator
                x, phase, DM, P, nu_ref, w = _align_case(rng, nsub, nchan, nbin)
                acc, wsum = pl.align_accumulate(x.astype(np.float32), phase, DM, P, nu_ref, w)
                assert np.array_equal(wsum, _lr_sum(w))
                ref, tol = _align_ref(x, freqs, phase, DM, P, nu_ref, w, nbin)
                wrong = {"rows_float32": _align_ref(x, freqs, phase, DM, P, nu_ref, w, nbin, f32=True)[0],
                         "nyquist": _align_ref(x, freqs, phase, DM, P, nu_ref, w, nbin, dropk=nbin // 2)[0],
                         "dc": _align_ref(x, freqs, phase, DM, P, nu_ref, w, nbin, dropk=0)[0]}
                if (w < 0).any():
                    wrong["abs_w"] = _align_ref(x, freqs, phase, DM, P, nu_ref, w, nbin, absw=True)[0]
                if nsub > 1:
                    wrong["subint0_P_nuref"] = _align_ref(x, freqs, phase, DM, np.full(nsub, P[0]),
                                                          np.full(nsub, nu_ref[0]), w, nbin)[0]
                used = tol[:, 0] > 0
                assert np.all(acc[~used] == 0.0)
                check(acc[used], ref[used], tol[used], {k: v[used] for k, v in wrong.items()},
                      "align_accumulate-%s-nchan%d-nsub%d" % (label, nchan, nsub))


# ---------------------------------------------------------------------------------------------------------------
# fused align_sum of pp_fit_batch
# ---------------------------------------------------------------------------------------------------------------
FUSED = [  # nchan, nsub, data type, float64 analytic model, chunk
    (37, 8, "float32", False, 3),
    (1, 5, "float64", True, 0),
    (300, 7, "int16", False, 3),
]


@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
@pytest.mark.parametrize("nchan,nsub,dtype,model64,chunk", FUSED,
                         ids=["nchan%d-%s%s" % (c[0], c[2], "-model64" if c[3] else "") for c in FUSED])
def test_fused_align_sum_against_float64(nbin, force, nchan, nsub, dtype, model64, chunk, monkeypatch):
    from pulseportraiture_b200 import pptoas
    L = nbin // 2
    nu0, bw = 800., 400.
    dDM = 0.0 if nchan == 1 else 2e-3
    cs = [synth.make_case(nchan, nbin, nu0, bw, 500 + 7 * nbin + s, dDM=dDM, sigma=0.5) for s in range(nsub)]
    freqs, P = cs[0]["freqs"], cs[0]["P"]
    data = np.stack([c["data"] for c in cs])
    nan_row = None
    if dtype == "float32":
        nan_row = (2, 5)
        data[2, 5, 10] = np.nan
        dev_data, x = data.astype(np.float32), data.copy()
        kw = {}
    elif dtype == "float64":
        dev_data, x = data, data.astype(np.float32).astype(np.float64)
        kw = {}
    else:
        raw, scl, offs, dec = pptoas.quantize_subints(data)
        dev_data, x = raw, dec.astype(np.float64)
        kw = dict(dat_scl=scl, dat_offs=offs)
    if model64:
        model = orc.gen_gaussian_portrait(dict(orc.read_gmodel(synth.GMODEL), alpha=-4.0), orc.get_bin_centers(nbin),
                                          freqs, P=P, tau_override=0.0)
    else:
        model = cs[0]["model"].astype(np.float32)
    Ps = P * (1.0 + 1e-3 * np.arange(nsub))
    flags = (1, 0, 0, 0, 0) if nchan == 1 else (1, 1, 0, 0, 0)
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        pl.set_model(model, freqs)
        if model64 and nbin >= 1024 and _pow2(nbin):
            assert pl.stats()["x_keep_frac"] < 1.0       # the cut-off drops harmonics of the model, not of the sum
        if chunk:
            pl.set_chunk(chunk)
        r = pl.fit_batch(dev_data, Ps, nu_fit_mode=0, DM_guess=dDM, fit_flags=flags, Ns=nbin, align=True, **kw)
    if nan_row is not None:
        assert r["noise"][nan_row] == 0.0 and np.all(r["noise"][~np.isnan(x).any(-1)] > 0)
    sig = r["noise"]
    ok = (sig > 0) & (r["return_code"] != 3)[:, None]
    w = np.where(ok, r["scales"] / np.where(sig > 0, sig, 1.0) ** 2, 0.0)
    assert np.abs(r["align_wsum"] - w.sum(0)).max() <= 1e-13 * np.abs(w).sum(0).max()
    xs = np.where(ok[..., None], x, 0.0)               # rows the sum leaves out (a NaN row among them)
    Xs = np.fft.rfft(xs, axis=-1)
    phi, DM, nu_out = r["params"][:, 0], r["params"][:, 1], r["nu_out"][:, 0]

    def ref_about(nu, dropk=None):
        th, A = theta_rows(freqs, phi, DM, Ps, nu)
        H = phasors(th, L)
        if dropk is not None:
            H[..., dropk] = 0.0
        return np.einsum("sn,snj->nj", w, irfft_rows(Xs * H, nbin)), A

    ref, A = ref_about(nu_out)
    aw = np.abs(w)
    eps = U32 * np.einsum("sn,snk->nk", aw, np.abs(Xs.real[..., 1:]) + np.abs(Xs.imag[..., 1:]))
    tol = (2.0 / nbin) * eps.sum(1) + np.einsum(
        "sn,sn->n", aw, np.linalg.norm(xs, axis=-1) * (c_fft64(nbin) + nsub * U + c_phase(A, L)))
    tol = tol[:, None]
    used = tol[:, 0] > 0
    wrong = {"nyquist": ref_about(nu_out, L)[0], "dc": ref_about(nu_out, 0)[0]}
    if nchan > 1:
        # nu_fit_mode 0: the fit's reference frequency is the mean of the used channels' frequencies
        nu_fit = np.array([freqs[ok[s]].mean() for s in range(nsub)])
        wrong["theta_about_nu_fit"] = ref_about(nu_fit)[0]
    label = "fused-%s-nchan%d-%s" % (PLAN_IDS[PLANS.index((nbin, force))], nchan, dtype)
    assert np.all(r["align_sum"][~used] == 0.0)
    check(r["align_sum"][used], ref[used], tol[used], {k: v[used] for k, v in wrong.items()}, label)
