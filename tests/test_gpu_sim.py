"""Simulated archives on the device (pp_simulate_batch / WidebandPlan.simulate_batch / pplib.make_fake_pulsar).

Clean rows against a float64 restatement at every row plan, under the error model of test_gpu_rotate (output
rounding 2^-24 |y|; phase 2 pi u (L (2 A + 1/2) + 2) and the reference's own long-double phase error; double
transforms u (40 log2 nbin + 40); the scattering factor 2 pi u (L + 4); each scaled by S ||m||, the 2-norm of the
row's model spectrum times its scale).  Noise against the numpy restatement of Philox4x32-10 + Box-Muller in
tests/sim_ref.py: |(out - clean) - sigma z| <= 2^-24 (|out| + |clean|) + sigma 2^-20 r.  Wrong references (DC or
Nyquist term dropped, sign of theta flipped, GM about nu_DM, subint 0's tau and P for every subint, model 0 for
every subint; subint-local noise counter, channel and bin swapped, another seed) must miss by >= 10x the tolerance.
Then invariance bit for bit (batch splitting, chunking, host vs device output, a fit before and after), int16 output
against pptoas.quantize_subints, recovery of injected parameters by the fit (pulls), and the refusals.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import pp_oracle as orc
from tests import sim_ref, synth
from tests.test_gpu_rotate import PLANS, PLAN_IDS, U, U32, _plan, c_fft64, c_phase, check, phasors, theta_rows

pytestmark = pytest.mark.gpu


def _models(rng, nmodel, nchan, nbin):
    """float64 portraits with a pulse, a DC offset and a Nyquist-frequency component"""
    j = np.arange(nbin)
    out = np.empty((nmodel, nchan, nbin))
    for m in range(nmodel):
        loc = rng.uniform(0, 1, (nchan, 1))
        d = (j / nbin - loc + 0.5) % 1.0 - 0.5
        out[m] = (3.0 + m) * np.exp(-0.5 * (d / 0.03) ** 2) + 0.7 - 0.3 * m + 0.4 * (-1.0) ** j
    return out


def _case(nbin, seed, nsub=5, nchan=7):
    rng = np.random.RandomState(seed)
    f0 = orc.make_freqs(nchan, 1500., 800.)
    freqs = np.stack([f0, f0 * 0.9 + 30.0])
    c = dict(models=_models(rng, 2, nchan, nbin), freqs=freqs, model_index=np.array([0, 1, 1, 0, 1][:nsub], np.int32),
             phase=rng.uniform(-0.5, 0.5, nsub), DM=rng.normal(0, 2e-3, nsub), P=rng.uniform(0.002, 0.006, nsub),
             nu_DM=rng.uniform(1200., 1800., nsub), GM=rng.normal(0, 1.0, nsub), nu_GM=rng.uniform(900., 1800., nsub),
             tau=rng.uniform(0.2, 2.0, nsub) / nbin, alpha=rng.uniform(-4.4, -3.6, nsub),
             nu_tau=rng.uniform(1100., 1900., nsub), scales=rng.uniform(0.5, 2.0, (nsub, nchan)))
    c["DM"][1] = 0.0
    c["GM"][2] = 0.0
    return c


def _clean_ref(c, nbin, dc=True, nyq=True, sign=1, gm_about_dm=False, sub0=False, model0=False):
    """irfft of S M e^{-2 pi i k theta} B in float64 (theta in long double); also the tolerance scale"""
    L = nbin // 2
    nsub = len(c["phase"])
    nchan = c["models"].shape[1]
    M = np.fft.rfft(c["models"], axis=-1)
    out = np.empty((nsub, nchan, nbin))
    scale = np.empty((nsub, nchan))
    k = np.arange(L + 1)
    for s in range(nsub):
        m = 0 if model0 else c["model_index"][s]
        f = c["freqs"][m]
        s0 = 0 if sub0 else s
        th, A = theta_rows(f, c["phase"][s:s + 1], c["DM"][s:s + 1], c["P"][s0:s0 + 1], c["nu_DM"][s:s + 1],
                           c["GM"][s:s + 1], (c["nu_DM"] if gm_about_dm else c["nu_GM"])[s:s + 1])
        H = phasors(th[0], L)
        H = np.conj(H) if sign > 0 else H
        taus = c["tau"][s0] * (f / c["nu_tau"][s]) ** c["alpha"][s]
        B = 1.0 / (1.0 + 2j * np.pi * np.outer(taus, k))
        Y = c["scales"][s][:, None] * M[m] * H * B
        if not dc:
            Y[:, 0] = 0.0
        if not nyq:
            Y[:, L] = 0.0
        out[s] = np.fft.irfft(Y, n=nbin, axis=-1)
        nm = np.linalg.norm(c["models"][m], axis=-1)
        scale[s] = c["scales"][s] * nm * (c_fft64(nbin) + c_phase(A[0], L) + 2 * np.pi * U * (L + 4))
    return out, scale


def _sim(pl, c, **kw):
    args = dict(model_index=c["model_index"], GM=c["GM"], nu_GM=c["nu_GM"], tau=c["tau"], alpha=c["alpha"],
                nu_tau=c["nu_tau"], scales=c["scales"])
    args.update(kw)
    return pl.simulate_batch(c["models"], c["freqs"], c["phase"], c["DM"], c["P"], c["nu_DM"], **args)


@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_clean_rows_against_float64(nbin, force, monkeypatch):
    c = _case(nbin, 11 + nbin + force)
    nchan = c["models"].shape[1]
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        out = np.asarray(_sim(pl, c), dtype=np.float64)
    ref, sc = _clean_ref(c, nbin)
    tol = U32 * np.abs(ref) + sc[..., None]
    wrong = {"dc": _clean_ref(c, nbin, dc=False)[0], "nyquist": _clean_ref(c, nbin, nyq=False)[0],
             "theta_sign": _clean_ref(c, nbin, sign=-1)[0], "GM_about_nuDM": _clean_ref(c, nbin, gm_about_dm=True)[0],
             "subint0_tau_P": _clean_ref(c, nbin, sub0=True)[0], "model0": _clean_ref(c, nbin, model0=True)[0]}
    check(out, ref, tol, wrong, "simulate-%s" % PLAN_IDS[PLANS.index((nbin, force))])


def _philox_swapped(seed, s_global, nchan, nbin):
    """the noise with channel and bin quad exchanged in the counter"""
    s = np.asarray(s_global, dtype=np.uint64)[:, None, None]
    n = np.arange(nchan, dtype=np.uint64)[None, :, None]
    q = np.arange((nbin + 3) // 4, dtype=np.uint64)[None, None, :]
    x = sim_ref.philox4x32_10((n + 0 * q + 0 * s, q + 0 * n + 0 * s, s & np.uint64(0xFFFFFFFF), s >> np.uint64(32)),
                              (seed & 0xFFFFFFFF, seed >> 32))
    z0, z1, _ = sim_ref.box_muller(x[0], x[1])
    z2, z3, _ = sim_ref.box_muller(x[2], x[3])
    return np.stack([z0, z1, z2, z3], axis=-1).reshape(z0.shape[:2] + (-1,))[..., :nbin]


@pytest.mark.parametrize("nbin,force", PLANS, ids=PLAN_IDS)
def test_noise_int16_and_outputs(nbin, force, monkeypatch):
    """noise against the restatement; int16 = quantize_subints(float) bit for bit; host = device output; chunking"""
    import torch
    from pulseportraiture_b200 import pptoas
    c = _case(nbin, 500 + nbin + force)
    nsub, nchan = c["scales"].shape
    rng = np.random.RandomState(nbin)
    sigma = rng.uniform(0.1, 2.0, (nsub, nchan))
    sigma[2, 3] = 0.0
    seed, first = 0x1234567890ABCDEF, 2 ** 32 - 3          # the subints cross the low word of the counter
    with _plan(nchan, nbin, force, monkeypatch) as pl:
        clean = np.asarray(_sim(pl, c), dtype=np.float64)
        kw = dict(noise_stds=sigma, seed=seed, first_subint=first)
        out = _sim(pl, c, **kw)
        raw, scl, offs = _sim(pl, c, quantize=True, **kw)
        dev = _sim(pl, c, device_out=True, **kw)
        draw, dscl, doffs = _sim(pl, c, quantize=True, device_out=True, **kw)
        pl.set_chunk(2)
        out_c2 = _sim(pl, c, **kw)
        raw_c2 = _sim(pl, c, quantize=True, **kw)[0]
    assert np.array_equal(out, dev.cpu().numpy()) and np.array_equal(out, out_c2)
    assert np.array_equal(raw, draw.cpu().numpy()) and np.array_equal(scl, dscl.cpu().numpy())
    assert np.array_equal(offs, doffs.cpu().numpy()) and np.array_equal(raw, raw_c2)
    qr, qs, qo, _ = pptoas.quantize_subints(out)
    assert np.array_equal(raw, qr) and np.array_equal(scl, qs) and np.array_equal(offs, qo)
    assert torch.is_tensor(dev) and dev.is_cuda and draw.dtype == torch.int16
    z, r = sim_ref.noise(seed, first + np.arange(nsub), nchan, nbin)
    out = out.astype(np.float64)
    diff = out - clean
    tol = U32 * (np.abs(out) + np.abs(clean)) + sigma[..., None] * sim_ref.Z_REL * r
    assert np.all(diff[2, 3] == 0.0)                         # sigma = 0: the clean row
    wrong = {"local_counter": sigma[..., None] * sim_ref.noise(seed, np.arange(nsub), nchan, nbin)[0],
             "chan_bin_swapped": sigma[..., None] * _philox_swapped(seed, first + np.arange(nsub), nchan, nbin),
             "other_seed": sigma[..., None] * sim_ref.noise(seed + 1, first + np.arange(nsub), nchan, nbin)[0]}
    keep = sigma > 0
    # (bins below 4 nchan left out of the first check: there the swapped counter meets the right one at q = n)
    check(diff[keep][:, 4 * nchan:], (sigma[..., None] * z)[keep][:, 4 * nchan:], tol[keep][:, 4 * nchan:],
          {k: v[keep][:, 4 * nchan:] for k, v in wrong.items()}, "noise-%s" % PLAN_IDS[PLANS.index((nbin, force))])
    check(diff[keep], (sigma[..., None] * z)[keep], tol[keep], {}, "noise-all-%s" % PLAN_IDS[PLANS.index((nbin, force))])


@pytest.mark.parametrize("nbin", [2048, 1000])
def test_batch_split_and_device_invariance(nbin):
    """one call of 12 subints = three calls of 4 with first_subint 0 / 4 / 8 = other chunkings, bit for bit"""
    from pulseportraiture_b200.engine import WidebandPlan
    rng = np.random.RandomState(3)
    nchan, nsub = 9, 12
    models = _models(rng, 1, nchan, nbin)[0]
    freqs = orc.make_freqs(nchan, 1400., 400.)
    phase, DM, P = rng.uniform(-.5, .5, nsub), rng.normal(0, 1e-3, nsub), rng.uniform(0.002, 0.004, nsub)
    sig = rng.uniform(0.5, 1.5, (nsub, nchan))
    with WidebandPlan(nchan, nbin) as pl:
        whole = pl.simulate_batch(models, freqs, phase, DM, P, noise_stds=sig, seed=99)
        parts = np.concatenate([pl.simulate_batch(models, freqs, phase[i:i + 4], DM[i:i + 4], P[i:i + 4],
                                                  noise_stds=sig[i:i + 4], seed=99, first_subint=i)
                                for i in (0, 4, 8)])
        chunked = []
        for ch in (1, 5, 7):
            pl.set_chunk(ch)
            chunked.append(pl.simulate_batch(models, freqs, phase, DM, P, noise_stds=sig, seed=99))
    assert np.array_equal(whole, parts)
    for o in chunked:
        assert np.array_equal(whole, o)


def test_mixed_output_kinds_list_inputs_and_chunked_host_inputs():
    """outputs of different memory kinds in one call (device raw, host DAT_SCL / DAT_OFFS), plain lists as inputs, and
    host per-subint inputs staged chunk by chunk: the same bytes as one all-device call"""
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    rng = np.random.RandomState(5)
    nchan, nbin, nsub = 6, 256, 7
    m = _models(rng, 2, nchan, nbin)
    f = np.stack([orc.make_freqs(nchan, 1400., 400.)] * 2)
    phase, DM, P = list(rng.uniform(-.5, .5, nsub)), list(rng.normal(0, 1e-3, nsub)), list(rng.uniform(0.002, 0.004, nsub))
    idx = [0, 1, 1, 0, 0, 1, 0]
    sig, sc = rng.uniform(0.5, 1.5, (nsub, nchan)), rng.uniform(0.5, 2.0, (nsub, nchan))
    cu = lambda v: torch.tensor(np.asarray(v), device="cuda")       # noqa: E731
    with WidebandPlan(nchan, nbin) as pl:
        ref = pl.simulate_batch(cu(m), cu(f), cu(phase), cu(DM), cu(P), model_index=cu(np.array(idx, np.int32)),
                                scales=cu(sc), noise_stds=cu(sig), seed=4, quantize=True, device_out=True)
        ref = [r.cpu().numpy() for r in ref]
        out = (torch.zeros((nsub, nchan, nbin), dtype=torch.int16, device="cuda"),
               np.zeros((nsub, nchan), np.float32), np.zeros((nsub, nchan), np.float32))
        pl.set_chunk(3)
        got = pl.simulate_batch(m, f, phase, DM, P, model_index=idx, scales=sc, noise_stds=sig, seed=4, quantize=True,
                                out=out)
        f32 = pl.simulate_batch(m, f, phase, DM, P, model_index=idx, scales=sc, noise_stds=sig, seed=4)
    assert np.array_equal(got[0].cpu().numpy(), ref[0])
    assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
    assert f32.shape == (nsub, nchan, nbin)


def test_fit_results_unchanged_by_simulate():
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nbin = 32, 512
    freqs, model = synth.example_model(nchan, nbin, 1500., 800.)
    cs = [synth.make_case(nchan, nbin, 1500., 800., 40 + s) for s in range(6)]
    data = np.stack([c["data"] for c in cs]).astype(np.float32)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        before = pl.fit_batch(data, synth.P_EXAMPLE, fit_flags=(1, 1, 0, 0, 0))
        pl.simulate_batch(np.stack([model, 2 * model]), np.stack([freqs + 10, freqs - 10]), 0.1, 1e-3, 0.003,
                          noise_stds=1.0, model_index=np.array([1, 0, 1], np.int32), quantize=True)
        after = pl.fit_batch(data, synth.P_EXAMPLE, fit_flags=(1, 1, 0, 0, 0))
    for k in before:
        assert before[k].tobytes() == after[k].tobytes(), k


def test_noise_statistics():
    """>= 10^7 noise-only samples: mean, variance, adjacent-bin, channel and subint correlations within 5 standard
    errors; get_noise_batch of the rows agrees with sigma"""
    from pulseportraiture_b200.engine import WidebandPlan
    nsub, nchan, nbin = 80, 64, 2048
    with WidebandPlan(nchan, nbin) as pl:
        x = pl.simulate_batch(np.zeros((nchan, nbin)), orc.make_freqs(nchan, 1500., 800.), np.zeros(nsub), 0.0, 0.003,
                              noise_stds=2.0, seed=2024, device_out=True)
        noise = pl.get_noise_batch(x)
    z = x.double().cpu().numpy() / 2.0
    n = z.size
    assert n >= 10 ** 7
    se = 1.0 / np.sqrt(n)
    assert abs(z.mean()) < 5 * se
    assert abs(z.var() - 1.0) < 5 * np.sqrt(2.0) * se
    for name, a, b in (("bin", z[..., 1:], z[..., :-1]), ("chan", z[:, 1:], z[:, :-1]), ("subint", z[1:], z[:-1])):
        r = float(np.mean(a * b))
        assert abs(r) < 5.0 / np.sqrt(a.size), (name, r)
    # get_noise_PS: the rms of the top quarter of each row's harmonics, sigma for white noise; ~1/sqrt(2 nharm/4)
    # relative scatter per row
    rel = noise / 2.0 - 1.0
    assert abs(rel.mean()) < 5 * np.sqrt(2.0 / nbin) * 2 / np.sqrt(rel.size)
    assert np.abs(rel).max() < 6 * np.sqrt(4.0 / nbin)


def _pulls(got, want, err):
    p = (got - want) / err
    return p, abs(p.mean()) < 4 / np.sqrt(len(p))


@pytest.mark.parametrize("quantize", [False, True], ids=["float32", "int16"])
def test_phi_dm_recovery(quantize):
    from pulseportraiture_b200.engine import WidebandPlan
    nsub, nchan, nbin, nu0 = 256, 64, 512, 1500.
    freqs, model = synth.example_model(nchan, nbin, nu0, 800.)
    rng = np.random.RandomState(17)
    phase, DM = rng.uniform(-0.4, 0.4, nsub), rng.normal(0, 5e-4, nsub)
    P = synth.P_EXAMPLE
    nu = np.full((nsub, 3), nu0)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        d = pl.simulate_batch(model, freqs, phase, DM, P, nu0, noise_stds=1.0, seed=5, quantize=quantize,
                              device_out=True)
        if quantize:
            r = pl.fit_batch(d[0], P, dat_scl=d[1], dat_offs=d[2], nu_fits=nu, nu_outs=nu)
        else:
            r = pl.fit_batch(d, P, nu_fits=nu, nu_outs=nu)
    assert np.all(r["return_code"] == 0)
    dphi = (r["params"][:, 0] - phase + 0.5) % 1.0 - 0.5
    for name, p in (("phi", dphi / r["param_errs"][:, 0]), ("DM", (r["params"][:, 1] - DM) / r["param_errs"][:, 1])):
        print("PULL %s %s mean %.3f std %.3f" % (name, quantize, p.mean(), p.std()))
        assert abs(p.mean()) < 4 / np.sqrt(nsub), name
        assert 0.85 <= p.std() <= 1.15, name


def test_scattering_recovery():
    """fit_flags (1, 1, 0, 1, 1) with log10 tau: tau and alpha pulls; the std bounds are loosened to [0.75, 1.3]
    (64 subints: the sample std of unit pulls has a standard error of 0.09)"""
    from pulseportraiture_b200.engine import WidebandPlan
    nsub, nchan, nbin, nu0 = 64, 64, 512, 1500.
    freqs, model = synth.example_model(nchan, nbin, nu0, 800.)
    rng = np.random.RandomState(23)
    phase, DM = rng.uniform(-0.3, 0.3, nsub), rng.normal(0, 3e-4, nsub)
    tau, alpha = np.full(nsub, 4.0 / nbin), np.full(nsub, -4.0)
    P = synth.P_EXAMPLE
    nu = np.full((nsub, 3), nu0)
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        d = pl.simulate_batch(model, freqs, phase, DM, P, nu0, tau=tau, alpha=alpha, nu_tau=nu0, noise_stds=0.3,
                              seed=8, device_out=True)
        r = pl.fit_batch(d, P, nu_fits=nu, nu_outs=nu, fit_flags=(1, 1, 0, 1, 1), log10_tau=True,
                         scat_guess=np.column_stack([1.3 * tau, np.full(nsub, -4.3)]))
    ok = r["return_code"] == 0
    assert ok.mean() > 0.95
    for name, p in (("log10tau", (r["params"][ok, 3] - np.log10(tau[ok])) / r["param_errs"][ok, 3]),
                    ("alpha", (r["params"][ok, 4] - alpha[ok]) / r["param_errs"][ok, 4]),
                    ("DM", (r["params"][ok, 1] - DM[ok]) / r["param_errs"][ok, 1])):
        print("PULL %s mean %.3f std %.3f" % (name, p.mean(), p.std()))
        assert abs(p.mean()) < 4 / np.sqrt(ok.sum()), name
        assert 0.75 <= p.std() <= 1.3, name


# TOAs of a dedispersed archive (restored) against those of the dispersed one, in sigma: the largest differences
# measured over the 64 subints of test_make_fake_pulsar_gettoas on a B200 were 0.074 (phase, at a common reference
# frequency) and 0.039 (DM); they come from the Nyquist harmonic alone, and the bound leaves a factor 2
DEDISP_SIGMA = 0.15


def test_make_fake_pulsar_gettoas(tmp_path):
    """make_fake_pulsar -> .npz -> GetTOAs.get_TOAs: phase and DM pulls; dedispersed=True restores to the same archive
    but for the Nyquist harmonic; quantize=True gives the TOAs of the decoded floats exactly"""
    from pulseportraiture_b200 import pplib, pptoas
    nsub, nchan, nbin, nu0 = 64, 64, 512, 1500.
    rng = np.random.RandomState(31)
    par = tmp_path / "fake.par"
    par.write_text("PSRJ J1234-5678\nF0 %.17g\nF1 -2e-13\nPEPOCH 55990\nDM 12.5\n" % (1.0 / synth.P_EXAMPLE))
    phase, dDM = rng.uniform(-0.4, 0.4, nsub), rng.normal(0, 5e-4, nsub)
    kw = dict(nsub=nsub, nchan=nchan, nbin=nbin, nu0=nu0, bw=800., tsub=60., phase=phase, dDM=dDM,
              noise_stds=1.0, seed=77, quiet=True)
    path = str(tmp_path / "fake.npz")
    d = pplib.make_fake_pulsar(synth.GMODEL, str(par), outfile=path, **kw)
    assert d.subints.shape == (nsub, 1, nchan, nbin) and d.subints.dtype == np.float64
    for k in pptoas._DB_FIELDS:
        assert k in d
    assert np.all(d.Ps > 0) and np.ptp(d.Ps) > 0 and d.dmc == 0 and d.DM == 12.5
    assert np.allclose(d.noise_stds[:, 0], 1.0, rtol=0.4)
    gt = pptoas.GetTOAs(path, synth.GMODEL, quiet=True)
    gt.get_TOAs(quiet=True)
    phis, errs, nu_ref = np.asarray(gt.phis[0]), np.asarray(gt.phi_errs[0]), np.array([v[0] for v in gt.nu_refs[0]])
    want = pplib.phase_transform(phase, 12.5 + dDM, np.inf, nu_ref, d.Ps, mod=False)
    p_phi = ((phis - want + 0.5) % 1.0 - 0.5) / errs
    p_dm = (np.asarray(gt.DMs[0]) - (12.5 + dDM)) / np.asarray(gt.DM_errs[0])
    for name, p in (("phi", p_phi), ("DM", p_dm)):
        print("PULL facade %s mean %.3f std %.3f" % (name, p.mean(), p.std()))
        assert abs(p.mean()) < 4 / np.sqrt(nsub), name
        assert 0.75 <= p.std() <= 1.3, name
    # dedispersed storage: restore_dispersion gives back the dispersed archive in every harmonic but the Nyquist one
    # (a rotation keeps only the real part of that term, so dedispersing and restoring does not return its noise),
    # and TOAs that agree at a common reference frequency within what that one harmonic's noise moves them
    dd = pplib.make_fake_pulsar(synth.GMODEL, str(par), dedispersed=True, **kw)
    assert dd.dmc == 1
    back = pptoas.restore_dispersion(dd)
    X = np.fft.rfft(np.asarray(d.subints)[:, 0], axis=-1)
    Y = np.fft.rfft(np.asarray(back.subints)[:, 0], axis=-1)
    assert np.abs(X - Y)[..., :nbin // 2].max() < 1e-4 * np.abs(X).max()
    g2 = pptoas.GetTOAs([dd], synth.GMODEL, quiet=True)
    g2.get_TOAs(quiet=True)
    nu2 = np.array([v[0] for v in g2.nu_refs[0]])
    phi2 = pplib.phase_transform(np.asarray(g2.phis[0]), np.asarray(g2.DMs[0]), nu2, nu_ref, d.Ps)
    dphi = np.max(np.abs(((phi2 - phis + 0.5) % 1.0 - 0.5) / errs))
    ddm = np.max(np.abs((np.asarray(g2.DMs[0]) - np.asarray(gt.DMs[0])) / np.asarray(gt.DM_errs[0])))
    print("DEDISPERSED max |dphi|/sigma %.4g max |dDM|/sigma %.4g" % (dphi, ddm))
    assert dphi < DEDISP_SIGMA and ddm < DEDISP_SIGMA
    # int16 storage: the TOAs of the decoded floats
    qpath = str(tmp_path / "q.npz")
    dq = pplib.make_fake_pulsar(synth.GMODEL, str(par), outfile=qpath, quantize=True, **kw)
    assert dq.raw_subints.dtype == np.int16
    dfloat = pptoas.DataBunch(**dict(dq))
    for k in pptoas._RAW_FIELDS:
        dfloat[k] = None
    g3 = pptoas.GetTOAs([dfloat], synth.GMODEL, quiet=True)
    g3.get_TOAs(quiet=True)
    g4 = pptoas.GetTOAs(qpath, synth.GMODEL, quiet=True)
    g4.get_TOAs(quiet=True)
    assert np.array_equal(g3.phis[0], g4.phis[0]) and np.array_equal(g3.DMs[0], g4.DMs[0])


def test_refusals_launch_nothing():
    import torch
    from pulseportraiture_b200 import _ffi
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nbin = 4, 64
    m = _models(np.random.RandomState(0), 2, nchan, nbin)
    f = np.tile(orc.make_freqs(nchan, 1500., 800.), (2, 1))
    base = dict(model_index=np.array([0, 1], np.int32), noise_stds=1.0)
    bad = {
        "model_index": dict(model_index=np.array([0, 2], np.int32)),
        "P": dict(P=np.array([0.003, 0.0])),
        "freqs": dict(freqs=np.where(np.arange(nchan) == 1, -1.0, f)),
        "nu_DM": dict(nu_DM=np.array([1400., -5.])),
        "nu_tau": dict(tau=0.01, alpha=-4.0, nu_tau=0.0),
        "noise_std": dict(noise_stds=np.array([[1.0, 1.0, -0.5, 1.0]] * 2)),
        "noise_std_device": dict(noise_stds=torch.tensor([[1.0] * 4, [1.0, 1.0, 1.0, -0.5]], dtype=torch.float64,
                                                         device="cuda")),
        "P_device": dict(P=torch.tensor([0.003, -1.0], dtype=torch.float64, device="cuda")),
    }
    with WidebandPlan(nchan, nbin) as pl:
        pl.simulate_batch(m, f, 0.1, 0.0, 0.003, **base)
        st0 = pl.stats()
        assert st0["launches"] > 0
        for what, kw in bad.items():
            args = dict(base, freqs=f, P=0.003, nu_DM=np.inf)
            args.update(kw)
            out = np.full((2, nchan, nbin), 7.0, np.float32)
            with pytest.raises(_ffi.PPError) as e:
                pl.simulate_batch(m, args.pop("freqs"), 0.1, 0.0, args.pop("P"), args.pop("nu_DM"), out=out, **args)
            print("REFUSED %s: %s" % (what, e.value))
            assert np.all(out == 7.0) and pl.stats() == st0, what
        with pytest.raises(_ffi.PPError, match="nmodel"):
            pl.simulate_batch(m[:0], f[:0], 0.1, 0.0, 0.003, out=np.zeros((1, nchan, nbin), np.float32))
        # no output at all, and nsub = 0 (a no-op), through the C ABI
        L = _ffi.lib()
        keep = [np.ascontiguousarray(v) for v in (m, f, [0.1, 0.2], [0.0, 0.0], [0.003, 0.003], [np.inf, np.inf])]
        a = _ffi.SimArgs()
        a.models, a.freqs, a.phase, a.DM, a.P, a.nu_DM = [k.ctypes.data for k in keep]
        a.nmodel, a.nsub = 2, 2
        o = _ffi.SimOut()
        assert L.pp_simulate_batch(pl._h, C.byref(a), C.byref(o)) < 0 and b"output" in L.pp_last_error()
        a.nsub = 0
        assert L.pp_simulate_batch(pl._h, C.byref(a), C.byref(o)) == 0
        assert pl.stats() == st0
