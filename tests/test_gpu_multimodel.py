"""Several models in one batch (pp_set_models + pp_fit_batch_models): a subint fit against its own model portrait and
frequency table in one call gives exactly what separate pp_fit_batch calls on each model's subints give."""
import ctypes as C

import numpy as np
import pytest

from tests import synth

pytestmark = pytest.mark.gpu

NCHAN = 48
# (nu0, bw, tau_s at the .gmodel reference frequency, P): different tables, the same scattered .gmodel at two periods
TABLES = [(1500., 800., 0.0, synth.P_EXAMPLE), (1380., 400., 2e-4, 0.0031), (1380., 400., 2e-4, 0.0047)]


def _models(nbin, floor_model=2):
    """models [3, nchan, nbin] float64, freqs [3, nchan]; model `floor_model` is float32-rounded with a noise floor,
    so that it keeps every harmonic while the analytic ones are cut off."""
    fs, ms = [], []
    for i, (nu0, bw, tau, P) in enumerate(TABLES):
        f, m = synth.example_model(NCHAN, nbin, nu0, bw, tau_s=tau, P=P)
        if i == floor_model:
            m = m.astype(np.float32).astype(np.float64) + np.random.RandomState(7).normal(0, 3e-2, m.shape)
        fs.append(f)
        ms.append(m)
    return np.stack(ms), np.stack(fs)


def _batch(nbin, nsub=12, seed0=900, tau_data_s=0.0):
    """data [nsub, nchan, nbin] and per-subint periods, subint s made from table index[s] (interleaved runs)"""
    index = np.array([0, 0, 1, 2, 2, 0, 1, 1, 2, 0, 2, 1], dtype=np.int32)[:nsub]
    data, P = [], []
    for s in range(nsub):
        nu0, bw, _, Pm = TABLES[index[s]]
        Ps = Pm * (1.0 + 1e-7 * s)
        c = synth.make_case(NCHAN, nbin, nu0, bw, seed0 + s, P=Ps, tau_data_s=tau_data_s)
        data.append(c["data"])
        P.append(Ps)
    return np.stack(data).astype(np.float32), np.array(P), index


def _rows(v, sel):
    return None if v is None else v[sel]


PER_SUBINT = ("chan_mask", "errs", "scat_guess", "dat_scl", "dat_offs", "DM_guess")


def _split(pl, models, freqs, data, P, index, stats=None, **kw):
    """the reference: one pp_fit_batch per model on that model's subints, scattered back into batch order
    (stats: a dict that receives each call's pl.stats() by model)"""
    out = None
    for m in range(models.shape[0]):
        sel = np.nonzero(index == m)[0]
        if sel.size == 0:
            continue
        pl.set_model(models[m], freqs[m])
        kws = {k: (_rows(v, sel) if k in PER_SUBINT else v) for k, v in kw.items()}
        r = pl.fit_batch(data[sel], P[sel], **kws)
        if stats is not None:
            stats[m] = pl.stats()
        if out is None:
            out = {k: np.zeros((len(index),) + v.shape[1:], v.dtype) for k, v in r.items()}
        for k, v in r.items():
            out[k][sel] = v
    return out


def _assert_same(a, b, what=""):
    assert sorted(a) == sorted(b)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), "%s %s differs" % (what, k)


def _mask(nsub):
    mask = np.ones((nsub, NCHAN), dtype=np.uint8)
    mask[1, 5:20] = 0
    mask[4, ::3] = 0
    return mask


@pytest.mark.parametrize("nbin", [512, 2048, 1536])
@pytest.mark.parametrize("dtype", ["f32", "i16", "f64"])
def test_phi_dm_one_call_equals_split_calls(nbin, dtype):
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    models, freqs = _models(nbin)
    data, P, index = _batch(nbin)
    nsub = len(P)
    kw = {}
    if dtype == "i16":
        scl = np.full((nsub, NCHAN), 0.01, np.float32)
        offs = np.full((nsub, NCHAN), 0.5, np.float32)
        data = np.round((data - 0.5) / 0.01).astype(np.int16)
        kw = dict(dat_scl=scl, dat_offs=offs)
    elif dtype == "f64":
        data = data.astype(np.float64)
    with WidebandPlan(NCHAN, nbin) as pl:
        for mask in (None, _mask(nsub)):
            kw["chan_mask"] = mask
            ref = _split(pl, models, freqs, data, P, index, **kw)
            pl.set_models(models, freqs)
            _assert_same(pl.fit_batch(data, P, model_index=index, **kw), ref, "host")
            # device data, models, tables and index
            dkw = {k: (torch.from_numpy(np.ascontiguousarray(v)).cuda() if isinstance(v, np.ndarray) else v)
                   for k, v in kw.items()}
            pl.set_models(torch.from_numpy(models).cuda(), torch.from_numpy(freqs).cuda())
            got = pl.fit_batch(torch.from_numpy(data).cuda(), P, model_index=torch.from_numpy(index).cuda(), **dkw)
            _assert_same(got, ref, "device")
            # chunks whose boundaries cut through the model runs: the (phi, DM) fit is chunk-invariant
            pl.set_chunk(5)
            _assert_same(pl.fit_batch(data, P, model_index=index, **kw), ref, "chunked")
            pl.set_chunk(0)


@pytest.mark.parametrize("flags", [(1, 1, 0, 1, 1), (1, 1, 1, 1, 1)])
def test_general_solver_one_call_equals_split_calls(flags):
    from pulseportraiture_b200.engine import WidebandPlan
    nbin = 1024
    models, freqs = _models(nbin)
    data, P, index = _batch(nbin, tau_data_s=1e-4)
    nsub = len(P)
    scat = np.tile([1e-4, -4.0], (nsub, 1))
    kw = dict(fit_flags=flags, log10_tau=True, scat_guess=scat, chan_mask=_mask(nsub))
    with WidebandPlan(NCHAN, nbin) as pl:
        pl.enable_timing(True)
        alone = {}
        ref = _split(pl, models, freqs, data, P, index, stats=alone, **kw)
        # the case exercises the per-model levels: the noise-floor model has no coarse stage of its own (its
        # subints sit the batch's coarse levels out), the analytic ones have one
        assert alone[2]["coarse_launches"] == 0
        assert alone[0]["coarse_launches"] > 0 and alone[1]["coarse_launches"] > 0
        pl.set_models(models, freqs)
        got = pl.fit_batch(data, P, model_index=index, **kw)
        assert pl.stats()["coarse_launches"] > 0
        _assert_same(got, ref, "one chunk")
        # several chunks: the coarse levels come from each model's first subint of the chunk; same optimum
        pl.set_chunk(5)
        b = pl.fit_batch(data, P, model_index=index, **kw)
    a = ref
    fit = np.array(flags, bool)
    # (a few of these mismatched synthetic fits stop at the pass limit either way: the bars hold for the converged)
    ok = (a["return_code"] == 0) & (b["return_code"] == 0)
    assert ok.sum() >= nsub - 3
    assert np.max(np.abs(a["params"] - b["params"])[ok][:, fit] / a["param_errs"][ok][:, fit]) < 1e-3
    assert np.max(np.abs(b["param_errs"][ok][:, fit] / a["param_errs"][ok][:, fit] - 1)) < 1e-5
    assert np.max(np.abs(b["chi2"][ok] / a["chi2"][ok] - 1)) < 1e-9


def test_one_model_through_set_models_is_set_model():
    from pulseportraiture_b200.engine import WidebandPlan
    nbin = 512
    models, freqs = _models(nbin)
    data, P, _ = _batch(nbin)
    with WidebandPlan(NCHAN, nbin) as pl:
        pl.set_model(models[0], freqs[0])
        ref = pl.fit_batch(data, P)
        gen = pl.fit_batch(data, P, fit_flags=(1, 1, 0, 1, 1), log10_tau=True)
        pl.set_models(models[:1], freqs[:1])
        _assert_same(pl.fit_batch(data, P, model_index=np.zeros(len(P), np.int32)), ref)
        _assert_same(pl.fit_batch(data, P), ref)
        _assert_same(pl.fit_batch(data, P, fit_flags=(1, 1, 0, 1, 1), log10_tau=True,
                                  model_index=np.zeros(len(P), np.int32)), gen)
        # the kept share of the cross-spectrum over several models is that over all their channels
        keep = []
        for m in range(3):
            pl.set_model(models[m], freqs[m])
            keep.append(pl.stats()["x_keep_frac"])
        assert min(keep) < 1.0 and max(keep) == 1.0
        pl.set_models(models, freqs)
        assert np.isclose(pl.stats()["x_keep_frac"], np.mean(keep), rtol=1e-12, atol=0)


def test_errors_leave_the_plan_usable():
    import torch
    from pulseportraiture_b200 import _ffi
    from pulseportraiture_b200.engine import WidebandPlan
    nbin = 512
    models, freqs = _models(nbin)
    data, P, index = _batch(nbin)
    with WidebandPlan(NCHAN, nbin) as pl:
        pl.set_models(models, freqs)
        ref = pl.fit_batch(data, P, model_index=index)
        bad = index.copy()
        bad[3] = 3
        for idx in (bad, torch.from_numpy(bad).cuda(), -1 - index):
            with pytest.raises(_ffi.PPError, match="model_index"):
                pl.fit_batch(data, P, model_index=idx)
        with pytest.raises(_ffi.PPError, match="model_index is required"):
            pl.fit_batch(data, P)
        with pytest.raises(_ffi.PPError, match="align_sum"):
            pl.fit_batch(data, P, model_index=index, align=True)
        f = freqs.copy()
        f[2, 7] = 0.0
        with pytest.raises(_ffi.PPError, match="not positive"):
            pl.set_models(models, f)
        m = np.ascontiguousarray(models, np.float32)
        fr = np.ascontiguousarray(freqs)
        assert pl._lib.pp_set_models(pl._h, 0, C.c_void_p(m.ctypes.data), C.c_void_p(fr.ctypes.data)) < 0
        assert b"nmodel" in pl._lib.pp_last_error()
        _assert_same(pl.fit_batch(data, P, model_index=index), ref, "after errors")


def test_multigpu_fitter_with_model_index_matches_one_plan():
    import torch
    from pulseportraiture_b200.engine import WidebandPlan
    from pulseportraiture_b200.multigpu import MultiGPUFitter
    nbin = 512
    models, freqs = _models(nbin)
    data, P, index = _batch(nbin, nsub=11)
    nd = torch.cuda.device_count()
    kw = dict(chan_mask=_mask(len(P)), model_index=index)
    with WidebandPlan(NCHAN, nbin) as pl:
        pl.set_models(models, freqs)
        one = pl.fit_batch(data, P, **kw)
    mf = MultiGPUFitter(NCHAN, nbin, [i % nd for i in range(2)])
    try:
        mf.set_models(models, freqs)
        _assert_same(mf.fit_batch(data, P, **kw), one)
    finally:
        mf.close()


def _write_scattered_gmodel(path, tau_s):
    src = open(synth.GMODEL).read().splitlines()
    out = ["TAU     %.8f 0" % tau_s if ln.startswith("TAU") else ln for ln in src]
    with open(path, "w") as f:
        f.write("\n".join(out) + "\n")


def test_get_toas_fits_an_archive_of_per_subint_models_in_one_call_per_flags_group(tmp_path, monkeypatch):
    """GetTOAs on an archive whose model differs per subint (a .gmodel with TAU != 0 at per-subint periods) on two
    frequency tables: one set_models and one fit_batch per fit_flags group (the 1-channel subint is its own group),
    and every result list equals what explicit per-model set_model + fit_batch calls give."""
    from pulseportraiture_b200 import engine, pptoas
    from pulseportraiture_b200.pplib import DataBunch, get_bin_centers
    nsub, nchan, nbin = 10, 32, 256
    gmodel = str(tmp_path / "scattered.gmodel")
    _write_scattered_gmodel(gmodel, 3e-4)
    tabs = [(1400., 400.), (1450., 300.)]
    which = np.array([0, 0, 1, 0, 1, 1, 0, 1, 0, 0])
    Ps = synth.P_EXAMPLE * (1.0 + 1e-4 * np.arange(nsub))
    cases = [synth.make_case(nchan, nbin, tabs[w][0], tabs[w][1], 4200 + s, P=Ps[s]) for s, w in enumerate(which)]
    freqs = np.stack([c["freqs"] for c in cases])
    ok_ichans = [np.arange(nchan)] * nsub
    ok_ichans[4] = np.array([7])                 # one usable channel: phase-only fit, its own flags group
    d = DataBunch(backend="GUPPI", backend_delay=0.0, bw=400.0, doppler_factors=np.ones(nsub), DM=0.0, dmc=0,
                  epochs=[pptoas.MJD(56000, 0.01 * i) for i in range(nsub)], filename="mm.npz", freqs=freqs,
                  frontend="L", integration_length=float(nsub), masks=None, nbin=nbin, nchan=nchan, npol=1,
                  nsub=nsub, nu0=1400.0, ok_ichans=ok_ichans, ok_isubs=np.arange(nsub),
                  parallactic_angles=np.zeros(nsub), phases=get_bin_centers(nbin), Ps=Ps,
                  SNRs=np.ones((nsub, 1, nchan)), source="J0000+0000", state="Intensity", subtimes=np.ones(nsub),
                  telescope="GBT", telescope_code="1", weights=np.ones((nsub, nchan)),
                  noise_stds=np.full((nsub, 1, nchan), 1.5), flux_prof=None, prof=None, prof_noise=None,
                  prof_SNR=None, subints=np.stack([c["data"] for c in cases])[:, None], raw_subints=None,
                  dat_scl=None, dat_offs=None)
    calls = []
    fit_batch = engine.WidebandPlan.fit_batch

    def counted(self, *a, **kw):
        calls.append(kw.get("model_index") is not None)
        return fit_batch(self, *a, **kw)
    monkeypatch.setattr(engine.WidebandPlan, "fit_batch", counted)

    def run():
        gt = pptoas.GetTOAs([d], gmodel, quiet=True)
        gt.get_TOAs(quiet=True)
        return gt
    new = run()
    assert calls == [True, True]                 # one call per flags group (the 1-channel subint is its own group)
    # the per-model loop: a model budget of one model sets and fits one model at a time
    calls.clear()
    monkeypatch.setattr(pptoas, "_MODEL_BUDGET_BYTES", engine.model_bytes(nchan, nbin))
    old = run()
    assert len(calls) == nsub and not any(calls)   # every subint has its own period, hence its own model
    for name in ("phis", "phi_errs", "DMs", "DM_errs", "GMs", "taus", "alphas", "scales", "scale_errs", "snrs",
                 "channel_snrs", "covariances", "red_chi2s", "nfevals", "rcs", "nu_fits", "nu_refs"):
        a, b = getattr(new, name), getattr(old, name)
        assert len(a) == len(b) == 1
        assert np.array_equal(np.asarray(a[0], dtype=float), np.asarray(b[0], dtype=float), equal_nan=True), name
    for a, b in zip(new.TOAs[0], old.TOAs[0]):
        assert (a.intday(), a.fracday()) == (b.intday(), b.fracday())
    assert [(t.MJD.intday(), t.MJD.fracday(), t.TOA_error) for t in new.TOA_list] == \
        [(t.MJD.intday(), t.MJD.fracday(), t.TOA_error) for t in old.TOA_list]
