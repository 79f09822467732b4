"""Cost of fitting every subint against its own model (pp_set_models + pp_fit_batch_models) on the bench shape,
512 chan x 2048 bin (config 2), float64 models (harmonic cut-off on, as in bench.py).

  engine   10 000 subints, nmodel = 1, 4, 64, 512 models assigned round-robin: TOA/s and ms_per_step from the host
           clock around one fit_batch call (results copied into pageable numpy arrays), ms_spectra / ms_pass from
           the plan's CUDA events.
           The model rows stop being L2-resident as the models multiply; this curve is the cost of the feature.
  loop     256 subints with one model per subint (per-subint periods and a scattered template): one pp_set_models +
           one pp_fit_batch_models call against the per-model loop (set_model + a 1-subint fit_batch per subint),
           alternated.

  facade   `multimodel_probe.py facade OUT.json [--root TREE]`: GetTOAs(...).get_TOAs() on a 256-subint
           512 x 2048 float64 archive with per-subint periods and a .gmodel with TAU != 0 (one model per subint),
           with the package imported from TREE (default: this tree).  Run it on two trees (the previous facade,
           one set_model + fit_batch per model, and this one), alternating, to compare the two facades.

  rows1024 `multimodel_probe.py rows1024 OUT.json [--root TREE]`: a one-model fit of 10 000 device-resident subints
           at 512 x 1024 (the generic k_spectra<512> row kernel), ms per call, package from TREE.

Writes one JSON document (card name and power limit included) to the path given (default
profiles/multimodel_probe.json).  Needs a CUDA device."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    import torch
    import bench
    from pulseportraiture_b200.engine import WidebandPlan, model_bytes
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "multimodel_probe.json")
    dev = "cuda:0"
    freqs, model = bench.make_model()
    nchan, nbin = model.shape
    res = {"gpu": gpu_info(), "shape": [nchan, nbin], "model_bytes": model_bytes(nchan, nbin), "engine": [], "loop": {}}

    nsub, steps = 10000, 3
    phi, dDM = bench.global_draws(nsub)
    data = bench.make_device_batch(model, freqs, phi, dDM, 11, dev)
    P = np.full(nsub, bench.P_EXAMPLE)
    with WidebandPlan(nchan, nbin) as pl:
        pl.enable_timing(True)
        for nmodel in (1, 4, 64, 512):
            # the same template on tables shifted by up to 1 MHz: nmodel distinct sets of model rows
            fr = np.stack([freqs + 1.0 * m / max(1, nmodel - 1) for m in range(nmodel)])
            # float64, as bench.py sets its model: the harmonic cut-off applies
            models = torch.from_numpy(model).to(dev).expand(nmodel, nchan, nbin).contiguous()
            pl.set_models(models, torch.from_numpy(fr).to(dev))
            idx = torch.from_numpy((np.arange(nsub) % nmodel).astype(np.int32)).to(dev)
            pl.fit_batch(data, P, model_index=idx)   # warm-up
            torch.cuda.synchronize()
            ts, sp, pa = [], [], []
            for _ in range(steps):
                t = time.perf_counter()
                pl.fit_batch(data, P, model_index=idx)
                ts.append(time.perf_counter() - t)
                st = pl.stats()
                sp.append(st["ms_spectra"]); pa.append(st["ms_pass"])
            res["engine"].append({"nmodel": nmodel, "toa_per_s": nsub / float(np.median(ts)),
                                  "ms_per_step": 1e3 * float(np.median(ts)),
                                  "ms_spectra": float(np.median(sp)), "ms_pass": float(np.median(pa))})
            print(res["engine"][-1], flush=True)
            del models
    del data

    # one model per subint: per-subint periods of a scattered template (the template depends on P)
    n = 256
    phi, dDM = bench.global_draws(n, seed=5)
    data = bench.make_device_batch(model, freqs, phi, dDM, 12, dev).cpu().numpy().astype(np.float64)
    P = bench.P_EXAMPLE * (1.0 + 1e-6 * np.arange(n))
    mFT = np.fft.rfft(model, axis=-1)
    k = np.arange(mFT.shape[-1])
    models = np.empty((n, nchan, nbin))
    for s in range(n):
        taus = 2e-5 / P[s] * (freqs / bench.NU0) ** -4.0
        models[s] = np.fft.irfft(mFT / (1.0 + 2j * np.pi * taus[:, None] * k[None, :]), n=nbin, axis=-1)
    fr = np.broadcast_to(freqs, (n, nchan))
    idx = np.arange(n, dtype=np.int32)
    with WidebandPlan(nchan, nbin) as pl:
        def old():
            for s in range(n):
                pl.set_model(models[s], freqs)
                pl.fit_batch(data[s:s + 1], P[s:s + 1])

        def new():
            pl.set_models(models, fr)
            pl.fit_batch(data, P, model_index=idx)
        old(); new()
        t_old, t_new = [], []
        for _ in range(2):
            t = time.perf_counter(); old(); t_old.append(time.perf_counter() - t)
            t = time.perf_counter(); new(); t_new.append(time.perf_counter() - t)
    res["loop"] = {"nsub": n, "data": "float64 host", "per_model_loop_toa_per_s": [n / t for t in t_old],
                   "one_call_toa_per_s": [n / t for t in t_new]}
    print(res["loop"], flush=True)
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


def facade(out_path, root):
    """wall time of GetTOAs.get_TOAs (model builds, H2D, fits, TOAs) on an archive whose model differs per subint"""
    sys.path.insert(0, root)
    import tempfile
    from pulseportraiture_b200 import pptoas                 # from TREE (before bench puts this tree first)
    from pulseportraiture_b200.pplib import DataBunch, get_bin_centers
    import bench
    assert os.path.dirname(os.path.abspath(pptoas.__file__)).startswith(os.path.abspath(root))
    freqs, model = bench.make_model()
    nchan, nbin = model.shape
    n = 256
    phi, dDM = bench.global_draws(n, seed=5)
    sub = bench.make_device_batch(model, freqs, phi, dDM, 12, "cuda:0").cpu().numpy().astype(np.float64)
    Ps = bench.P_EXAMPLE * (1.0 + 1e-6 * np.arange(n))    # per-subint folding periods
    tmp = tempfile.mkdtemp()
    gmodel = os.path.join(tmp, "scattered.gmodel")
    with open(bench.GMODEL) as f, open(gmodel, "w") as g:    # TAU = 20 us at the .gmodel's FREQ, not fit
        g.write("".join("TAU     0.00002000 0\n" if ln.startswith("TAU") else ln for ln in f))
    d = DataBunch(backend="GUPPI", backend_delay=0.0, bw=bench.BW, doppler_factors=np.ones(n), DM=0.0, dmc=0,
                  epochs=[pptoas.MJD(56000 + i // 100, 0.01 * (i % 100)) for i in range(n)], filename="probe.npz",
                  freqs=np.tile(freqs, (n, 1)), frontend="Rcvr_800", integration_length=float(n), masks=None,
                  nbin=nbin, nchan=nchan, npol=1, nsub=n, nu0=bench.NU0, ok_ichans=[np.arange(nchan)] * n,
                  ok_isubs=np.arange(n), parallactic_angles=np.zeros(n), phases=get_bin_centers(nbin), Ps=Ps,
                  SNRs=np.ones((n, 1, nchan)), source="J0000+0000", state="Intensity", subtimes=np.ones(n),
                  telescope="GBT", telescope_code="1", weights=np.ones((n, nchan)),
                  noise_stds=np.full((n, 1, nchan), bench.SIGMA), flux_prof=None, prof=None, prof_noise=None,
                  prof_SNR=None, subints=sub[:, None], raw_subints=None, dat_scl=None, dat_offs=None)
    rates, fit_rates = [], []
    for rep in range(3):                                     # the first call warms up (module load, plan)
        gt = pptoas.GetTOAs([d], gmodel, quiet=True)
        t0 = time.perf_counter()
        gt.get_TOAs(quiet=True)
        dt = time.perf_counter() - t0
        if rep:
            rates.append(n / dt)
            fit_rates.append(n / gt.fit_durations[0])
    res = {"gpu": gpu_info(), "tree": os.path.abspath(root), "nsub": n, "shape": [nchan, nbin],
           "data": "float64 host, per-subint periods, TAU != 0 (one model per subint)",
           "get_TOAs_toa_per_s": rates, "fit_only_toa_per_s": fit_rates,
           "phis_checksum": float(np.sum(gt.phis[0])), "DMs_checksum": float(np.sum(gt.DMs[0]))}
    print(res, flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


def rows1024(out_path, root):
    """one-model fit_batch at nbin 1024 (generic k_spectra<512> rows), 512 chan, 10 000 device-resident subints:
    ms per call from the host clock around a synchronised call, with the package imported from TREE"""
    sys.path.insert(0, root)
    import torch
    from pulseportraiture_b200 import pplib
    from pulseportraiture_b200.engine import WidebandPlan
    import bench
    assert os.path.dirname(os.path.abspath(pplib.__file__)).startswith(os.path.abspath(root))
    nchan, nbin, nsub = 512, 1024, 10000
    freqs = np.linspace(bench.NU0 - bench.BW / 2 + bench.BW / (2.0 * nchan), bench.NU0 + bench.BW / 2 - bench.BW / (2.0 * nchan), nchan)
    _, _, model = pplib.read_model(bench.GMODEL, pplib.get_bin_centers(nbin), freqs, bench.P_EXAMPLE, quiet=True)
    phi, dDM = bench.global_draws(nsub)
    data = bench.make_device_batch(model, freqs, phi, dDM, 11, "cuda:0", nchan, nbin)
    P = np.full(nsub, bench.P_EXAMPLE)
    ms, out = [], None
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_model(model, freqs)
        for rep in range(6):
            torch.cuda.synchronize()
            t = time.perf_counter()
            out = pl.fit_batch(data, P, pinned_results=True)
            ms.append(1e3 * (time.perf_counter() - t))
        phis = np.array(out["params"][:, 0])
    res = {"gpu": gpu_info(), "tree": os.path.abspath(root), "shape": [nchan, nbin], "nsub": nsub,
           "ms_per_call": ms[1:], "phis_checksum": float(phis.sum())}
    print(res, flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] in ("facade", "rows1024"):
        root = sys.argv[sys.argv.index("--root") + 1] if "--root" in sys.argv else ROOT
        (facade if sys.argv[1] == "facade" else rows1024)(sys.argv[2], root)
    else:
        main()
