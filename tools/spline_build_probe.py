"""Time pplib.make_spline_model and its steps on the device, and the same steps in numpy float64 on the host cores,
in one run; write profiles/spline_build_b200.json (or --out).

Shapes: 512 x 2048 (the Gram side: nchan < nbin) and 4096 x 1024 (the covariance side).  Device steps are timed with
CUDA events on the plan's stream around each engine call, inputs already on the device (the time includes the copy of
the result to the host); the host eigen decomposition and splprep by the host clock.  The card's name and power limit
are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def portrait(nchan, nbin, seed=1):
    rng = np.random.RandomState(seed)
    x = (np.arange(nbin) + 0.5) / nbin
    f = np.linspace(-1, 1, nchan)
    g = lambda c, s: np.exp(-0.5 * ((x - c) / s) ** 2)      # noqa: E731
    port = g(0.4, 0.03)[None] + 0.3 * np.sin(2 * f)[:, None] * (g(0.42, 0.03) * np.cos(6 * np.pi * (x - 0.42)))[None] \
        + 0.2 * np.cos(3 * f)[:, None] * (g(0.38, 0.04) * np.sin(4 * np.pi * (x - 0.38)))[None]
    return port + 0.01 * rng.standard_normal(port.shape)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # noqa: BLE001
        q = "not read (%s)" % e
    return name, q


def timed(stream, fn, reps):
    import torch
    fn()                                    # warm-up: module load, plan buffers
    best = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        r = fn()
        b.record(stream)
        b.synchronize()
        best.append(a.elapsed_time(b))
    return float(np.median(best)), r


def host(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), r


def probe(nchan, nbin, m, reps):
    import torch
    import scipy.interpolate as si
    import scipy.linalg as sl
    from pulseportraiture_b200 import pplib
    from pulseportraiture_b200.engine import WidebandPlan
    from tests.test_cpu_spline_build import lowpass
    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(dev)
    X = portrait(nchan, nbin)
    w = np.ones(nchan)
    Xd, wd = torch.as_tensor(X, device=dev), torch.as_tensor(w, device=dev)
    gram = nchan <= nbin
    pl = WidebandPlan(nchan, nbin, stream=st.cuda_stream)
    plr = WidebandPlan(m + 1, nbin, stream=st.cuda_stream)
    out = dict(nchan=nchan, nbin=nbin, side="gram" if gram else "covariance", m=m)
    dv = {}
    dv["moments_ms"], (mu, M) = timed(st, lambda: pl.pca_moments(Xd, wd, gram=gram), reps)
    dim = M.shape[0]
    eigh = lambda: sl.eigh(M, subset_by_index=[dim - m, dim - 1])     # noqa: E731
    t_eigh, (vals, Uv) = host(eigh, reps)
    Uv = np.ascontiguousarray(Uv[:, ::-1])
    mud = torch.as_tensor(mu, device=dev)
    if gram:
        Ud = torch.as_tensor(Uv, device=dev)
        dv["backproject_ms"], E = timed(st, lambda: pl.pca_backproject(Xd, wd, mud, Ud), reps)
    else:
        E = Uv
    rows = torch.as_tensor(np.ascontiguousarray(np.vstack([mu[None], E.T])), device=dev)
    dv["lowpass_ms"], (sm, kc) = timed(st, lambda: plr.lowpass_rows(rows), reps)
    Ed = torch.as_tensor(np.ascontiguousarray(E), device=dev)
    msd = torch.as_tensor(sm[0].copy(), device=dev)
    dv["project_ms"], P = timed(st, lambda: pl.pca_project(Xd, msd, Ed), reps)
    f = np.linspace(1100., 1900., nchan)
    t_spl, _ = host(lambda: si.splprep(P[:, :2].T, u=f, w=np.full(nchan, 100.), k=3, s=2.0 * nchan), reps)
    out["device_ms"] = dv
    out["host_eigh_ms"], out["host_splprep_ms"] = t_eigh, t_spl
    t0 = time.perf_counter()
    r = pplib.make_spline_model(X, f, noise_stds=np.full(nchan, 0.01), max_ncomp=m, norm=None)
    out["make_spline_model_ms"] = 1e3 * (time.perf_counter() - t0)   # first call at this shape: plans created
    t0 = time.perf_counter()
    r = pplib.make_spline_model(X, f, noise_stds=np.full(nchan, 0.01), max_ncomp=m, norm=None)
    out["make_spline_model_warm_ms"] = 1e3 * (time.perf_counter() - t0)
    out["ncomp"] = int(r.ncomp)
    # the same steps in numpy float64 on the host cores
    nh = {}

    def np_moments():
        mu_ = (w[:, None] * X).sum(0) / w.sum()
        D = np.sqrt(w)[:, None] * (X - mu_)
        return mu_, (D @ D.T if gram else D.T @ D) / w.sum()
    nh["moments_ms"], _ = host(np_moments, reps)
    if gram:
        nh["backproject_ms"], _ = host(lambda: (np.sqrt(w)[:, None] * (X - mu)).T @ Uv, reps)
    nh["lowpass_ms"], _ = host(lambda: lowpass(np.vstack([mu[None], E.T])), 1)
    nh["project_ms"], _ = host(lambda: (X - sm[0]) @ E, reps)
    out["host_numpy_ms"] = nh
    out["host_threads"] = os.cpu_count()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "spline_build_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, q = card()
    res = dict(card=name, power_limit_and_max_sm_clock=q, shapes=[probe(512, 2048, 10, a.reps),
                                                                  probe(4096, 1024, 10, a.reps)])
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
