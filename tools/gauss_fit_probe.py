"""Throughput of the evolving-Gaussian portrait fit (pp_fit_gaussian_portraits).

Portraits fit per second and model evaluations per fit for batches of 1 / 16 / 64 portraits of
512 x 2048 with 3 and 8 components, tau and alpha free, next to one scipy.optimize.least_squares fit of
the same problem on the host (the numpy restatement of tests/test_cpu_gaussfit.py, analytic Jacobian).
Prints one JSON line per measurement; the first names the card and its power limit.

    python tools/gauss_fit_probe.py [--out FILE] [--no-scipy]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True).strip().splitlines()[0]
        name, power, clock = [v.strip() for v in out.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:   # the measurement still stands; say what is missing
        return dict(gpu="unknown (%s)" % e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-scipy", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from pulseportraiture_b200.engine import WidebandPlan
    from tests.test_cpu_gaussfit import make_problem, model_time, restate
    nchan, nbin, sigma = 512, 2048, 0.05
    lines = [dict(card())]
    for ngauss in (3, 8):
        code = "000"
        p_true, freqs, nu_ref, _, _ = make_problem(code, nchan, nbin, tau=1.5, seed=ngauss, ngauss=ngauss,
                                                   sigma=sigma)
        clean = model_time(code, p_true, freqs, nu_ref, nbin)
        rng = np.random.RandomState(1)
        free = np.ones(len(p_true), bool)
        init = p_true * (1 + 0.01 * rng.randn(len(p_true)))
        with WidebandPlan(nchan, nbin) as pl:
            pl.set_freqs(freqs)
            for nport in (1, 16, 64):
                data = clean[None] + sigma * rng.randn(nport, nchan, nbin)
                errs = np.full((nport, nchan), sigma)
                x0 = np.tile(init, (nport, 1))
                pl.fit_gaussian_portraits(data, errs, code, x0, free, nu_ref)          # warm-up
                best = np.inf
                for _ in range(args.reps):
                    t0 = time.perf_counter()
                    r = pl.fit_gaussian_portraits(data, errs, code, x0, free, nu_ref)   # returns synchronised
                    best = min(best, time.perf_counter() - t0)
                lines.append(dict(what="device", ngauss=ngauss, nport=nport, nchan=nchan, nbin=nbin,
                                  seconds=best, portraits_per_s=nport / best,
                                  nfeval_mean=float(r["nfeval"].mean()),
                                  converged=int((r["return_code"] == 0).sum())))
                print(json.dumps(lines[-1]), flush=True)
        if not args.no_scipy:
            from scipy.optimize import least_squares
            data = clean + sigma * rng.randn(nchan, nbin)
            errs = np.full(nchan, sigma)
            nev = [0]

            def fun(q):
                nev[0] += 1
                rr = restate(code, q, freqs, nu_ref, nbin, data, errs)
                sw = np.sqrt(rr["w"])
                return np.concatenate([(sw * rr["R"].real).ravel(), (sw * rr["R"].imag).ravel()])

            def jac(q):
                rr = restate(code, q, freqs, nu_ref, nbin, data, errs)
                sw = np.sqrt(rr["w"])[:, None, :]
                return -np.concatenate([(sw * rr["J"].real).transpose(0, 2, 1).reshape(-1, len(q)),
                                        (sw * rr["J"].imag).transpose(0, 2, 1).reshape(-1, len(q))])
            t0 = time.perf_counter()
            res = least_squares(fun, init, jac=jac, method="lm", xtol=1e-10, ftol=1e-10)
            lines.append(dict(what="host scipy lm (numpy restatement)", ngauss=ngauss, nport=1,
                              seconds=time.perf_counter() - t0, nfev=int(res.nfev), njev=int(res.njev or 0)))
            print(json.dumps(lines[-1]), flush=True)
    print(json.dumps(lines[0]), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
