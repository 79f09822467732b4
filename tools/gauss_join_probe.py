"""Throughput of the evolving-Gaussian portrait fit with join parameters (pp_fit_gaussian_portraits_join).

Three archives of 256 channels x 2048 bins joined into one 768-channel portrait (the restatement of
tests/test_cpu_gaussjoin.py with the two later archives rotated by phase and DM offsets), 3 components, tau and
alpha fixed, every component parameter and every (phi_j, DM_j) free.  For batches of 1 and 16 portraits the
joined fit and the unjoined fit of the same portraits (no join groups, P = 3 + 6 ngauss) are timed alternately in
one process: portraits per second and evaluations per fit.  The pass kernel's device time per evaluation is taken
from a separate torch.profiler run (CUDA activity) of one evaluation (max_iter < 0) of each.  Prints one JSON line
per measurement; the first names the card and its power limit.

    python tools/gauss_join_probe.py [--out FILE] [--reps 3]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.gauss_fit_probe import card  # noqa: E402


def pass_ms(fn):
    """Device time [ms] of the k_gfit_pass launches of fn(), by torch.profiler's CUDA activity."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot, n = 0.0, 0
    for e in prof.events():
        if "k_gfit_pass" in e.name:
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            n += 1
    return tot / 1e3, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    from pulseportraiture_b200.engine import WidebandPlan
    from tests.test_cpu_gaussjoin import PSPIN, make_join_problem, model_time_join
    nchan, nbin, njoin, ngauss, sigma, code = 768, 2048, 2, 3, 0.05, "000"
    lines = [dict(card())]
    print(json.dumps(lines[0]), flush=True)
    p_true, freqs, nu_ref, _, _, jc = make_join_problem(code, nchan, nbin, njoin, seed=7, ngauss=ngauss, sigma=sigma)
    clean = model_time_join(code, p_true, freqs, nu_ref, nbin, jc, PSPIN)
    ia = len(p_true) - 2 * njoin - 1
    rng = np.random.RandomState(1)
    init = p_true.copy()
    init[2:ia] *= 1 + 0.01 * rng.randn(ia - 2)
    free = np.ones(len(p_true), bool)
    free[1] = free[ia] = False
    cases = {"joined": dict(x=init, free=free, kw=dict(join_chan=jc, P=PSPIN)),
             "unjoined": dict(x=init[:ia + 1], free=free[:ia + 1], kw={})}
    with WidebandPlan(nchan, nbin) as pl:
        pl.set_freqs(freqs)
        for nport in (1, 16):
            data = clean[None] + sigma * rng.randn(nport, nchan, nbin)
            errs = np.full((nport, nchan), sigma)
            best = {k: np.inf for k in cases}
            res = {}
            for k, c in cases.items():   # warm-up
                pl.fit_gaussian_portraits(data, errs, code, np.tile(c["x"], (nport, 1)), c["free"], nu_ref, **c["kw"])
            for _ in range(args.reps):
                for k, c in cases.items():
                    x0 = np.tile(c["x"], (nport, 1))
                    t0 = time.perf_counter()
                    res[k] = pl.fit_gaussian_portraits(data, errs, code, x0, c["free"], nu_ref, **c["kw"])
                    best[k] = min(best[k], time.perf_counter() - t0)   # returns synchronised
            for k, c in cases.items():
                x0 = np.tile(c["x"], (nport, 1))
                ms, nl = pass_ms(lambda: pl.fit_gaussian_portraits(data, errs, code, x0, c["free"], nu_ref,
                                                                   max_iter=-1, **c["kw"]))
                r = res[k]
                lines.append(dict(what=k, nport=nport, nchan=nchan, nbin=nbin, ngauss=ngauss,
                                  njoin=njoin if k == "joined" else 0, nparam=int(len(c["x"])),
                                  seconds=best[k], portraits_per_s=nport / best[k],
                                  nfeval_mean=float(r["nfeval"].mean()),
                                  converged=int((r["return_code"] == 0).sum()),
                                  pass_ms_per_evaluation=ms, pass_launches=nl))
                print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(json.dumps(l) for l in lines) + "\n")


if __name__ == "__main__":
    main()
