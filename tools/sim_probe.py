"""Throughput of the simulated-archive kernels on one GPU, beside the fit of the same rows.

10 000 subints of 512 x 2048 (bench.py's portrait shape) from the example .gmodel, every output device-resident:
  - WidebandPlan.simulate_batch with float32 output and with int16 (+ DAT_SCL / DAT_OFFS) output: ms per call,
    subints/s and GB/s written (output bytes over the call time);
  - the closed loop simulate (int16) -> fit_batch on those rows: TOA/s;
  - fit_batch on the float32 rows of the same simulate call, alternated with the simulate calls: the step time
    and stats()["ms_spectra"] (the data-transform kernels, CUDA events).
Times are host clocks around calls that end in a device synchronise, medians over --reps repetitions after one
warm-up of every shape.  The card's name and power limit (nvidia-smi, read-only query) go beside the numbers.

    python tools/sim_probe.py --out profiles/sim_b200.json
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

NCHAN, NBIN, NU0, BW = 512, 2048, 1500.0, 800.0
GMODEL = os.path.join(ROOT, "tests", "golden", "example.gmodel")
P_EXAMPLE = 1.0 / 345.67890123456789


def gpu_info():
    q = ["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        name, plim, smax = [v.strip() for v in subprocess.check_output(q, text=True).strip().split(",")]
        return {"name": name, "power_limit": plim, "sm_max_clock": smax}
    except Exception as e:   # the numbers are still worth keeping; say that the card was not identified
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nsub", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sim_b200.json"))
    args = ap.parse_args()
    import torch
    from pulseportraiture_b200 import pplib
    from pulseportraiture_b200.engine import WidebandPlan
    if not torch.cuda.is_available():
        raise SystemExit("sim_probe needs a CUDA device")
    dev = torch.device("cuda", 0)
    nsub = args.nsub
    freqs = np.linspace(NU0 - BW / 2 + BW / (2.0 * NCHAN), NU0 + BW / 2 - BW / (2.0 * NCHAN), NCHAN)
    model = pplib.read_model(GMODEL, pplib.get_bin_centers(NBIN), freqs, P_EXAMPLE, quiet=True, device=True)[2]
    model = np.ascontiguousarray(model, dtype=np.float64)
    rng = np.random.RandomState(1)
    phase = torch.tensor(rng.uniform(-0.5, 0.5, nsub), device=dev)
    DM = torch.tensor(rng.normal(0.0, 1e-3, nsub), device=dev)
    P = torch.full((nsub,), P_EXAMPLE, dtype=torch.float64, device=dev)
    nu_DM = torch.full((nsub,), NU0, dtype=torch.float64, device=dev)
    sigma = torch.full((nsub, NCHAN), 1.0, dtype=torch.float64, device=dev)
    out32 = torch.empty((nsub, NCHAN, NBIN), dtype=torch.float32, device=dev)
    raw = torch.empty((nsub, NCHAN, NBIN), dtype=torch.int16, device=dev)
    scl = torch.empty((nsub, NCHAN), dtype=torch.float32, device=dev)
    offs = torch.empty((nsub, NCHAN), dtype=torch.float32, device=dev)
    pl = WidebandPlan(NCHAN, NBIN)
    pl.set_model(model, freqs)

    def sim(quantize, seed):
        o = (raw, scl, offs) if quantize else out32
        return pl.simulate_batch(model, freqs, phase, DM, P, nu_DM, noise_stds=sigma, seed=seed, quantize=quantize,
                                 out=o)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    # warm-up of every shape
    sim(False, 0)
    sim(True, 0)
    pl.fit_batch(out32, P_EXAMPLE, pinned_results=True)
    pl.fit_batch(raw, P_EXAMPLE, dat_scl=scl, dat_offs=offs, pinned_results=True)
    t_f32, t_i16, t_fit, t_spec, t_fit16, t_loop, k_f32, t_clean, k_clean = [], [], [], [], [], [], [], [], []
    for rep in range(args.reps):      # simulate and fit alternate, on the same plan and the same rows
        pl.enable_timing(True)        # ms_total: CUDA events around the simulate kernels (no host checks, no set-up)
        t_f32.append(timed(lambda: sim(False, rep + 1))[0])
        k_f32.append(pl.stats()["ms_total"])
        t_clean.append(timed(lambda: pl.simulate_batch(model, freqs, phase, DM, P, nu_DM, out=out32))[0])
        k_clean.append(pl.stats()["ms_total"])
        t_fit.append(timed(lambda: pl.fit_batch(out32, P_EXAMPLE, pinned_results=True))[0])
        t_spec.append(pl.stats()["ms_spectra"])
        pl.enable_timing(False)
        t_i16.append(timed(lambda: sim(True, rep + 1))[0])
        t_fit16.append(timed(lambda: pl.fit_batch(raw, P_EXAMPLE, dat_scl=scl, dat_offs=offs,
                                                  pinned_results=True))[0])
        t_loop.append(timed(lambda: (sim(True, 100 + rep),
                                     pl.fit_batch(raw, P_EXAMPLE, dat_scl=scl, dat_offs=offs,
                                                  pinned_results=True)))[0])
    r = pl.fit_batch(raw, P_EXAMPLE, dat_scl=scl, dat_offs=offs)
    med = lambda v: float(np.median(v))                          # noqa: E731
    rows = nsub * NCHAN
    b32 = rows * NBIN * 4.0
    b16 = rows * (NBIN * 2.0 + 8.0)
    res = {
        "gpu": gpu_info(),
        "shape": {"nsub": nsub, "nchan": NCHAN, "nbin": NBIN, "model": "tests/golden/example.gmodel"},
        "method": "host clock around calls ending in a device synchronise; median of %d repetitions after a "
                  "warm-up; simulate and fit alternate on one plan; all outputs device-resident" % args.reps,
        "simulate_f32": {"ms": 1e3 * med(t_f32), "subints_per_s": nsub / med(t_f32),
                         "GB_per_s_written": b32 / med(t_f32) / 1e9, "all_ms": [1e3 * t for t in t_f32]},
        "simulate_f32_kernels_ms": med(k_f32),
        "simulate_f32_no_noise": {"ms": 1e3 * med(t_clean), "kernels_ms": med(k_clean)},
        "simulate_i16": {"ms": 1e3 * med(t_i16), "subints_per_s": nsub / med(t_i16),
                         "GB_per_s_written": b16 / med(t_i16) / 1e9, "all_ms": [1e3 * t for t in t_i16]},
        "fit_f32": {"ms": 1e3 * med(t_fit), "ms_spectra": med(t_spec), "all_ms": [1e3 * t for t in t_fit]},
        "fit_i16": {"ms": 1e3 * med(t_fit16), "all_ms": [1e3 * t for t in t_fit16]},
        "loop_simulate_i16_fit": {"ms": 1e3 * med(t_loop), "toa_per_s": nsub / med(t_loop)},
        "ratio_simulate_f32_over_fit_f32": med(t_f32) / med(t_fit),
        "ratio_simulate_i16_over_fit_i16": med(t_i16) / med(t_fit16),
        "loop_return_codes_converged": float(np.mean(r["return_code"] == 0)),
    }
    pl.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
