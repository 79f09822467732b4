#!/usr/bin/env python
"""Benchmark of the wideband-TOA hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA)
    python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm
    python bench.py ... --dump-outputs DIR                   # + the last timed step's result arrays, DIR/*.npy

Workload (config 2): phi+DM fit, 512 chan x 2048 bin, 10k subints per GPU per
step, synthetic portraits from example.gmodel (rotated model + white noise).
One "step" = the complete hot path over the batch: per-channel rfft + noise +
cross-spectrum (K1/K2), FFTFIT initial guess (K4), Newton solve with fused
rotate-reduce passes (K3/K3'), epilogue, D2H of the result arrays.

value  : TOAs/s, inputs resident in HBM when the timed region starts.
e2e    : TOAs/s through the same C-ABI call with HOST (pinned) input buffers,
         H2D copies inside the timed region (on a smaller batch, stated).
For N > 1 launch with torchrun (one rank per GPU); subints are sharded with no
data-path collective ("weak" scaling: fixed work per GPU).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NCHAN, NBIN, NU0, BW = 512, 2048, 1500.0, 800.0
P_EXAMPLE = 1.0 / 345.67890123456789
SIGMA = 1.5
GMODEL = os.path.join(ROOT, "tests", "golden", "example.gmodel")
N_PASS_CONTRACT = 5          # SURVEY 8d: bytes/TOA = 4*nchan*nbin*(2+N_pass)
BYTES_PER_TOA_CONTRACT = 4 * NCHAN * NBIN * (2 + N_PASS_CONTRACT)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------
# synthetic inputs
# ------------------------------------------------------------------------------
def make_model():
    from pulseportraiture_b200 import pplib
    freqs = np.linspace(NU0 - BW / 2 + BW / (2.0 * NCHAN), NU0 + BW / 2 - BW / (2.0 * NCHAN), NCHAN)
    phases = pplib.get_bin_centers(NBIN)
    _, _, model = pplib.read_model(GMODEL, phases, freqs, P_EXAMPLE, quiet=True)
    return freqs, model


def make_device_batch(model, freqs, phi_np, dDM_np, seed, device, nchan=NCHAN, nbin=NBIN, nu0=NU0,
                      scatter=None):
    """data_s = rotate(model, -phi_s, -dDM_s) + N(0, sigma^2) as float32 on the
    GPU (torch is plumbing here: untimed setup).  scatter = (tau [rot] at nu0, alpha) scatters the
    model first (config 3)."""
    import torch
    from pulseportraiture_b200.pplib import Dconst
    nsub = len(phi_np)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    mFT = torch.fft.rfft(torch.from_numpy(model).to(device), dim=-1)      # [nchan, nharm] c128
    k = torch.arange(mFT.shape[-1], device=device, dtype=torch.float64)
    if scatter is not None:
        taus = torch.from_numpy(scatter[0] * (freqs / nu0) ** scatter[1]).to(device)
        mFT = mFT / (1.0 + 2j * np.pi * taus[:, None] * k[None, :])
    nu2 = torch.from_numpy(freqs ** -2.0 - nu0 ** -2.0).to(device)
    out = torch.empty((nsub, nchan, nbin), dtype=torch.float32, device=device)
    phi = torch.from_numpy(np.asarray(phi_np, dtype=np.float64)).to(device)
    dDM = torch.from_numpy(np.asarray(dDM_np, dtype=np.float64)).to(device)
    step = max(1, (128 * NCHAN * NBIN) // (nchan * nbin))
    for a in range(0, nsub, step):
        b = min(nsub, a + step)
        shifts = -phi[a:b, None] - (Dconst * dDM[a:b, None] / P_EXAMPLE) * nu2[None, :]
        ph = torch.exp(2j * np.pi * (shifts[:, :, None] * k[None, None, :]))
        clean = torch.fft.irfft(mFT[None] * ph, n=nbin, dim=-1)
        noise = torch.randn(clean.shape, generator=g, device=device, dtype=torch.float32)
        out[a:b] = clean.to(torch.float32) + SIGMA * noise
    return out


def global_draws(n, seed=777):
    """phi_s ~ U(-0.5, 0.5), dDM_s ~ N(3e-4, 2e-4) of subint s of the global batch: a function of the
    global subint index only, so every world size fits the same batch."""
    rng = np.random.default_rng(seed)
    return rng.random(n) - 0.5, 3e-4 + 2e-4 * rng.standard_normal(n)


# ------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference, one subint per task)
# ------------------------------------------------------------------------------
def _cpu_worker(args):
    seed, = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    from oracle import pp_oracle as orc
    from tests import synth
    c = synth.make_case(NCHAN, NBIN, NU0, BW, seed)
    t = time.perf_counter()
    noise = orc.get_noise(c["data"], chans=True)
    res, _, _ = orc.toa_core(c["data"], c["model"], c["P"], c["freqs"], noise)
    return time.perf_counter() - t, float(res.phi)


def cpu_baseline(nsamples=None, cores=None):
    """Time the CPU oracle (numpy/scipy port of the reference path:
    get_noise -> FFTFIT guess -> fit_portrait_full trust-ncg) on a bounded
    sample of the same workload, one process per host core."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    nsamples = nsamples or max(16, 2 * cores)
    from tests import synth
    synth.example_model(NCHAN, NBIN, NU0, BW)        # warm the model cache before forking
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(9000 + i,) for i in range(cores)])          # warm-up
        t0 = time.perf_counter()
        out = pool.map(_cpu_worker, [(9100 + i,) for i in range(nsamples)], chunksize=1)
        wall = time.perf_counter() - t0
    per = float(np.mean([o[0] for o in out]))
    return {"value": nsamples / wall, "unit": "TOAs/s", "cores": cores, "kind": "port",
            "sample": "%d subints of 512x2048 (oracle port: get_noise + FFTFIT guess + "
                      "fit_portrait_full trust-ncg), %d processes, %.2f s/TOA/core"
                      % (nsamples, cores, per)}


# ------------------------------------------------------------------------------
def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    nsamp = max(8, cores)
    vals = []
    for _ in range(args.warmup and 1):
        cpu_baseline(nsamp, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        vals.append(cpu_baseline(nsamp, cores))
    wall = time.perf_counter() - t0
    v = float(np.mean([x["value"] for x in vals]))
    line = {"impl": "reference", "metric": "wideband TOAs/sec (phi+DM fit, 512ch x 2048bin)",
            "value": v, "unit": "TOAs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "phi+DM batch fit, 512 chan x 2048 bin (config 2), "
                                   "bounded sample of %d subints per step" % nsamp},
            "cpu_baseline": dict(vals[-1], value=v),
            "e2e": {"value": v, "unit": "TOAs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


# FP64 thread-instructions the two main kernels execute (ncu source counters of the committed captures,
# profiles/r02_k_spectra16.md, r02_k_pass2.md, traffic_r02.json): per (row, thread) and per harmonic
FP64_PER_THREAD_ROW_SPECTRA = 712.3
FP64_PER_HARMONIC_PASS2 = 17.56

# per-subint scalars that travel in the host-side gather (TOA-level results; the per-channel arrays
# stay with the rank that computed them, as an archive's scales stay with its TOA file)
GATHER_KEYS = ("params", "param_errs", "nu_out", "cov", "chi2", "red_chi2", "snr", "nfeval",
               "return_code", "lag_index")


# --dump-outputs: array bytes written in all, leaving room under 64 MB for the .npy headers
DUMP_BYTES = 60 * 10 ** 6


def dump_outputs(res, nsub, outdir, seed=0):
    """Write the arrays of one fit_batch call, every one indexed by subint first, as outdir/<name>.npy.
    float32 arrays stay float32, everything else is written as float64 (integer codes are exact there).
    When the batch does not fit DUMP_BYTES, every array keeps the same seeded sample of subints (sorted),
    as many as fit: the rows depend only on nsub and seed, so two builds run with the same arguments
    write arrays that compare element for element."""
    arrs = {k: np.asarray(v) for k, v in res.items()}
    dts = {k: np.float32 if a.dtype == np.float32 else np.float64 for k, a in arrs.items()}
    row_bytes = sum(np.dtype(dts[k]).itemsize * (a.size // nsub) for k, a in arrs.items())
    rows = min(nsub, DUMP_BYTES // row_bytes)
    idx = np.arange(nsub) if rows == nsub else np.sort(np.random.default_rng(seed).choice(nsub, rows, replace=False))
    os.makedirs(outdir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(outdir, k + ".npy"), a[idx].astype(dts[k]))
    return rows


def pack_toa_level(res, n):
    cols = [np.asarray(res[k][:n], dtype=np.float64).reshape(n, -1) for k in GATHER_KEYS]
    return np.ascontiguousarray(np.concatenate(cols, axis=1))


def unpack_toa_level(pack):
    out, c = {}, 0
    for k, w in zip(GATHER_KEYS, (5, 5, 3, 25, 1, 1, 1, 1, 1, 1)):
        out[k] = pack[:, c:c + w] if w > 1 else pack[:, c]
        c += w
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from pulseportraiture_b200.engine import WidebandPlan
    from pulseportraiture_b200.multigpu import shard_range, bind_to_gpu_numa, SharedGather

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local = env_int("LOCAL_RANK", 0)
    gloo = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gloo = dist.new_group(backend="gloo")     # host-side gather of the result arrays: no NCCL on the data path
    if args.gpus != world and rank == 0 and world == 1 and args.gpus > 1:
        print("note: --gpus %d without torchrun: running 1 rank" % args.gpus, file=sys.stderr)
    torch.cuda.set_device(local)
    try:
        all_cpus = os.sched_getaffinity(0)
    except AttributeError:
        all_cpus = None
    # each rank (and the page-locked buffers it allocates from here on) stays on its GPU's NUMA node
    numa = bind_to_gpu_numa(local) if not args.no_numa else {"cpus": 0, "bound": False}
    dev = torch.device("cuda", local)
    nsub = args.nsub
    freqs, model = make_model()
    stream = torch.cuda.Stream(device=dev)
    plan = WidebandPlan(NCHAN, NBIN, device=local, stream=stream)
    plan.set_model(np.ascontiguousarray(model, dtype=np.float64), freqs)   # float64, the reference's model type
    if args.chunk:
        plan.set_chunk(args.chunk)
    if args.fft:
        plan.set_fft_precision(args.fft)
    # ONE global batch of world * nsub subints (weak scaling: nsub per GPU), sharded in contiguous ranges
    nglob = world * nsub
    phi_all, dDM_all = global_draws(nglob)
    a0, b0 = shard_range(nglob, rank, world)
    data = make_device_batch(model, freqs, phi_all[a0:b0], dDM_all[a0:b0], 777 + rank, dev)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shg = SharedGather(nsub, 44, group=gloo, tag="toa") if world > 1 else None

    def gather_packed(pack):
        """Host-side gather of packed TOA-level rows on rank 0: shared memory + a gloo barrier."""
        if world == 1:
            return unpack_toa_level(pack)
        allrows = shg.gather(pack)
        return unpack_toa_level(allrows) if rank == 0 else None

    def gather(res, n):
        return gather_packed(pack_toa_level(res, n))

    class AsyncGather(object):
        """The gather of step k runs on a host thread while step k + 1 computes (the result arrays are
        packed out of the plan's page-locked buffers first: the next call overwrites them); join()
        inside the timed region waits for the last one."""

        def __init__(self):
            self.thread, self.out = None, None

        def submit(self, res, n):
            self.join()
            pack = pack_toa_level(res, n)

            def work():
                self.out = gather_packed(pack)
            self.thread = threading.Thread(target=work)
            self.thread.start()

        def join(self):
            if self.thread is not None:
                self.thread.join()
                self.thread = None
            return self.out

    def step(d=data, n=nsub):
        return plan.fit_batch(d, P_EXAMPLE, nsub=n, tol=args.tol, max_iter=args.max_iter,
                              pinned_results=True)

    for _ in range(args.warmup):
        res = step()
        glob = gather(res, nsub)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        launches = 0
        ag = AsyncGather()
        # per-kernel CUDA-event times are taken over the timed steps themselves (events around every launch on
        # the plan's stream), so that they are at the clocks the step sustains under its power cap
        plan.enable_timing(True)
        st_sum, npass_sum = None, 0.0
        for _ in range(args.steps):
            res = step()
            st_i = plan.stats()
            npass_sum += float(np.sum(res["nfeval"]))
            ag.submit(res, nsub)                 # gathered on rank 0 while the next step computes
            launches += st_i["launches"]
            if st_sum is None:
                st_sum = dict(st_i)
            else:
                for k_ in ("ms_spectra", "ms_guess", "ms_pass", "ms_update", "ms_total", "pass_launches"):
                    st_sum[k_] += st_i[k_]
        plan.enable_timing(False)
        glob = ag.join()                         # ... the last one inside the timed region
        ev1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        # res still holds the last timed step's arrays: the next fit_batch call on this plan overwrites them
        dump_outputs(res, nsub, args.dump_outputs)
    tt = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_max = float(tt.item())
    value = world * nsub * args.steps / (ms_max * 1e-3)

    # sanity of the timed work on the GATHERED global batch: parameters recovered, every subint converged
    ok = mean_pass = pull_rms = None
    if rank == 0:
        ok = int(np.sum(glob["return_code"] == 0))
        mean_pass = float(np.mean(glob["nfeval"]))
        pull = (glob["params"][:, 1] - dDM_all) / glob["param_errs"][:, 1]
        pull_rms = float(np.sqrt(np.mean(pull ** 2)))

    # ---- strong scaling (extra key): a fixed global batch of nsub subints split over the ranks ------
    strong = None
    if world > 1:
        sa, sb = shard_range(nsub, rank, world)
        ns_loc = sb - sa

        def strong_step():
            r = plan.fit_batch(data[:ns_loc], P_EXAMPLE, nsub=ns_loc, tol=args.tol, max_iter=args.max_iter,
                               pinned_results=True)
            gather(r, ns_loc)
        strong_step()
        barrier()
        ts = time.perf_counter()
        for _ in range(args.steps):
            strong_step()
        barrier()
        tsv = torch.tensor([time.perf_counter() - ts], device=dev, dtype=torch.float64)
        dist.all_reduce(tsv, op=dist.ReduceOp.MAX)
        strong = {"global_subints": nsub, "value": nsub * args.steps / float(tsv.item()), "unit": "TOAs/s",
                  "ms_per_step": 1e3 * float(tsv.item()) / args.steps,
                  "note": "the same %d-subint batch split over %d GPUs, host-side gather inside the timed region"
                          % (nsub, world)}

    # ---- per-kernel times for the roofline: averages over the timed steps --------
    st = dict(st_sum)
    for k_ in ("ms_spectra", "ms_guess", "ms_pass", "ms_update", "ms_total"):
        st[k_] = st_sum[k_] / args.steps
    st["pass_launches"] = int(round(st_sum["pass_launches"] / args.steps))
    B = 4.0 * NCHAN * NBIN                                               # bytes of one portrait
    npass = npass_sum / args.steps                                       # subint-passes over X per step
    keep = float(st.get("x_keep_frac", 1.0)) or 1.0                      # share of X the model's harmonic cut-off keeps
    pass_bytes = npass * B * keep                                        # kept X re-read per pass
    spec_bytes = (1.0 + keep) * B * nsub                                 # read portrait + write kept X
    hbm_peak, peak_src = peaks()
    fp64_peak = plan.measure_fp64()                                      # DFMA thread-instructions / s, measured here
    n_spec = -(-nsub // st["chunk"])
    fp64_spec = FP64_PER_THREAD_ROW_SPECTRA * 64.0 * NCHAN * nsub        # 64 threads per channel row
    fp64_pass = FP64_PER_HARMONIC_PASS2 * (NBIN // 2) * keep * NCHAN * npass
    kern = {
        "k_spectra": {"algorithmic_bytes_per_launch": spec_bytes / n_spec, "launches": n_spec,
                      "ms": st["ms_spectra"],
                      "achieved_gbs": spec_bytes / (st["ms_spectra"] * 1e-3) / 1e9,
                      "fp64_inst": fp64_spec, "fp64_frac": fp64_spec / (st["ms_spectra"] * 1e-3) / fp64_peak},
        "k_pass2": {"algorithmic_bytes_per_launch": pass_bytes / max(1, st["pass_launches"]),
                    "launches": st["pass_launches"], "ms": st["ms_pass"],
                    "achieved_gbs": pass_bytes / (st["ms_pass"] * 1e-3) / 1e9,
                    "fp64_inst": fp64_pass, "fp64_frac": fp64_pass / (st["ms_pass"] * 1e-3) / fp64_peak},
        "k_guess": {"ms": st["ms_guess"]}, "k_update2": {"ms": st["ms_update"]},
    }
    for k in ("k_spectra", "k_pass2"):
        kern[k]["frac"] = kern[k]["achieved_gbs"] / hbm_peak
    dom = "k_spectra" if st["ms_spectra"] >= st["ms_pass"] else "k_pass2"
    desc = {"k_spectra": "k_spectra16 (FP64 rfft + noise + cross-spectrum, K1/K2)",
            "k_pass2": "k_pass2 (fused rotate-reduce objective pass, K3)"}[dom]
    mp_t = npass / nsub
    ms_step = ms_max / args.steps
    roof = {"bound": "hbm", "kernel": desc, "achieved": kern[dom]["achieved_gbs"],
            "peak": hbm_peak, "unit": "GB/s", "frac": kern[dom]["frac"], "peak_source": peak_src,
            "traffic": None,
            "algorithmic_bytes_per_launch": kern[dom]["algorithmic_bytes_per_launch"],
            "launches": kern[dom]["launches"], "kernels": kern, "ms_total": st["ms_total"],
            "timing": "CUDA events around every launch of the timed steps, averaged per step",
            "chunk_subints": st["chunk"],
            # the whole step on the bytes it actually moves: portrait in, X out, X back in once per pass
            "x_keep_frac": keep,
            # the same kernel time against the bytes it moved before the harmonic cut-off (read portrait + write ALL of
            # X): comparable with the round-1 figure; the kernel is FP64-bound, its time does not depend on the stores
            "frac_on_full_x_bytes": 2.0 * B * nsub / (kern["k_spectra"]["ms"] * 1e-3) / (hbm_peak * 1e9),
            "note": "dominant kernel k_spectra16 is FP64-pipe bound (roofline.fp64); frac counts the algorithmic bytes "
                    "it moves now (portrait in + kept x_keep_frac of X out)",
            "step_bytes_per_toa_actual": B * (1.0 + keep * (1.0 + mp_t)),
            "step_frac_actual_bytes": nsub * B * (1.0 + keep * (1.0 + mp_t)) / (ms_step * 1e-3) / (hbm_peak * 1e9),
            # secondary bound: both main kernels are FP64 co-limited
            "fp64": {"peak_dfma_per_s": fp64_peak, "how": "pp_measure_fp64: independent DFMA chains, 4 CTAs x 256 threads per SM, "
                                                          "best of 3, measured in this run",
                     "k_spectra_frac": kern["k_spectra"]["fp64_frac"], "k_pass2_frac": kern["k_pass2"]["fp64_frac"],
                     "fp64_inst_source": "ncu thread-instruction counters: %.0f per (row, thread) in k_spectra16, %.2f per "
                                         "harmonic in k_pass2 (profiles/)" % (FP64_PER_THREAD_ROW_SPECTRA, FP64_PER_HARMONIC_PASS2)},
            # NOT a roofline fraction: throughput against SURVEY 8d's estimate, which assumed 5 passes over X
            "survey_contract_bytes_per_toa": BYTES_PER_TOA_CONTRACT,
            "throughput_vs_survey_5pass_estimate": value / world * BYTES_PER_TOA_CONTRACT / (hbm_peak * 1e9)}
    tfile = os.path.join(ROOT, "profiles", "traffic_r02.json")
    if not os.path.isfile(tfile):
        tfile = os.path.join(ROOT, "profiles", "traffic_r01.json")
    if os.path.isfile(tfile):
        try:   # DRAM bytes per launch from the committed ncu capture, scaled to this launch size
            tj = json.load(open(tfile))
            kern["k_pass2"]["traffic"] = tj["k_pass2_dram_bytes_per_subint_pass"] * \
                npass / max(1, st["pass_launches"])
            kern["k_spectra"]["traffic"] = tj["k_spectra_dram_bytes_per_subint"] * nsub / n_spec
            roof["traffic"] = kern[dom]["traffic"]
        except Exception:  # noqa: BLE001
            pass

    # ---- e2e: host (pinned) buffers through the same C-ABI call --------------------------
    n_e2e = min(nsub, args.e2e_nsub)
    host = torch.empty((n_e2e, NCHAN, NBIN), dtype=torch.float32).pin_memory()
    host.copy_(data[:n_e2e])
    torch.cuda.synchronize()
    hnp = host.numpy()
    step(hnp, n_e2e)                                   # warm the staging buffers
    barrier()
    t0 = time.perf_counter()
    reps = max(1, args.e2e_steps)
    for _ in range(reps):
        r_e = step(hnp, n_e2e)
        gather(r_e, n_e2e)
    barrier()
    e2e_wall = time.perf_counter() - t0
    te = torch.tensor([e2e_wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    d2h = sum(v.nbytes for v in r_e.values())
    # the ceiling of this leg: a bare page-locked host -> device copy of the same buffer, every rank at once
    stage = torch.empty((n_e2e, NCHAN, NBIN), dtype=torch.float32, device=dev)
    stage.copy_(host, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        stage.copy_(host, non_blocking=True)
    barrier()
    tc = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    del stage
    h2d_ceiling = world * hnp.nbytes * reps / float(tc.item()) / 1e9
    e2e_gbs = world * hnp.nbytes * reps / float(te.item()) / 1e9
    e2e = {"value": world * n_e2e * reps / float(te.item()), "unit": "TOAs/s",
           "h2d_bytes_per_step": int(hnp.nbytes), "d2h_bytes_per_step": int(d2h),
           "subints_per_step": n_e2e, "steps": reps,
           "h2d_gbs_per_gpu": e2e_gbs / world, "h2d_gbs_total": e2e_gbs,
           "h2d_copy_ceiling_gbs_total": h2d_ceiling, "frac_of_copy_ceiling": e2e_gbs / h2d_ceiling,
           "note": "the ceiling is a bare cudaMemcpyAsync of the same page-locked buffers by all %d ranks at once: "
                   "the e2e leg is bound by the host's H2D bandwidth, which the ranks share" % world,
           "numa_bound": numa}

    # ---- the same call fed with the PSRFITS representation of the same portraits: int16 samples
    # with per-(subint, channel) DAT_SCL / DAT_OFFS, as archives store them (half the PCIe bytes)
    e2e_i16 = None
    try:
        d = data[:n_e2e]
        lo, hi = d.amin(dim=-1), d.amax(dim=-1)
        offs = (0.5 * (hi + lo)).to(torch.float32)
        scl = ((hi - lo) / 65000.0).to(torch.float32)
        raw = torch.clamp(torch.round((d - offs[..., None]) / scl[..., None]), -32768, 32767).to(torch.int16)
        hraw = torch.empty(raw.shape, dtype=torch.int16).pin_memory()
        hraw.copy_(raw)
        hscl, hoffs = scl.cpu().numpy(), offs.cpu().numpy()
        del raw, d
        torch.cuda.synchronize()
        rnp = hraw.numpy()

        def step16():
            return plan.fit_batch(rnp, P_EXAMPLE, nsub=n_e2e, tol=args.tol, max_iter=args.max_iter,
                                  pinned_results=True, dat_scl=hscl, dat_offs=hoffs)
        step16()
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            r16 = step16()
            gather(r16, n_e2e)
        barrier()
        t16 = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t16, op=dist.ReduceOp.MAX)
        e2e_i16 = {"value": world * n_e2e * reps / float(t16.item()), "unit": "TOAs/s",
                   "h2d_bytes_per_step": int(rnp.nbytes + hscl.nbytes + hoffs.nbytes),
                   "d2h_bytes_per_step": int(sum(v.nbytes for v in r16.values())),
                   "converged": "%d/%d" % (int((r16["return_code"] == 0).sum()), n_e2e),
                   "note": "same portraits as int16 + DAT_SCL/DAT_OFFS (PSRFITS DATA column), pp_fit_args_t.data_type = PP_DATA_I16"}
        del hraw
    except Exception as exc:  # noqa: BLE001
        e2e_i16 = {"error": str(exc)}
    del host

    facade = config3 = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            facade = facade_timing(data, freqs, model, args.facade_nsub)
        except Exception as exc:  # noqa: BLE001
            facade = {"error": repr(exc)}
        del data
        torch.cuda.empty_cache()
        try:
            config3 = config3_timing(dev, args.c3_nsub)
        except Exception as exc:  # noqa: BLE001
            config3 = {"error": repr(exc)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        if all_cpus is not None:
            os.sched_setaffinity(0, all_cpus)          # the CPU arm uses every host core
        cpu = cpu_baseline()

    if rank == 0:
        line = {"metric": "wideband TOAs/sec (phi+DM fit, 512ch x 2048bin)",
                "value": value, "unit": "TOAs/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "phi+DM batch fit, 512 chan x 2048 bin x %d subints per GPU "
                                       "(config 2), FFTFIT guess + Newton solve, noise measured"
                                       % nsub,
                           "sharding": "one global batch of %d subints in contiguous ranges, one rank per GPU; TOA-level result "
                                       "arrays gathered on rank 0 through shared memory inside the timed region (no NCCL on the data path)"
                                       % nglob,
                           "l2": "inputs (%.1f GB per GPU) larger than L2" % (nsub * B / 1e9),
                           "tol_sigma": min(args.tol, 1e-4) if args.tol else 1e-4, "mean_passes": mean_pass,
                           "solver": "Newton steps on the 4th-order local model of the per-channel sums; finishes "
                                     "without another pass when the estimated truncation shift is < 1e-4 sigma",
                           "fft_arith": "f64",
                           "converged": "%d/%d" % (ok, nglob),
                           "dDM_pull_rms": pull_rms},
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "roofline": roof, "cpu_baseline": cpu, "e2e_i16": e2e_i16, "strong_scaling": strong,
                "facade": facade, "config3": config3,
                "host_wall_ms_per_step": 1e3 * wall / args.steps}
        emit(line)
    if world > 1:
        shg.close()
        dist.destroy_process_group()
    return 0


def facade_timing(data, freqs, model, nsub):
    """What a reference user calls: GetTOAs(...).get_TOAs() on an archive of config-2 shape held as
    float64 (the reference's array type: no host conversion pass, PP_DATA_F64) and as the int16 +
    DAT_SCL/DAT_OFFS PSRFITS representation (the documented ingest for PSRFITS-origin data).  Wall time of
    the whole call: model build, H2D from pageable memory, fit, TOA objects."""
    from pulseportraiture_b200 import pptoas
    from pulseportraiture_b200.pplib import DataBunch, get_bin_centers
    nsub = min(nsub, data.shape[0])
    sub32 = data[:nsub].cpu().numpy()
    raw, scl, offs, dec = pptoas.quantize_subints(sub32)
    common = dict(backend="GUPPI", backend_delay=0.0, bw=BW, doppler_factors=np.ones(nsub), DM=0.0, dmc=0,
                  epochs=[pptoas.MJD(56000 + i // 100, 0.01 * (i % 100)) for i in range(nsub)], filename="bench.npz",
                  freqs=np.tile(freqs, (nsub, 1)), frontend="Rcvr_800", integration_length=float(nsub), masks=None,
                  nbin=NBIN, nchan=NCHAN, npol=1, nsub=nsub, nu0=NU0, ok_ichans=[np.arange(NCHAN)] * nsub,
                  ok_isubs=np.arange(nsub), parallactic_angles=np.zeros(nsub), phases=get_bin_centers(NBIN),
                  Ps=np.full(nsub, P_EXAMPLE), SNRs=np.ones((nsub, 1, NCHAN)), source="J0000+0000", state="Intensity",
                  subtimes=np.ones(nsub), telescope="GBT", telescope_code="1", weights=np.ones((nsub, NCHAN)),
                  noise_stds=np.full((nsub, 1, NCHAN), SIGMA), flux_prof=None, prof=None, prof_noise=None, prof_SNR=None)
    out = {"nsub": nsub, "unit": "TOAs/s"}
    for name, extra in (("get_TOAs_f64", dict(subints=sub32[:, None].astype(np.float64))),
                        ("get_TOAs_i16", dict(subints=dec[:, None], raw_subints=raw, dat_scl=scl, dat_offs=offs))):
        fields = dict(common, raw_subints=None, dat_scl=None, dat_offs=None)
        fields.update(extra)
        d = DataBunch(**fields)
        best = None
        for _ in range(3):
            gt = pptoas.GetTOAs([d], GMODEL, quiet=True)
            t0 = time.perf_counter()
            gt.get_TOAs(quiet=True)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        out[name] = nsub / best
        out[name + "_fit_only"] = nsub / gt.fit_durations[0]
    return out


def config3_timing(dev, nsub):
    """Config 3 (BASELINE.json configs[2]) as an extra key: five-parameter scattering fits, 4096 chan x
    1024 bin, fit_flags [1,1,0,1,1] and [1,1,1,1,1], inputs resident in HBM (bounded batch)."""
    import torch
    from pulseportraiture_b200 import pplib
    from pulseportraiture_b200.engine import WidebandPlan
    nchan, nbin, nu0, bw = 4096, 1024, 600.0, 400.0
    tau_s, alpha = 50e-6, -4.0
    freqs = np.linspace(nu0 - bw / 2 + bw / (2.0 * nchan), nu0 + bw / 2 - bw / (2.0 * nchan), nchan)
    _, _, model = pplib.read_model(GMODEL, pplib.get_bin_centers(nbin), freqs, P_EXAMPLE, quiet=True)
    phi, dDM = global_draws(nsub, 5)
    data = make_device_batch(model, freqs, phi, dDM, 5, dev, nchan, nbin, nu0,
                             scatter=(tau_s / P_EXAMPLE, alpha))
    torch.cuda.synchronize()
    out = {"workload": "config 3: 4096 chan x 1024 bin x %d subints, tau = 50 us at 600 MHz, alpha = -4, "
                       "log10_tau, start tau = 0.8 x truth; evaluations = coarse (low harmonics of a channel "
                       "subset) + full passes, launches are per batch" % nsub, "unit": "TOAs/s"}
    with WidebandPlan(nchan, nbin, device=dev.index or 0) as pl:
        pl.set_model(np.ascontiguousarray(model, dtype=np.float64), freqs)
        scat = np.tile([0.8 * (tau_s / P_EXAMPLE) * (freqs.mean() / nu0) ** alpha, alpha], (nsub, 1))
        for flags in ((1, 1, 0, 1, 1), (1, 1, 1, 1, 1)):
            kw = dict(fit_flags=flags, log10_tau=True, scat_guess=scat, pinned_results=True)
            for _ in range(2):
                r = pl.fit_batch(data, P_EXAMPLE, **kw)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                r = pl.fit_batch(data, P_EXAMPLE, **kw)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / 3
            pull = (r["params"][:, 1] - dDM) / r["param_errs"][:, 1]
            st = pl.stats()
            out["flags_" + "".join(map(str, flags))] = {
                "value": nsub / dt, "ms_per_batch": 1e3 * dt, "mean_evaluations": float(r["nfeval"].mean()),
                "full_pass_launches": int(st["pass_launches"]), "coarse_launches": int(st["coarse_launches"]),
                "converged": "%d/%d" % (int((r["return_code"] == 0).sum()), nsub),
                "dDM_pull_rms": float(np.sqrt(np.mean(pull ** 2)))}
    del data
    return out


_JSON_FD = None


def emit(line):
    text = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(text.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, text)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nsub", type=int, default=10000, help="subints per GPU per step")
    ap.add_argument("--chunk", type=int, default=0, help="subints per pipeline chunk (0=auto)")
    ap.add_argument("--fft", type=int, default=0, help="FFT arithmetic: 0 auto, 32, 64")
    ap.add_argument("--tol", type=float, default=0.0)
    ap.add_argument("--max-iter", type=int, default=0)
    ap.add_argument("--e2e-nsub", type=int, default=1024)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the facade and config-3 extra keys")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--facade-nsub", type=int, default=256)
    ap.add_argument("--c3-nsub", type=int, default=512)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result arrays of the last timed step as DIR/<name>.npy (a seeded sample of "
                         "subints where the batch exceeds 60 MB; with several ranks, rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the arrays of --impl ours")
    # stdout carries exactly one JSON line: anything libraries write to fd 1 (e.g. NCCL's version
    # banner under NCCL_DEBUG=VERSION) is sent to stderr, the line goes to the saved descriptor
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
