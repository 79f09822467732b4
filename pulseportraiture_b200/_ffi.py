"""ctypes binding of the C ABI in ``include/ppb200.h`` (libppb200.so).

The shared library is built in-tree by :func:`build` (``nvcc`` for sm_100a).
There is NO CPU fallback: if the library is missing or no CUDA device is
present, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libppb200.so")
INCLUDE = os.path.join(ROOT, "include")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
              "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]

# symbols declared in include/ppb200.h (checked by the CPU test-suite)
SYMBOLS = ["pp_plan_create", "pp_plan_destroy", "pp_plan_set_stream",
           "pp_plan_set_chunk", "pp_plan_set_fft_precision", "pp_plan_set_model_steps", "pp_plan_set_coarse", "pp_plan_set_model_cutoff", "pp_set_freqs", "pp_set_model_f64",
           "pp_set_model", "pp_set_models", "pp_set_models_f64", "pp_fit_batch", "pp_fit_batch_models",
           "pp_fit_phase_shift_batch", "pp_fit_phase_shift_batch_bounds", "pp_rotate_batch", "pp_rotate_full_batch", "pp_apply_response_batch",
           "pp_align_accumulate", "pp_gen_gaussian_portrait", "pp_gen_gaussian_portrait_f64", "pp_gen_spline_portrait",
           "pp_get_noise_batch", "pp_get_noise_cut_batch", "pp_get_noise_fit_batch", "pp_measure_fp64", "pp_fit_gaussian_portraits",
           "pp_fit_gaussian_portraits_join",
           "pp_simulate_batch", "pp_pca_moments", "pp_pca_project", "pp_lowpass_rows",
           "pp_plan_enable_timing", "pp_get_stats", "pp_host_alloc",
           "pp_host_free", "pp_last_error",
           "pp_abi_version"]


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC)
                  if f.endswith((".cu", ".cuh", ".h"))) + \
        [os.path.join(INCLUDE, "ppb200.h")]


def needs_build() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into libppb200.so for sm_100a (nvcc cross-compiles
    without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.isfile(nvcc):
        nvcc = "nvcc"
    cmd = [nvcc] + NVCC_FLAGS + ["-I", INCLUDE, "-o", LIB_PATH,
                                  os.path.join(CSRC, "pp_api.cu")]
    if verbose:
        print(" ".join(cmd))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


class FitArgs(C.Structure):
    _fields_ = [
        ("data", C.c_void_p),
        ("nsub", C.c_int32),
        ("semantics", C.c_int32),
        ("P", C.c_void_p),
        ("errs", C.c_void_p),
        ("chan_mask", C.c_void_p),
        ("weights", C.c_void_p),
        ("init", C.c_void_p),
        ("DM_guess", C.c_void_p),
        ("snrs", C.c_void_p),
        ("nu_fits", C.c_void_p),
        ("nu_fit_mode", C.c_int32),
        ("nu_outs", C.c_void_p),
        ("fit_flags", C.c_uint8 * 5),
        ("log10_tau", C.c_int32),
        ("option", C.c_int32),
        ("is_toa", C.c_int32),
        ("Ns", C.c_int32),
        ("max_iter", C.c_int32),
        ("tol", C.c_double),
        ("scat_guess", C.c_void_p),
        ("data_type", C.c_int32),
        ("dat_scl", C.c_void_p),
        ("dat_offs", C.c_void_p),
        ("bounds", C.c_void_p),
    ]


class FitOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "params", "param_errs", "nu_out", "cov", "chi2", "red_chi2", "snr",
        "nfeval", "return_code", "scales", "scale_errs", "channel_snrs",
        "noise", "lag_index", "phi_guess", "chan_sums", "align_sum", "align_wsum")]


class PShiftOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "phase", "phase_err", "scale", "scale_err", "snr", "red_chi2",
        "lag_index")]


class GfitArgs(C.Structure):
    _fields_ = [
        ("nport", C.c_int32),
        ("data", C.c_void_p),
        ("errs", C.c_void_p),
        ("model_code", C.c_char_p),
        ("ngauss", C.c_int32),
        ("nu_ref", C.c_double),
        ("init", C.c_void_p),
        ("fit_flags", C.c_void_p),
        ("bounds", C.c_void_p),
        ("max_iter", C.c_int32),
        ("tol", C.c_double),
    ]


class GfitOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "params", "param_errs", "cov", "chi2", "red_chi2", "nfeval", "return_code",
        "jtr", "jtj", "model")]


class GfitJoin(C.Structure):
    _fields_ = [
        ("njoin", C.c_int32),
        ("join_chan", C.c_void_p),
        ("P", C.c_double),
    ]


class SimArgs(C.Structure):
    _fields_ = [
        ("models", C.c_void_p),
        ("freqs", C.c_void_p),
        ("nmodel", C.c_int32),
        ("model_index", C.c_void_p),
        ("nsub", C.c_int32),
        ("first_subint", C.c_int64),
        ("seed", C.c_uint64),
    ] + [(n, C.c_void_p) for n in ("phase", "DM", "P", "nu_DM", "GM", "nu_GM", "tau", "alpha", "nu_tau",
                                   "scales", "noise_std")]


class SimOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("data", "raw", "dat_scl", "dat_offs")]


class Stats(C.Structure):
    _fields_ = [("launches", C.c_int64), ("pass_launches", C.c_int64),
                ("pass_rows", C.c_int64), ("ms_spectra", C.c_double),
                ("ms_guess", C.c_double), ("ms_pass", C.c_double),
                ("ms_update", C.c_double), ("ms_total", C.c_double),
                ("chunk", C.c_int32), ("timing_enabled", C.c_int32),
                ("coarse_launches", C.c_int64), ("ms_coarse", C.c_double),
                ("x_keep_frac", C.c_double)]


_lib = None


def lib():
    """The loaded library (raises if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "pulseportraiture_b200: %s is missing.  Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` "
            "(needs nvcc).  There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int32
    L.pp_plan_create.argtypes = [i32, i32, i32, C.POINTER(vp)]
    L.pp_plan_create.restype = C.c_int
    L.pp_plan_destroy.argtypes = [vp]
    L.pp_plan_destroy.restype = None
    L.pp_plan_set_stream.argtypes = [vp, vp]
    L.pp_plan_set_stream.restype = C.c_int
    L.pp_plan_set_chunk.argtypes = [vp, i32]
    L.pp_plan_set_chunk.restype = C.c_int
    L.pp_plan_set_fft_precision.argtypes = [vp, i32]
    L.pp_plan_set_fft_precision.restype = C.c_int
    L.pp_plan_set_model_steps.argtypes = [vp, i32]
    L.pp_plan_set_model_steps.restype = C.c_int
    L.pp_plan_set_coarse.argtypes = [vp, C.c_double]
    L.pp_plan_set_coarse.restype = C.c_int
    L.pp_plan_set_model_cutoff.argtypes = [vp, C.c_double]
    L.pp_plan_set_model_cutoff.restype = C.c_int
    L.pp_set_freqs.argtypes = [vp, vp]
    L.pp_set_freqs.restype = C.c_int
    L.pp_set_model.argtypes = [vp, vp, vp]
    L.pp_set_model.restype = C.c_int
    L.pp_set_model_f64.argtypes = [vp, vp, vp]
    L.pp_set_model_f64.restype = C.c_int
    L.pp_fit_batch.argtypes = [vp, C.POINTER(FitArgs), C.POINTER(FitOut)]
    L.pp_fit_batch.restype = C.c_int
    L.pp_set_models.argtypes = [vp, i32, vp, vp]
    L.pp_set_models.restype = C.c_int
    L.pp_set_models_f64.argtypes = [vp, i32, vp, vp]
    L.pp_set_models_f64.restype = C.c_int
    L.pp_fit_batch_models.argtypes = [vp, C.POINTER(FitArgs), vp, C.POINTER(FitOut)]
    L.pp_fit_batch_models.restype = C.c_int
    L.pp_fit_phase_shift_batch.argtypes = [vp, vp, i32, vp, i32, vp, i32,
                                           C.POINTER(PShiftOut)]
    L.pp_fit_phase_shift_batch.restype = C.c_int
    L.pp_fit_phase_shift_batch_bounds.argtypes = [vp, vp, i32, vp, i32, vp, i32, C.c_double, C.c_double,
                                                  C.POINTER(PShiftOut)]
    L.pp_fit_phase_shift_batch_bounds.restype = C.c_int
    L.pp_rotate_batch.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    L.pp_rotate_batch.restype = C.c_int
    L.pp_rotate_full_batch.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    L.pp_rotate_full_batch.restype = C.c_int
    L.pp_apply_response_batch.argtypes = [vp, vp, vp, i32, vp]
    L.pp_apply_response_batch.restype = C.c_int
    L.pp_align_accumulate.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.pp_align_accumulate.restype = C.c_int
    L.pp_gen_gaussian_portrait.argtypes = [vp, C.c_char_p, vp, i32, C.c_double, C.c_double, vp]
    L.pp_gen_gaussian_portrait.restype = C.c_int
    L.pp_gen_gaussian_portrait_f64.argtypes = [vp, C.c_char_p, vp, i32, C.c_double, C.c_double, vp]
    L.pp_gen_gaussian_portrait_f64.restype = C.c_int
    L.pp_gen_spline_portrait.argtypes = [vp, vp, vp, i32, vp, i32, vp, i32, vp]
    L.pp_gen_spline_portrait.restype = C.c_int
    L.pp_get_noise_batch.argtypes = [vp, vp, i32, vp]
    L.pp_get_noise_batch.restype = C.c_int
    L.pp_get_noise_cut_batch.argtypes = [vp, vp, i32, i32, vp]
    L.pp_get_noise_cut_batch.restype = C.c_int
    L.pp_get_noise_fit_batch.argtypes = [vp, vp, i32, C.c_double, vp]
    L.pp_get_noise_fit_batch.restype = C.c_int
    L.pp_measure_fp64.argtypes = [vp, C.POINTER(C.c_double)]
    L.pp_measure_fp64.restype = C.c_int
    L.pp_fit_gaussian_portraits.argtypes = [vp, C.POINTER(GfitArgs), C.POINTER(GfitOut)]
    L.pp_fit_gaussian_portraits.restype = C.c_int
    L.pp_fit_gaussian_portraits_join.argtypes = [vp, C.POINTER(GfitArgs), C.POINTER(GfitJoin), C.POINTER(GfitOut)]
    L.pp_fit_gaussian_portraits_join.restype = C.c_int
    L.pp_simulate_batch.argtypes = [vp, C.POINTER(SimArgs), C.POINTER(SimOut)]
    L.pp_simulate_batch.restype = C.c_int
    L.pp_pca_moments.argtypes = [vp, vp, vp, i32, vp, vp]
    L.pp_pca_moments.restype = C.c_int
    L.pp_pca_project.argtypes = [vp, vp, vp, vp, vp, i32, i32, vp]
    L.pp_pca_project.restype = C.c_int
    L.pp_lowpass_rows.argtypes = [vp, vp, i32, vp, vp]
    L.pp_lowpass_rows.restype = C.c_int
    L.pp_plan_enable_timing.argtypes = [vp, i32]
    L.pp_plan_enable_timing.restype = C.c_int
    L.pp_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.pp_get_stats.restype = C.c_int
    L.pp_host_alloc.argtypes = [C.c_uint64]
    L.pp_host_alloc.restype = C.c_void_p
    L.pp_host_free.argtypes = [vp]
    L.pp_host_free.restype = None
    L.pp_last_error.argtypes = []
    L.pp_last_error.restype = C.c_char_p
    L.pp_abi_version.argtypes = []
    L.pp_abi_version.restype = C.c_int
    _lib = L
    return L


class PPError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().pp_last_error().decode("utf-8", "replace")
        raise PPError("%s failed (%d): %s" % (what, rc, msg))
