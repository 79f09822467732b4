"""Reference-compatible ``pptoas.GetTOAs`` (pptoas.py:75-743) re-plumbed to
batch: every archive's subints go to the GPU in one ``pp_fit_batch`` call.

PSRCHIVE is not a dependency: an "archive" is the ``DataBunch`` that
``pplib.load_data`` would return (field list pplib.py:2803-2813), given either
directly or as an ``.npz`` file holding those fields (``save_databunch`` /
``load_data`` below).  Epochs are two-part MJDs (:class:`MJD`).
"""
from __future__ import annotations

import sys
import time

import numpy as np

from . import pplib
from .pplib import DataBunch, read_model, gen_gaussian_portrait, scattering_alpha  # noqa: F401
from .pplib import get_plan, _f32, _dev, _mdl
from .engine import model_bytes

# device memory GetTOAs.get_TOAs lets one archive's models take at once (pp_set_models); more models are set and
# fit in several rounds
_MODEL_BUDGET_BYTES = 4 << 30

max_nfile = 999                                  # pptoas.py:18-23
rm_baseline = bool(pplib.F0_fact)                # pptoas.py:25-29


class MJD(object):
    """Two-part MJD (integer day + fraction), the part of psrchive.MJD that
    get_TOAs and write_TOAs use (in_days, intday, fracday, +)."""

    def __init__(self, day=0, frac=0.0):
        if frac == 0.0 and not float(day).is_integer():
            frac, day = float(day) - np.floor(day), int(np.floor(day))
        d = int(day) + int(np.floor(frac))
        self._day, self._frac = d, float(frac - np.floor(frac))

    def intday(self):
        return self._day

    def fracday(self):
        return self._frac

    def in_days(self):
        return self._day + self._frac

    def __add__(self, other):
        if not isinstance(other, MJD):
            other = MJD(0, float(other))
        return MJD(self._day + other._day, self._frac + other._frac)

    def __repr__(self):
        return "MJD(%d + %.15f)" % (self._day, self._frac)


class TOA:
    """TOA attributes bundled together (pptoas.py:31-73)."""

    def __init__(self, archive, frequency, MJD, TOA_error, telescope,
                 telescope_code, DM=None, DM_error=None, flags={}):
        self.archive = archive
        self.frequency = frequency
        self.MJD = MJD
        self.TOA_error = TOA_error
        self.telescope = telescope
        self.telescope_code = telescope_code
        self.DM = DM
        self.DM_error = DM_error
        self.flags = flags
        for flag in flags.keys():
            setattr(self, flag, flags[flag])

    def write_TOA(self, inf_is_zero=True, outfile=None):
        """Print / append this TOA as a loosely IPTA-formatted line (pptoas.py:65-73)."""
        pplib.write_TOAs(self, inf_is_zero=inf_is_zero, outfile=outfile, append=True)


# optional: the subints as the archive stores them (PSRFITS DATA column, pol 0): int16
# [nsub, nchan, nbin] with DAT_SCL / DAT_OFFS [nsub, nchan]; get_TOAs hands them to the device as they are
_RAW_FIELDS = ["raw_subints", "dat_scl", "dat_offs"]
_DB_FIELDS = ["backend", "backend_delay", "bw", "doppler_factors", "DM", "dmc",
              "epochs", "filename", "freqs", "frontend", "integration_length",
              "masks", "nbin", "nchan", "noise_stds", "npol", "nsub", "nu0",
              "ok_ichans", "ok_isubs", "parallactic_angles", "phases", "Ps",
              "SNRs", "source", "state", "subints", "subtimes", "telescope",
              "telescope_code", "weights",
              # optional products of load_data(flux_prof=True / return_arch) that callers test for
              "flux_prof", "prof", "prof_noise", "prof_SNR"]


def save_databunch(path, data):
    """Write the load_data field contract (pplib.py:2803-2813) to ``.npz``."""
    out = {}
    for k in _DB_FIELDS:
        v = data[k]
        if v is None:
            continue
        if k == "epochs":
            out["epochs_day"] = np.array([e.intday() for e in v])
            out["epochs_frac"] = np.array([e.fracday() for e in v])
        elif k == "ok_ichans":
            m = np.zeros((data["nsub"], data["nchan"]), dtype=np.uint8)
            for i, idx in enumerate(v):
                m[i, np.asarray(idx, dtype=int)] = 1
            out["ok_mask"] = m
        else:
            out[k] = np.asarray(v)
    for k in _RAW_FIELDS:
        if data.get(k) is not None:
            out[k] = np.asarray(data[k])
    np.savez(path, **out)


def quantize_subints(subints):
    """int16 samples + DAT_SCL / DAT_OFFS per (subint, channel) for float subints [nsub, nchan, nbin],
    and the float32 portrait a PSRFITS reader decodes from them (raw * scl + offs in float32)."""
    x = np.asarray(subints, dtype=np.float64)
    lo, hi = x.min(axis=-1), x.max(axis=-1)
    offs = (0.5 * (hi + lo)).astype(np.float32)
    scl = np.where(hi > lo, (hi - lo) / 65000.0, 1.0).astype(np.float32)
    raw = np.clip(np.rint((x - offs[..., None]) / scl[..., None]), -32768, 32767).astype(np.int16)
    decoded = raw.astype(np.float32) * scl[..., None] + offs[..., None]
    return raw, scl, offs, decoded


def load_data(filename, **kwargs):
    """PSRCHIVE-free stand-in for pplib.load_data (pplib.py:2650-2814): reads
    the same fields from an ``.npz`` written by :func:`save_databunch`."""
    z = np.load(filename, allow_pickle=False)
    d = {}
    for k in z.files:
        v = z[k]
        d[k] = v.item() if v.shape == () else v
    d["epochs"] = [MJD(int(a), float(b)) for a, b in zip(d.pop("epochs_day"), d.pop("epochs_frac"))]
    m = d.pop("ok_mask")
    d["ok_ichans"] = [np.where(row)[0] for row in m]
    d["arch"] = None
    for k in _DB_FIELDS + _RAW_FIELDS:
        d.setdefault(k, None)
    d["filename"] = str(filename)
    for k in ("backend", "frontend", "source", "state", "telescope", "telescope_code"):
        d[k] = None if d[k] is None else str(d[k])
    return DataBunch(**d)


def _freq_tables(freqs):
    """Distinct rows of a [nsub, nchan] frequency array and the row each subint uses."""
    freqs = np.asarray(freqs, dtype=np.float64)
    if freqs.ndim == 2 and len(freqs) and (freqs == freqs[0]).all():   # the usual archive: one table (no sort)
        return freqs[:1].copy(), np.zeros(len(freqs), dtype=int)
    tables, table_of = np.unique(freqs, axis=0, return_inverse=True)
    return tables, np.asarray(table_of).reshape(-1)


def weighted_mean(data, errs=1.0):
    """pplib.py:686-705."""
    data = np.asarray(data, dtype=np.float64)
    errs = np.ones(len(data)) * errs if np.isscalar(errs) else np.asarray(errs, dtype=np.float64)
    iis = np.where(errs > 0.0)[0]
    mean, sum_weights = np.average(data[iis], weights=errs[iis] ** -2.0, returned=True)
    return mean, sum_weights ** -0.5


def restore_dispersion(d):
    """What ``load_data(..., dededisperse=True)`` returns for an archive stored dedispersed
    (dmc = 1; pptoas.py:256-265): the dispersive delays of the stored DM are put back, about the
    centre frequency as ``arch.dededisperse()`` does, on the device (pplib.rotate_data)."""
    out = DataBunch(**d)
    out.subints = pplib.rotate_data(np.asarray(d.subints, dtype=np.float64), 0.0, -float(d.DM),
                                    np.asarray(d.Ps, dtype=np.float64), np.asarray(d.freqs, dtype=np.float64),
                                    float(d.nu0))
    for k in _RAW_FIELDS:                        # the stored samples no longer describe the subints
        out[k] = None
    out.dmc = 0
    return out


def tscrunch_databunch(d):
    """PSRCHIVE-free stand-in for ``load_data(..., tscrunch=True)`` (pplib.py:2690): the good
    subints are averaged per channel with their weights (what ``arch.tscrunch()`` does for subints
    folded with one ephemeris), the epoch and period are the duration-weighted means, the channel
    noise levels are re-measured from the averaged profiles (get_noise on the device) and the
    per-channel S/N add in quadrature."""
    ok = np.asarray(d.ok_isubs, dtype=int)
    if not len(ok):
        return d
    sub = np.asarray(d.subints, dtype=np.float64)[ok]            # [nok, npol, nchan, nbin]
    w = np.asarray(d.weights, dtype=np.float64)[ok]              # [nok, nchan]
    wsum = w.sum(axis=0)
    avg = (sub * w[:, None, :, None]).sum(axis=0) / np.where(wsum > 0, wsum, 1.0)[None, :, None]
    npol, nchan, nbin = avg.shape
    tw = np.asarray(d.subtimes, dtype=np.float64)[ok]
    tw = tw / tw.sum() if tw.sum() > 0 else np.full(len(ok), 1.0 / len(ok))
    days = np.array([d.epochs[i].intday() for i in ok], dtype=np.float64)
    fracs = np.array([d.epochs[i].fracday() for i in ok], dtype=np.float64)
    day0 = int(days.min())
    epoch = MJD(day0, float(np.sum(tw * ((days - day0) + fracs))))
    noise = pplib.get_plan(nchan, nbin).get_noise_batch(pplib._f32(avg))     # [npol, nchan]
    snrs = np.sqrt((np.asarray(d.SNRs, dtype=np.float64)[ok] ** 2).sum(axis=0))
    okc = np.where(wsum > 0)[0]
    out = DataBunch(**d)
    out.update(subints=avg[None], weights=wsum[None], noise_stds=noise[None], SNRs=snrs[None],
               masks=None, nsub=1, ok_isubs=np.array([0]), ok_ichans=[okc], epochs=[epoch],
               Ps=np.array([float(np.sum(tw * np.asarray(d.Ps, dtype=np.float64)[ok]))]),
               freqs=np.asarray(d.freqs, dtype=np.float64)[ok][:1],
               doppler_factors=np.array([float(np.sum(tw * np.asarray(d.doppler_factors)[ok]))]),
               parallactic_angles=np.array([float(np.sum(tw * np.asarray(d.parallactic_angles)[ok]))]),
               subtimes=np.array([float(np.asarray(d.subtimes, dtype=np.float64)[ok].sum())]))
    for k in _RAW_FIELDS:
        out[k] = None
    return out


class GetTOAs:
    """Measure TOAs and DMs from wideband data (pptoas.py:75-743)."""

    def __init__(self, datafiles, modelfile, quiet=False):
        if isinstance(datafiles, (list, tuple)):
            self.datafiles = list(datafiles)
        elif isinstance(datafiles, str) and not datafiles.endswith(".npz"):
            self.datafiles = [line.strip() for line in open(datafiles, "r").readlines()
                              if line.strip()]             # metafile (pptoas.py:93-95)
        else:
            self.datafiles = [datafiles]
        if len(self.datafiles) > max_nfile:
            print("Too many archives.  See/change max_nfile(=%d) in pptoas.py." % max_nfile)
            sys.exit()
        self.is_FITS_model = False
        self.modelfile = modelfile
        for name in ("obs", "doppler_fs", "nu0s", "nu_fits", "nu_refs", "ok_idatafiles",
                     "ok_isubs", "epochs", "MJDs", "Ps", "phis", "phi_errs", "TOAs",
                     "TOA_errs", "DM0s", "DMs", "DM_errs", "DeltaDM_means", "DeltaDM_errs",
                     "GMs", "GM_errs", "taus", "tau_errs", "alphas", "alpha_errs", "scales",
                     "scale_errs", "snrs", "channel_snrs", "profile_fluxes",
                     "profile_flux_errs", "fluxes", "flux_errs", "flux_freqs", "red_chi2s",
                     "channel_red_chi2s", "covariances", "nfevals", "rcs", "fit_durations",
                     "order", "TOA_list", "zap_channels"):
            setattr(self, name, [])                         # pptoas.py:102-143
        self.instrumental_response_dict = self.ird = {'DM': 0.0, 'wids': [], 'irf_types': []}
        self.quiet = quiet

    def _model_depends_on_P(self, fit_scat, add_instrumental_response):
        """True when the model portrait differs from subint to subint through the period: a .gmodel
        with TAU != 0 (seconds -> rotations, pplib.py:2944-2945) or a DM-smearing instrumental
        response (pptoaslib.py:175).  The reference rebuilds the model per subint (pptoas.py:356-394)."""
        if add_instrumental_response and self.ird['DM']:
            return True
        if isinstance(self.modelfile, np.ndarray) or pplib.is_spline_model(self.modelfile) or fit_scat:
            return False
        return read_model(self.modelfile, quiet=True)[4][1] != 0.0

    def _model_for(self, phases, freqs_row, P, fit_scat=False, add_instrumental_response=False, chan_bw=None):
        model = self._bare_model_for(phases, freqs_row, P, fit_scat)
        if add_instrumental_response and (self.ird['DM'] or len(self.ird['wids'])):   # pptoas.py:388-394
            from .pptoaslib import add_instrumental_response as _air
            model = _air(model, freqs_row, self.ird['DM'], P, self.ird['wids'], self.ird['irf_types'],
                         chan_bw=chan_bw)
        return model

    def _bare_model_for(self, phases, freqs_row, P, fit_scat=False):
        if isinstance(self.modelfile, np.ndarray):
            self.model_name, self.ngauss = "array", 0
            return self.modelfile
        if pplib.is_spline_model(self.modelfile):           # pptoas.py:376-379
            self.ngauss = 0
            self.model_name, model = pplib.read_spline_model(self.modelfile, freqs_row, len(phases),
                                                             quiet=True, device=True)
            return model
        if not fit_scat:
            self.model_name, self.ngauss, model = read_model(self.modelfile, phases, freqs_row, P,
                                                             quiet=True, device=True)
            return model
        # scattering is fit: use the unscattered portrait (pptoas.py:364-375)
        (self.model_name, self.model_code, self.model_nu_ref, self.ngauss, self.gparams,
         model_fit_flags, self.alpha, model_fit_alpha) = read_model(self.modelfile, quiet=True)
        unscat_params = np.copy(self.gparams)
        unscat_params[1] = 0.0
        return pplib.gen_gaussian_portrait_device(self.model_code, unscat_params, 0.0, phases,
                                                  freqs_row, self.model_nu_ref)

    def get_TOAs(self, datafile=None, tscrunch=False, nu_refs=None, DM0=None,
                 bary=True, fit_DM=True, fit_GM=False, fit_scat=False,
                 log10_tau=True, scat_guess=None, fix_alpha=False,
                 print_phase=False, print_flux=False, print_parangle=False,
                 add_instrumental_response=False, addtnl_toa_flags={},
                 method='trust-ncg', bounds=None, nu_fits=None, show_plot=False,
                 quiet=None):
        """Measure wideband TOAs (pptoas.py:150-743).  Same keyword arguments
        as the reference; results fill the attribute lists of the instance."""
        if quiet is None:
            quiet = self.quiet
        if show_plot:
            raise NotImplementedError("show_plot needs matplotlib and is outside the hot path")
        if method not in pplib._RC_MAP:                     # pptoaslib.py:1003-1005
            print("Method '%s' is not implemented." % method)
            sys.exit()
        self.tscrunch = tscrunch
        self.add_instrumental_response = add_instrumental_response
        self.nfit = 1 + int(bool(fit_DM)) + int(bool(fit_GM)) + 2 * int(bool(fit_scat)) - \
            int(bool(fix_alpha))
        self.fit_phi, self.fit_DM, self.fit_GM = True, fit_DM, fit_GM
        self.fit_tau = self.fit_alpha = fit_scat
        if fit_scat:
            self.fit_alpha = not fix_alpha
        self.fit_flags = [int(self.fit_phi), int(self.fit_DM), int(self.fit_GM),
                          int(self.fit_tau), int(self.fit_alpha)]
        if not fit_scat:
            log10_tau = False                               # pptoas.py:229-230
        self.log10_tau = log10_tau
        self.scat_guess, self.DM0, self.bary = scat_guess, DM0, bary
        nu_ref_tuple, nu_fit_tuple = nu_refs, nu_fits
        start = time.time()
        datafiles = self.datafiles if datafile is None else [datafile]
        for iarch, datafile in enumerate(datafiles):
            try:
                data = datafile if isinstance(datafile, dict) else load_data(datafile)
            except (RuntimeError, IOError, OSError):
                if not quiet:
                    print("Cannot load_data(%s).  Skipping it." % datafile)
                continue
            if data.get("dmc"):                             # pptoas.py:256-265
                if not quiet:
                    print("%s is dedispersed (dmc = 1).  Restoring the dispersion." % data.filename)
                data = restore_dispersion(data)
            if tscrunch:                                    # load_data(..., tscrunch=True), pptoas.py:253
                data = tscrunch_databunch(data)
            if not len(data.ok_isubs):
                if not quiet:
                    print("No subints to fit for %s.  Skipping it." % data.filename)
                continue
            self.ok_idatafiles.append(iarch)
            self._archives = getattr(self, "_archives", {})
            self._archives[iarch] = data
            d = data
            nsub, nchan, nbin = int(d.nsub), int(d.nchan), int(d.nbin)
            ok_isubs = np.asarray(d.ok_isubs, dtype=int)
            source = d.source if d.source is not None else "noname"  # noqa: F841
            obs = DataBunch(telescope=d.telescope, backend=d.backend, frontend=d.frontend)
            freqs = np.asarray(d.freqs, dtype=np.float64)
            Ps = np.asarray(d.Ps, dtype=np.float64)
            DM_stored = float(d.DM)
            DM0_arch = DM_stored if self.DM0 is None else self.DM0
            MJDs = np.array([e.in_days() for e in d.epochs], dtype=np.double)
            # Per-subint frequency tables (freqs = data.freqs[isub], pptoas.py:346): the reference
            # rebuilds the model for every subint (pptoas.py:356-379); here subints that share a
            # table share one model and one batch.
            tables, table_of = _freq_tables(freqs)
            if self._model_depends_on_P(fit_scat, add_instrumental_response):
                # one model per (frequency table, period): subints with their own period get their own
                # model and batch, as in the reference's per-subint loop
                # (the smearing width uses the spacing of the subint's first two usable channels: the
                # reference evaluates instrumental_response_port_FT on freqsx, pptoas.py:390-392)
                def cbw(i):
                    okc_ = np.asarray(d.ok_ichans[i], dtype=int)
                    if not (add_instrumental_response and self.ird['DM']) or len(okc_) < 2:
                        return 0.0
                    return float(abs(freqs[i, okc_[1]] - freqs[i, okc_[0]]))
                keys = [(int(table_of[i]), float(Ps[i]), cbw(i) if i in set(ok_isubs) else 0.0) for i in range(nsub)]
                uniq = sorted(set(keys[i] for i in ok_isubs))
                table_of = np.array([uniq.index(k) if k in uniq else -1 for k in keys])
                tables = np.array([tables[k[0]] for k in uniq])
                models = {t: self._model_for(d.phases, tables[t], uniq[t][1], fit_scat, add_instrumental_response,
                                             chan_bw=uniq[t][2] or None)
                          for t in range(len(uniq))}
            else:
                models = {t: self._model_for(d.phases, tables[t], Ps[ok_isubs[table_of[ok_isubs] == t][0]],
                                             fit_scat, add_instrumental_response)
                          for t in np.unique(table_of[ok_isubs])}
            model = models[table_of[ok_isubs[0]]]

            mask = np.zeros((nsub, nchan), dtype=np.uint8)
            for isub in ok_isubs:
                mask[isub, np.asarray(d.ok_ichans[isub], dtype=int)] = 1
            nok = mask.sum(axis=1)
            subints = _dev(np.asarray(d.subints)[:, 0])      # float64 goes to the device as it is
            errs = np.ascontiguousarray(np.asarray(d.noise_stds)[:, 0], dtype=np.float64)
            snrs = np.ascontiguousarray(np.asarray(d.SNRs)[:, 0], dtype=np.float64)
            weights = np.ascontiguousarray(d.weights, dtype=np.float64)
            if nu_fit_tuple is None and fit_scat:
                # the scattering start value needs nu_fit_tau on the host (pptoas.py:402, 431-441)
                nu_fits_in = np.zeros((nsub, 3))
                nu_fits_in[ok_isubs, :] = pplib.guess_fit_freq_batch(freqs[ok_isubs], snrs[ok_isubs],
                                                                    mask[ok_isubs])[:, None]
                empty = nu_fits_in[:, 0] == 0
                nu_fits_in[empty] = freqs[empty].mean(axis=1)[:, None]
                mode = 0
            elif nu_fit_tuple is None:
                nu_fits_in, mode = None, 1                 # guess_fit_freq, pptoas.py:402
            else:
                nu_fits_in = np.tile([nu_fit_tuple[0], nu_fit_tuple[0], nu_fit_tuple[-1]],
                                     (nsub, 1)).astype(np.float64)
                mode = 0
            nu_outs_in = None
            if nu_ref_tuple is not None:
                nu_outs_in = np.full((nsub, 3), np.nan)
                if nu_ref_tuple[0]:
                    nu_outs_in[:, 0] = nu_outs_in[:, 1] = nu_ref_tuple[0]
                if nu_ref_tuple[-1]:
                    nu_outs_in[:, 2] = nu_ref_tuple[-1]
                    if bary:
                        nu_outs_in[:, 2] /= np.asarray(d.doppler_factors)
            scat_in = None
            if fit_scat:                                    # pptoas.py:427-441
                scat_in = np.zeros((nsub, 2))
                for isub in ok_isubs:
                    if self.scat_guess is not None:
                        tau_guess_s, tau_guess_ref, alpha_guess = self.scat_guess
                        tau_guess = (tau_guess_s / Ps[isub]) * \
                            (nu_fits_in[isub, 2] / tau_guess_ref) ** alpha_guess
                    else:
                        alpha_guess = getattr(self, "alpha", scattering_alpha)
                        if hasattr(self, "gparams"):
                            tau_guess = (self.gparams[1] / Ps[isub]) * \
                                (nu_fits_in[isub, 2] / self.model_nu_ref) ** alpha_guess
                        else:
                            tau_guess = 0.0
                    scat_in[isub] = [tau_guess, alpha_guess]
            if method == 'TNC':                             # bounds act with TNC only (pptoaslib.py:1008)
                if bounds is None:                          # pptoas.py:461-469
                    tau_bounds = (np.log10((10 * nbin) ** -1), None) if self.log10_tau else (0.0, None)
                    bounds = [(None, None), (None, None), (None, None), tau_bounds, (-10.0, 10.0)]
                fit_bounds = pplib._check_bounds(bounds, 5)
            else:
                fit_bounds = None
            pl = get_plan(nchan, nbin)
            self._models = getattr(self, "_models", {})
            self._models[iarch] = np.asarray(model, dtype=np.float64)
            self._model_tables = getattr(self, "_model_tables", {})
            self._model_tables[iarch] = (table_of, {t: np.asarray(m, dtype=np.float64)
                                                    for t, m in models.items()})

            # subints with a single usable channel are fit for phase only
            # (pptoas.py:475-478); two channels drop GM (479-483)
            # Every model of the archive goes to the plan in one pp_set_models call (several when they exceed
            # _MODEL_BUDGET_BYTES of device memory) and every flags group is one fit_batch: each subint is fit
            # against its own model (pp_fit_batch_models), as the reference's per-subint loop does.
            flags_by_sub = {}
            for isub in ok_isubs:
                if nok[isub] == 1:
                    flags = (1, 0, 0, 0, 0)
                elif nok[isub] == 2 and self.fit_DM and self.fit_GM:
                    flags = tuple(self.fit_flags[:2] + [0] + self.fit_flags[3:])
                else:
                    flags = tuple(self.fit_flags)
                flags_by_sub[isub] = flags
            model_ids = sorted(models)
            per_call = max(1, int(_MODEL_BUDGET_BYTES // model_bytes(nchan, nbin)))
            work = []                                  # (model ids set at once, flags, subints)
            for m0 in range(0, len(model_ids), per_call):
                mset = model_ids[m0:m0 + per_call]
                inset = set(mset)
                groups = {}
                for isub in ok_isubs:
                    if int(table_of[isub]) in inset:
                        groups.setdefault(flags_by_sub[isub], []).append(isub)
                for flags, isubs in sorted(groups.items()):
                    work.append((mset, flags, isubs))
            res, flags_of = {}, {}
            fit_start = time.time()
            mset_on = None
            for mset, flags, isubs in work:
                if mset is not mset_on:
                    ms = [_mdl(models[t]) for t in mset]
                    dt = np.float32 if all(m.dtype == np.float32 for m in ms) else np.float64
                    pl.set_models(np.stack([np.asarray(m, dtype=dt) for m in ms]),
                                  np.stack([tables[t] for t in mset]))
                    local = {t: i for i, t in enumerate(mset)}
                    mset_on = mset
                idx = np.asarray(isubs, dtype=int)
                model_index = None if len(mset) == 1 else \
                    np.array([local[int(table_of[i])] for i in isubs], dtype=np.int32)
                if len(idx) > 1 and np.all(np.diff(idx) == 1):
                    idx = slice(int(idx[0]), int(idx[-1]) + 1)      # a contiguous range: views, no gather copy
                nidx = len(isubs)
                raw_kw = {}
                if d.get("raw_subints") is not None:       # stored samples go to the device as they are
                    batch = np.ascontiguousarray(np.asarray(d.raw_subints, dtype=np.int16)[idx])
                    raw_kw = dict(dat_scl=np.ascontiguousarray(np.asarray(d.dat_scl, dtype=np.float32)[idx]),
                                  dat_offs=np.ascontiguousarray(np.asarray(d.dat_offs, dtype=np.float32)[idx]))
                else:
                    batch = np.ascontiguousarray(subints[idx])
                r = pl.fit_batch(
                    batch, Ps[idx], errs=errs[idx], **raw_kw,
                    chan_mask=mask[idx], weights=weights[idx], DM_guess=np.full(nidx, DM_stored),
                    snrs=snrs[idx], nu_fits=None if nu_fits_in is None else nu_fits_in[idx],
                    nu_fit_mode=mode, nu_outs=None if nu_outs_in is None else nu_outs_in[idx],
                    fit_flags=flags, log10_tau=self.log10_tau, option=0, is_toa=True,
                    Ns=100, semantics="full", bounds=fit_bounds,
                    scat_guess=None if scat_in is None else scat_in[idx], model_index=model_index)
                for k, v in r.items():                     # results of all groups, by subint
                    if isinstance(v, np.ndarray) and len(v) == nidx:
                        if k not in res:
                            res[k] = np.zeros((nsub,) + v.shape[1:], dtype=v.dtype)
                        res[k][idx] = v
                for isub in isubs:
                    flags_of[isub] = flags
            fit_duration = time.time() - fit_start

            phis = np.zeros(nsub); phi_errs = np.zeros(nsub)
            TOAs = np.zeros(nsub, dtype="object"); TOA_errs = np.zeros(nsub, dtype="object")
            DMs = np.zeros(nsub); DM_errs = np.zeros(nsub)
            GMs = np.zeros(nsub); GM_errs = np.zeros(nsub)
            taus = np.zeros(nsub); tau_errs = np.zeros(nsub)
            alphas = np.zeros(nsub); alpha_errs = np.zeros(nsub)
            scales = np.zeros([nsub, nchan]); scale_errs = np.zeros([nsub, nchan])
            snrs_out = np.zeros(nsub); channel_snrs = np.zeros([nsub, nchan])
            profile_fluxes = np.zeros([nsub, nchan]); profile_flux_errs = np.zeros([nsub, nchan])
            fluxes = np.zeros(nsub); flux_errs = np.zeros(nsub); flux_freqs = np.zeros(nsub)
            red_chi2s = np.zeros(nsub)
            covariances = np.zeros([nsub, self.nfit, self.nfit])
            nfevals = np.zeros(nsub, dtype="int"); rcs = np.zeros(nsub, dtype="int")
            nu_fits_arr = list(np.zeros([nsub, 3])); nu_refs_arr = list(np.zeros([nsub, 3]))
            # everything that is the same arithmetic for every subint, for all of them at once
            okm = mask.astype(bool)
            okm[np.setdiff1d(np.arange(nsub), ok_isubs)] = False
            if res:
                scales[okm] = res["scales"][okm]
                scale_errs[okm] = res["scale_errs"][okm]
                channel_snrs[okm] = res["channel_snrs"][okm]
            fmax = np.where(okm, freqs, -np.inf).max(axis=1)
            fmin = np.where(okm, freqs, np.inf).min(axis=1)
            if nu_fits_in is None:                          # pptoas.py:400-407
                nu_fit_vals = np.zeros(nsub)
                nu_fit_vals[ok_isubs] = pplib.guess_fit_freq_batch(freqs[ok_isubs], snrs[ok_isubs], mask[ok_isubs])
            doppler = np.asarray(d.doppler_factors, dtype=np.float64)
            subtimes = np.asarray(d.subtimes)
            parangles = np.asarray(d.parallactic_angles) if print_parangle else None
            tmplt = self.modelfile if isinstance(self.modelfile, str) else "array"
            fe_be = d.frontend + "_" + d.backend
            chbw = abs(d.bw) / nchan
            ifit_of = {}
            for isub in ok_isubs:
                flags = flags_of[isub]
                par, perr = res["params"][isub], res["param_errs"][isub]
                nu_out = res["nu_out"][isub]
                P = Ps[isub]
                phi, phi_err = par[0], perr[0]
                DM, DM_err = par[1], perr[1]
                GM, GM_err = par[2], perr[2]
                # TOA (pptoas.py:528-531)
                TOA_mjd = d.epochs[isub] + MJD(0, ((phi * P) + d.backend_delay) / (3600 * 24.))
                TOA_err = phi_err * P * 1e6
                # Doppler correction (pptoas.py:539-549)
                if self.bary:
                    df = doppler[isub]
                    if flags[1]:
                        DM *= df
                    if flags[2]:
                        GM *= df ** 3
                else:
                    df = 1.0
                if print_flux:                              # pptoas.py:554-577
                    okc = np.nonzero(okm[isub])[0]
                    means = np.asarray(models[table_of[isub]])[okc].mean(axis=1)
                    profile_fluxes[isub, okc] = means * scales[isub, okc]
                    profile_flux_errs[isub, okc] = abs(means) * scale_errs[isub, okc]
                    fluxes[isub], flux_errs[isub] = weighted_mean(profile_fluxes[isub, okc],
                                                                 profile_flux_errs[isub, okc])
                    flux_freqs[isub], _ = weighted_mean(freqs[isub, okc], profile_flux_errs[isub, okc])
                nu_refs_arr[isub] = list(nu_out)
                if nu_fits_in is not None:                  # pptoas.py:400-407
                    nu_fits_arr[isub] = list(nu_fits_in[isub])
                else:
                    nu_fits_arr[isub] = [nu_fit_vals[isub]] * 3
                phis[isub], phi_errs[isub] = phi, phi_err
                TOAs[isub], TOA_errs[isub] = TOA_mjd, TOA_err
                DMs[isub], DM_errs[isub] = DM, DM_err
                GMs[isub], GM_errs[isub] = GM, GM_err
                if flags not in ifit_of:
                    ifit_of[flags] = np.where(flags)[0]
                ifit = ifit_of[flags]
                cm = res["cov"][isub][np.ix_(ifit, ifit)]
                if cm.shape == covariances[isub].shape:
                    covariances[isub] = cm
                else:                                       # pptoas.py:596-600
                    for ii, a_ in enumerate(ifit):
                        for jj, b_ in enumerate(ifit):
                            if a_ < self.nfit and b_ < self.nfit:
                                covariances[isub][a_, b_] = cm[ii, jj]
                snr, gof = res["snr"][isub], res["red_chi2"][isub]
                toa_flags = {}                              # pptoas.py:604-651
                DM_out, DM_err_out = (DM, DM_err) if flags[1] else (None, None)
                if flags[2]:
                    toa_flags['gm'], toa_flags['gm_err'] = GM, GM_err
                if flags[3]:                                # pptoas.py:611-624
                    tau_r, tau_e = par[3], perr[3]
                    if self.log10_tau:
                        toa_flags['scat_time'] = 10 ** tau_r * P / df * 1e6
                        toa_flags['log10_scat_time'] = tau_r + np.log10(P / df)
                        toa_flags['log10_scat_time_err'] = tau_e
                    else:
                        toa_flags['scat_time'] = tau_r * P / df * 1e6
                        toa_flags['scat_time_err'] = tau_e * P / df * 1e6
                    toa_flags['scat_ref_freq'] = nu_out[2] * df
                    toa_flags['scat_ind'] = par[4]
                if flags[4]:
                    toa_flags['scat_ind_err'] = perr[4]
                toa_flags['be'] = d.backend
                toa_flags['fe'] = d.frontend
                toa_flags['f'] = fe_be
                toa_flags['nbin'] = nbin
                toa_flags['nch'] = nchan
                toa_flags['nchx'] = int(nok[isub])
                toa_flags['bw'] = fmax[isub] - fmin[isub]
                toa_flags['chbw'] = chbw
                toa_flags['subint'] = int(isub)
                toa_flags['tobs'] = subtimes[isub]
                toa_flags['fratio'] = fmax[isub] / fmin[isub]
                toa_flags['tmplt'] = tmplt
                toa_flags['snr'] = snr
                if nu_ref_tuple is not None and nu_ref_tuple[0] is not None and np.all(flags[:2]):
                    toa_flags['phi_DM_cov'] = cm[0, 1]
                toa_flags['gof'] = gof
                if print_phase:
                    toa_flags['phs'], toa_flags['phs_err'] = phi, phi_err
                if print_flux:
                    toa_flags['flux'] = fluxes[isub]
                    toa_flags['flux_err'] = flux_errs[isub]
                    toa_flags['flux_ref_freq'] = flux_freqs[isub]
                if print_parangle:
                    toa_flags['par_angle'] = parangles[isub]
                for k, v in addtnl_toa_flags.items():
                    toa_flags[k] = v
                self.TOA_list.append(TOA(d.filename, nu_out[0], TOA_mjd, TOA_err,
                                         d.telescope, d.telescope_code, DM_out, DM_err_out,
                                         toa_flags))
            oks = np.asarray(ok_isubs if res else [], dtype=int)
            taus[oks], tau_errs[oks] = res["params"][oks, 3], res["param_errs"][oks, 3]
            alphas[oks], alpha_errs[oks] = res["params"][oks, 4], res["param_errs"][oks, 4]
            nfevals[oks] = res["nfeval"][oks]
            rcs[oks] = [pplib.scipy_return_code(c, method) for c in res["return_code"][oks]]   # pptoaslib.py:1017
            snrs_out[oks] = res["snr"][oks]
            red_chi2s[oks] = res["red_chi2"][oks]
            # per-archive Delta-DM mean (pptoas.py:665-682)
            DeltaDMs = DMs - DM0_arch
            if np.all(DM_errs[ok_isubs]):
                DM_weights = DM_errs[ok_isubs] ** -2
            else:
                DM_weights = np.ones(len(ok_isubs))
            DeltaDM_mean, DeltaDM_var = np.average(DeltaDMs[ok_isubs], weights=DM_weights,
                                                   returned=True)
            DeltaDM_var = DeltaDM_var ** -1
            if len(ok_isubs) > 1:
                DeltaDM_var *= np.sum(((DeltaDMs[ok_isubs] - DeltaDM_mean) ** 2) * DM_weights) / \
                    (len(ok_isubs) - 1)
            DeltaDM_err = DeltaDM_var ** 0.5
            self.order.append(d.filename); self.obs.append(obs)
            self.doppler_fs.append(d.doppler_factors); self.nu0s.append(d.nu0)
            self.nu_fits.append(nu_fits_arr); self.nu_refs.append(nu_refs_arr)
            self.ok_isubs.append(ok_isubs); self.epochs.append(d.epochs)
            self.MJDs.append(MJDs); self.Ps.append(Ps)
            self.phis.append(phis); self.phi_errs.append(phi_errs)
            self.TOAs.append(TOAs); self.TOA_errs.append(TOA_errs)
            self.DM0s.append(DM0_arch); self.DMs.append(DMs); self.DM_errs.append(DM_errs)
            self.DeltaDM_means.append(DeltaDM_mean); self.DeltaDM_errs.append(DeltaDM_err)
            self.GMs.append(GMs); self.GM_errs.append(GM_errs)
            self.taus.append(taus); self.tau_errs.append(tau_errs)
            self.alphas.append(alphas); self.alpha_errs.append(alpha_errs)
            self.scales.append(scales); self.scale_errs.append(scale_errs)
            self.snrs.append(snrs_out); self.channel_snrs.append(channel_snrs)
            self.profile_fluxes.append(profile_fluxes)
            self.profile_flux_errs.append(profile_flux_errs)
            self.fluxes.append(fluxes); self.flux_errs.append(flux_errs)
            self.flux_freqs.append(flux_freqs)
            self.covariances.append(covariances); self.red_chi2s.append(red_chi2s)
            self.nfevals.append(nfevals); self.rcs.append(rcs)
            self.fit_durations.append(fit_duration)
            if not quiet:
                print("--------------------------")
                print(d.filename)
                print("~%.4f sec/TOA" % (fit_duration / len(ok_isubs)))
                print("Med. TOA error is %.3f us" % (np.median(phi_errs[ok_isubs]) * Ps.mean() * 1e6))
        self._models = getattr(self, "_models", {})
        tot_duration = time.time() - start
        if not quiet and len(self.ok_isubs):
            print("--------------------------")
            print("Total time: %.2f sec, ~%.4f sec/TOA" % (
                tot_duration, tot_duration / (np.array(list(map(len, self.ok_isubs))).sum())))

    def get_narrowband_TOAs(self, datafile=None, tscrunch=False, fit_scat=False, log10_tau=True,
                            scat_guess=None, print_phase=False, print_flux=False,
                            print_parangle=False, add_instrumental_response=False,
                            addtnl_toa_flags={}, method='trust-ncg', bounds=None, show_plot=False,
                            quiet=None):
        """Measure one TOA per (subint, channel) with the 1-D FFTFIT (pptoas.py:745-1132): every
        usable channel profile against its model channel, ``fit_phase_shift(prof, model_prof, err,
        Ns=100)`` -- all profiles of an archive in one ``pp_fit_phase_shift_batch`` call.  As in the
        reference the scattering fit is not active in this method (tau = 0)."""
        if quiet is None:
            quiet = self.quiet
        if show_plot:
            raise NotImplementedError("show_plot needs matplotlib and is outside the hot path")
        self.fit_flags = [1, 0]
        self.log10_tau = False
        start = time.time()
        datafiles = self.datafiles if datafile is None else [datafile]
        for iarch, datafile in enumerate(datafiles):
            try:
                d = datafile if isinstance(datafile, dict) else load_data(datafile)
            except (RuntimeError, IOError, OSError):
                if not quiet:
                    print("Cannot load_data(%s).  Skipping it." % datafile)
                continue
            if d.get("dmc"):                                # pptoas.py:817-826
                d = restore_dispersion(d)
            if tscrunch:
                d = tscrunch_databunch(d)
            if not len(d.ok_isubs):
                continue
            self.ok_idatafiles.append(iarch)
            nsub, nchan, nbin = int(d.nsub), int(d.nchan), int(d.nbin)
            ok_isubs = np.asarray(d.ok_isubs, dtype=int)
            freqs = np.asarray(d.freqs, dtype=np.float64)
            Ps = np.asarray(d.Ps, dtype=np.float64)
            tables, table_of = _freq_tables(freqs)          # freqs = data.freqs[isub], pptoas.py:927
            models = {t: self._model_for(d.phases, tables[t], Ps[ok_isubs[table_of[ok_isubs] == t][0]], False,
                                         add_instrumental_response)
                      for t in np.unique(table_of[ok_isubs])}
            model_of = [models[t] for t in table_of]
            pl = get_plan(nchan, nbin)
            fit_start = time.time()
            profs = _f32(np.asarray(d.subints)[ok_isubs, 0]).reshape(len(ok_isubs) * nchan, nbin)
            noise = np.ascontiguousarray(np.asarray(d.noise_stds)[ok_isubs, 0], dtype=np.float64)
            okmask = np.zeros((len(ok_isubs), nchan), dtype=bool)
            for i, isub in enumerate(ok_isubs):
                okmask[i, np.asarray(d.ok_ichans[isub], dtype=int)] = True
            okmask &= noise > 0
            if len(models) == 1:
                mstack = _f32(model_of[ok_isubs[0]])
            else:                                           # one model row per profile
                mstack = _f32(np.concatenate([model_of[isub] for isub in ok_isubs]))
            r = pl.fit_phase_shift_batch(profs, mstack, noise=np.where(okmask, noise, 1.0).ravel(),
                                         Ns=100)
            fit_duration = time.time() - fit_start
            shape = (nsub, nchan)
            phis, phi_errs = np.zeros(shape), np.zeros(shape)
            TOAs, TOA_errs = np.zeros(shape, dtype="object"), np.zeros(shape, dtype="object")
            taus, tau_errs = np.zeros(shape), np.zeros(shape)
            scales, scale_errs = np.zeros(shape), np.zeros(shape)
            channel_snrs, channel_red_chi2s = np.zeros(shape), np.zeros(shape)
            profile_fluxes, profile_flux_errs = np.zeros(shape), np.zeros(shape)
            MJDs = np.array([e.in_days() for e in d.epochs], dtype=np.double)
            obs = DataBunch(telescope=d.telescope, backend=d.backend, frontend=d.frontend)
            get = lambda k: r[k].reshape(len(ok_isubs), nchan)  # noqa: E731
            for i, isub in enumerate(ok_isubs):
                P = Ps[isub]
                for ichan in np.where(okmask[i])[0]:
                    phase, phase_err = get("phase")[i, ichan], get("phase_err")[i, ichan]
                    toa = d.epochs[isub] + MJD(0, ((phase * P) + d.backend_delay) / (3600 * 24.))
                    toa_err = phase_err * P * 1e6                                  # [us]
                    phis[isub, ichan], phi_errs[isub, ichan] = phase, phase_err
                    TOAs[isub, ichan], TOA_errs[isub, ichan] = toa, toa_err
                    scales[isub, ichan] = get("scale")[i, ichan]
                    scale_errs[isub, ichan] = get("scale_err")[i, ichan]
                    channel_snrs[isub, ichan] = get("snr")[i, ichan]
                    channel_red_chi2s[isub, ichan] = get("red_chi2")[i, ichan]
                    if print_flux:
                        mm = model_of[isub][ichan].mean()
                        profile_fluxes[isub, ichan] = mm * scales[isub, ichan]
                        profile_flux_errs[isub, ichan] = abs(mm) * scale_errs[isub, ichan]
                    toa_flags = {'be': d.backend, 'fe': d.frontend, 'f': "%s_%s" % (d.frontend, d.backend),
                                 'nbin': nbin, 'bw': abs(d.bw) / nchan, 'subint': int(isub), 'chan': int(ichan),
                                 'tobs': d.subtimes[isub],
                                 'tmplt': self.modelfile if isinstance(self.modelfile, str) else "array",
                                 'snr': channel_snrs[isub, ichan], 'gof': channel_red_chi2s[isub, ichan]}
                    if print_phase:
                        toa_flags['phs'], toa_flags['phs_err'] = phase, phase_err
                    if print_flux:
                        toa_flags['flux'] = profile_fluxes[isub, ichan]
                        toa_flags['flux_err'] = profile_flux_errs[isub, ichan]
                    if print_parangle:
                        toa_flags['par_angle'] = d.parallactic_angles[isub]
                    toa_flags.update(addtnl_toa_flags)
                    self.TOA_list.append(TOA(d.filename, freqs[isub, ichan], toa, toa_err, d.telescope,
                                             d.telescope_code, None, None, toa_flags))
            for name, val in (("order", d.filename), ("obs", obs), ("doppler_fs", d.doppler_factors),
                              ("ok_isubs", ok_isubs), ("epochs", d.epochs), ("MJDs", MJDs), ("Ps", Ps),
                              ("phis", phis), ("phi_errs", phi_errs), ("TOAs", TOAs), ("TOA_errs", TOA_errs),
                              ("taus", taus), ("tau_errs", tau_errs), ("scales", scales),
                              ("scale_errs", scale_errs), ("channel_snrs", channel_snrs),
                              ("profile_fluxes", profile_fluxes), ("profile_flux_errs", profile_flux_errs),
                              ("channel_red_chi2s", channel_red_chi2s), ("fit_durations", fit_duration)):
                if not hasattr(self, name):
                    setattr(self, name, [])
                getattr(self, name).append(val)
            if not quiet:
                print("--------------------------")
                print(d.filename)
                print("~%.6f sec/TOA" % (fit_duration / max(1, int(okmask.sum()))))
                print("Med. TOA error is %.3f us" % (np.median(phi_errs[phi_errs > 0]) * Ps.mean() * 1e6))
        if not quiet and len(self.ok_idatafiles):
            tot = time.time() - start
            print("--------------------------")
            print("Total time: %.2f sec, ~%.6f sec/TOA" % (tot, tot / max(1, len(self.TOA_list))))

    def get_channels_to_zap(self, SNR_threshold=8.0, rchi2_threshold=1.3, iterate=True,
                            show=False):
        """Flag channels by per-channel reduced chi-squared and S/N (pptoas.py:1208-1285).
        NB: get_TOAs(...) needs to have been called first.  The data are rotated onto the
        model with the fitted parameters on the device (show_fit, pptoas.py:1398-1399);
        the per-channel residual sums are host arithmetic."""
        if show:
            raise NotImplementedError("plots need matplotlib")
        from .pplib import scattering_portrait_FT, scattering_times
        for k, iarch in enumerate(self.ok_idatafiles):
            d = self._archives[iarch]
            table_of, models = self._model_tables[iarch]
            nchan, nbin = int(d.nchan), int(d.nbin)
            pl = get_plan(nchan, nbin)
            freqs = np.asarray(d.freqs, dtype=np.float64)
            ok_isubs = np.asarray(self.ok_isubs[k], dtype=int)
            phi, DM, GM = self.phis[k][ok_isubs], self.DMs[k][ok_isubs].copy(), self.GMs[k][ok_isubs].copy()
            if self.bary:                                   # back to the fitted values (1353-1355)
                df = np.asarray(self.doppler_fs[k])[ok_isubs]
                DM /= df
                GM /= df ** 3
            nus = np.array([self.nu_refs[k][i] for i in ok_isubs], dtype=np.float64)
            rot = np.empty((len(ok_isubs), nchan, nbin), dtype=np.float32)
            for t in np.unique(table_of[ok_isubs]):         # one rotation batch per frequency table
                sel = np.where(table_of[ok_isubs] == t)[0]
                pl.set_freqs(freqs[ok_isubs[sel[0]]])
                rot[sel] = pl.rotate_batch(_f32(np.asarray(d.subints)[ok_isubs[sel], 0]), phi[sel], DM[sel],
                                           np.asarray(d.Ps)[ok_isubs[sel]], nus[sel, 0], GM=GM[sel],
                                           nu_GM=nus[sel, 1])
            channel_red_chi2s, zap_channels = [], []
            for j, isub in enumerate(ok_isubs):
                ok_ichans = np.asarray(d.ok_ichans[isub], dtype=int)
                model0 = models[table_of[isub]]
                model = model0
                if self.taus[k][isub] != 0.0:               # 1388-1394
                    tau = 10 ** self.taus[k][isub] if self.log10_tau else self.taus[k][isub]
                    taus = scattering_times(tau, self.alphas[k][isub], freqs[isub], nus[j, 2])
                    model = np.fft.irfft(scattering_portrait_FT(taus, nbin) *
                                         np.fft.rfft(model0, axis=1), axis=1)
                model_scaled = self.scales[k][isub][:, None] * model
                noise = np.asarray(d.noise_stds)[isub, 0]
                csnr = self.channel_snrs[k][isub]
                thr = (SNR_threshold ** 2.0 / len(ok_ichans)) ** 0.5
                red, bad = [], []
                for c in ok_ichans:
                    rc2 = np.sum(((rot[j, c] - model_scaled[c]) / noise[c]) ** 2.0) / (nbin - 2)
                    red.append(rc2)
                    if rc2 > rchi2_threshold or np.isnan(rc2):
                        bad.append(int(c))
                    elif SNR_threshold and csnr[c] < thr:
                        bad.append(int(c))
                if iterate and SNR_threshold and len(bad):  # 1262-1277
                    old_len, added_new = len(bad), True
                    while added_new and (len(ok_ichans) - len(bad)):
                        thr = (SNR_threshold ** 2.0 / (len(ok_ichans) - len(bad))) ** 0.5
                        for c in ok_ichans:
                            if int(c) not in bad and csnr[c] < thr:
                                bad.append(int(c))
                        added_new = bool(len(bad) - old_len)
                        old_len = len(bad)
                channel_red_chi2s.append(red)
                zap_channels.append(bad)
            self.channel_red_chi2s.append(channel_red_chi2s)
            self.zap_channels.append(zap_channels)
