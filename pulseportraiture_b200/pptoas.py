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


def _chan_mask(nsub, nchan, ok_ichans, isubs):
    """uint8 [nsub, nchan]: 1 at the usable channels ok_ichans[i] of every subint i in isubs, 0 elsewhere."""
    m = np.zeros((nsub, nchan), dtype=np.uint8)
    for i in isubs:
        m[i, np.asarray(ok_ichans[i], dtype=int)] = 1
    return m


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
            out["ok_mask"] = _chan_mask(data["nsub"], data["nchan"], v, range(len(v)))
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


# the result lists of GetTOAs (pptoas.py:102-143): the TOA methods append one entry per archive fitted, except
# TOA_list (one per TOA) and ok_idatafiles (one per archive loaded)
_RESULT_LISTS = ("obs", "doppler_fs", "nu0s", "nu_fits", "nu_refs", "ok_idatafiles",
                 "ok_isubs", "epochs", "MJDs", "Ps", "phis", "phi_errs", "TOAs",
                 "TOA_errs", "DM0s", "DMs", "DM_errs", "DeltaDM_means", "DeltaDM_errs",
                 "GMs", "GM_errs", "taus", "tau_errs", "alphas", "alpha_errs", "scales",
                 "scale_errs", "snrs", "channel_snrs", "profile_fluxes",
                 "profile_flux_errs", "fluxes", "flux_errs", "flux_freqs", "red_chi2s",
                 "channel_red_chi2s", "covariances", "nfevals", "rcs", "fit_durations",
                 "order", "TOA_list", "zap_channels")


def _archive_entries(d):
    """The result-list entries that describe the archive itself, the same for both TOA methods."""
    return dict(order=d.filename, obs=DataBunch(telescope=d.telescope, backend=d.backend, frontend=d.frontend),
                doppler_fs=d.doppler_factors, ok_isubs=np.asarray(d.ok_isubs, dtype=int), epochs=d.epochs,
                MJDs=np.array([e.in_days() for e in d.epochs], dtype=np.double),
                Ps=np.asarray(d.Ps, dtype=np.float64))


def _nu_fit_guesses(d, mask):
    """[nsub, 3] nu_fits: guess_fit_freq (pptoas.py:402) of every subint in ok_isubs over its usable channels (mask),
    0 for the other subints."""
    ok_isubs = np.asarray(d.ok_isubs, dtype=int)
    out = np.zeros((int(d.nsub), 3))
    out[ok_isubs, :] = pplib.guess_fit_freq_batch(np.asarray(d.freqs, dtype=np.float64)[ok_isubs],
                                                  np.asarray(d.SNRs, dtype=np.float64)[ok_isubs, 0],
                                                  mask[ok_isubs])[:, None]
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
        for name in _RESULT_LISTS:
            setattr(self, name, [])
        # by index into datafiles: the archive as fitted, and (table_of, models) of get_TOAs, for get_channels_to_zap
        self._archives, self._model_tables = {}, {}
        self.instrumental_response_dict = self.ird = {'DM': 0.0, 'wids': [], 'irf_types': []}
        self.quiet = quiet

    def _append_archive(self, entries):
        """Append one archive's results, {result-list name: entry}, to the lists _RESULT_LISTS names."""
        for name, value in entries.items():
            getattr(self, name).append(value)

    def _archives_to_fit(self, datafile, tscrunch, quiet):
        """(iarch, DataBunch) of every archive that loads and has subints to fit, listed in ok_idatafiles and kept in
        _archives (pptoas.py:247-265)."""
        datafiles = self.datafiles if datafile is None else [datafile]
        for iarch, datafile in enumerate(datafiles):
            try:
                d = datafile if isinstance(datafile, dict) else load_data(datafile)
            except (RuntimeError, IOError, OSError):
                if not quiet:
                    print("Cannot load_data(%s).  Skipping it." % datafile)
                continue
            if d.get("dmc"):                                # pptoas.py:256-265
                if not quiet:
                    print("%s is dedispersed (dmc = 1).  Restoring the dispersion." % d.filename)
                d = restore_dispersion(d)
            if tscrunch:                                    # load_data(..., tscrunch=True), pptoas.py:253
                d = tscrunch_databunch(d)
            if not len(d.ok_isubs):
                if not quiet:
                    print("No subints to fit for %s.  Skipping it." % d.filename)
                continue
            self.ok_idatafiles.append(iarch)
            self._archives[iarch] = d
            yield iarch, d

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

    def _model_tables_of(self, d, fit_scat, add_instrumental_response, by_period):
        """(tables, table_of, models): an archive's frequency tables, each subint's index into them (-1: not fit) and
        the model of every index an ok subint uses.  The reference builds a model per subint (freqs = data.freqs[isub],
        pptoas.py:346, 356-379); here subints share one when they share a table, or with by_period a (table, period)."""
        freqs = np.asarray(d.freqs, dtype=np.float64)
        Ps = np.asarray(d.Ps, dtype=np.float64)
        ok_isubs = np.asarray(d.ok_isubs, dtype=int)
        tables, table_of = _freq_tables(freqs)
        if not by_period:
            models = {t: self._model_for(d.phases, tables[t], Ps[ok_isubs[table_of[ok_isubs] == t][0]],
                                         fit_scat, add_instrumental_response)
                      for t in np.unique(table_of[ok_isubs])}
            return tables, table_of, models

        # (the smearing width uses the spacing of the subint's first two usable channels: the
        # reference evaluates instrumental_response_port_FT on freqsx, pptoas.py:390-392)
        def cbw(i):
            okc_ = np.asarray(d.ok_ichans[i], dtype=int)
            if not (add_instrumental_response and self.ird['DM']) or len(okc_) < 2:
                return 0.0
            return float(abs(freqs[i, okc_[1]] - freqs[i, okc_[0]]))
        ok = set(ok_isubs)
        keys = [(int(table_of[i]), float(Ps[i]), cbw(i) if i in ok else 0.0) for i in range(int(d.nsub))]
        uniq = sorted(set(keys[i] for i in ok_isubs))
        table_of = np.array([uniq.index(k) if k in uniq else -1 for k in keys])
        tables = np.array([tables[k[0]] for k in uniq])
        models = {t: self._model_for(d.phases, tables[t], uniq[t][1], fit_scat, add_instrumental_response,
                                     chan_bw=uniq[t][2] or None)
                  for t in range(len(uniq))}
        return tables, table_of, models

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
        start = time.time()
        for iarch, d in self._archives_to_fit(datafile, tscrunch, quiet):
            by_period = self._model_depends_on_P(fit_scat, add_instrumental_response)
            tables, table_of, models = self._model_tables_of(d, fit_scat, add_instrumental_response, by_period)
            mask = _chan_mask(int(d.nsub), int(d.nchan), d.ok_ichans, d.ok_isubs)
            if method == 'TNC' and bounds is None:          # pptoas.py:461-469
                # bounds is rebound: the later archives keep this box, its tau floor from this archive's nbin
                tau_bounds = (np.log10((10 * int(d.nbin)) ** -1), None) if self.log10_tau else (0.0, None)
                bounds = [(None, None), (None, None), (None, None), tau_bounds, (-10.0, 10.0)]
            nu_fits_in, mode, nu_outs_in, scat_in, fit_bounds = self._fit_inputs(d, mask, nu_refs, nu_fits,
                                                                                 fit_scat, method, bounds)
            self._model_tables[iarch] = (table_of, {t: np.asarray(m, dtype=np.float64) for t, m in models.items()})
            res, flags_of, fit_duration = self._fit_archive(d, tables, table_of, models, mask, nu_fits_in, mode,
                                                            nu_outs_in, scat_in, fit_bounds)
            out = _archive_entries(d)
            out.update(nu0s=d.nu0, fit_durations=fit_duration)
            out.update(self._subint_toas(d, models, table_of, mask, res, flags_of, nu_fits_in, nu_refs,
                                         print_phase, print_flux, print_parangle, addtnl_toa_flags))
            out.update(self._archive_arrays(d, res, out["DMs"], out["DM_errs"], method))
            self._append_archive(out)
            if not quiet:
                ok_isubs = out["ok_isubs"]
                print("--------------------------")
                print(d.filename)
                print("~%.4f sec/TOA" % (fit_duration / len(ok_isubs)))
                print("Med. TOA error is %.3f us" % (np.median(out["phi_errs"][ok_isubs]) * out["Ps"].mean() * 1e6))
        tot_duration = time.time() - start
        if not quiet and len(self.ok_isubs):
            print("--------------------------")
            print("Total time: %.2f sec, ~%.4f sec/TOA" % (
                tot_duration, tot_duration / (np.array(list(map(len, self.ok_isubs))).sum())))

    def _fit_inputs(self, d, mask, nu_ref_tuple, nu_fit_tuple, fit_scat, method, bounds):
        """Start values and bounds of an archive's fit (pptoas.py:400-469): nu_fits [nsub, 3] and nu_fit_mode
        (None and 1: the device guesses nu_fit), nu_outs [nsub, 3] or None, the scattering start values
        [nsub, 2] or None, and the bounds as fit_batch takes them."""
        nsub = int(d.nsub)
        ok_isubs = np.asarray(d.ok_isubs, dtype=int)
        freqs = np.asarray(d.freqs, dtype=np.float64)
        Ps = np.asarray(d.Ps, dtype=np.float64)
        if nu_fit_tuple is None and fit_scat:
            # the scattering start value needs nu_fit_tau on the host (pptoas.py:402, 431-441)
            nu_fits_in = _nu_fit_guesses(d, mask)
            empty = nu_fits_in[:, 0] == 0
            nu_fits_in[empty] = freqs[empty].mean(axis=1)[:, None]
            mode = 0
        elif nu_fit_tuple is None:
            nu_fits_in, mode = None, 1                     # guess_fit_freq, pptoas.py:402
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
                if self.bary:
                    nu_outs_in[:, 2] /= np.asarray(d.doppler_factors)
        scat_in = None
        if fit_scat:                                        # pptoas.py:427-441
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
        # bounds act with TNC only (pptoaslib.py:1008)
        fit_bounds = pplib._check_bounds(bounds, 5) if method == 'TNC' else None
        return nu_fits_in, mode, nu_outs_in, scat_in, fit_bounds

    def _fit_archive(self, d, tables, table_of, models, mask, nu_fits_in, mode, nu_outs_in, scat_in, fit_bounds):
        """Fit every subint in ok_isubs against its own model: ([nsub, ...] fit_batch results, fit_flags by subint,
        wall time of the fits).  Subints with a single usable channel are fit for phase only (pptoas.py:475-478); two
        channels drop GM (479-483).  Every model goes to the plan in one pp_set_models call (several when they exceed
        _MODEL_BUDGET_BYTES of device memory) and every flags group is one fit_batch (pp_fit_batch_models)."""
        nsub, nchan, nbin = int(d.nsub), int(d.nchan), int(d.nbin)
        ok_isubs = np.asarray(d.ok_isubs, dtype=int)
        Ps = np.asarray(d.Ps, dtype=np.float64)
        nok = mask.sum(axis=1)
        subints = _dev(np.asarray(d.subints)[:, 0])          # float64 goes to the device as it is
        errs = np.ascontiguousarray(np.asarray(d.noise_stds)[:, 0], dtype=np.float64)
        snrs = np.ascontiguousarray(np.asarray(d.SNRs)[:, 0], dtype=np.float64)
        weights = np.ascontiguousarray(d.weights, dtype=np.float64)
        pl = get_plan(nchan, nbin)
        flags_of = {}
        for isub in ok_isubs:
            if nok[isub] == 1:
                flags_of[isub] = (1, 0, 0, 0, 0)
            elif nok[isub] == 2 and self.fit_DM and self.fit_GM:
                flags_of[isub] = tuple(self.fit_flags[:2] + [0] + self.fit_flags[3:])
            else:
                flags_of[isub] = tuple(self.fit_flags)
        model_ids = sorted(models)
        per_call = max(1, int(_MODEL_BUDGET_BYTES // model_bytes(nchan, nbin)))
        res = {}
        fit_start = time.time()
        for m0 in range(0, len(model_ids), per_call):      # every round holds the model of some ok subint
            mset = model_ids[m0:m0 + per_call]
            ms = [_mdl(models[t]) for t in mset]
            dt = np.float32 if all(m.dtype == np.float32 for m in ms) else np.float64
            pl.set_models(np.stack([np.asarray(m, dtype=dt) for m in ms]), np.stack([tables[t] for t in mset]))
            local = {t: i for i, t in enumerate(mset)}
            groups = {}
            for isub in ok_isubs:
                if int(table_of[isub]) in local:
                    groups.setdefault(flags_of[isub], []).append(isub)
            for flags, isubs in sorted(groups.items()):
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
                    chan_mask=mask[idx], weights=weights[idx], DM_guess=np.full(nidx, float(d.DM)),
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
        return res, flags_of, time.time() - fit_start

    def _subint_toas(self, d, models, table_of, mask, res, flags_of, nu_fits_in, nu_ref_tuple,
                     print_phase, print_flux, print_parangle, addtnl_toa_flags):
        """Append a TOA with its flags per fitted subint to TOA_list (pptoas.py:528-651); the per-subint results."""
        nsub, nchan, nbin = int(d.nsub), int(d.nchan), int(d.nbin)
        ok_isubs = np.asarray(d.ok_isubs, dtype=int)
        freqs = np.asarray(d.freqs, dtype=np.float64)
        Ps = np.asarray(d.Ps, dtype=np.float64)
        nok = mask.sum(axis=1)
        phis = np.zeros(nsub); phi_errs = np.zeros(nsub)
        TOAs = np.zeros(nsub, dtype="object"); TOA_errs = np.zeros(nsub, dtype="object")
        DMs = np.zeros(nsub); DM_errs = np.zeros(nsub)
        GMs = np.zeros(nsub); GM_errs = np.zeros(nsub)
        scales = np.zeros([nsub, nchan]); scale_errs = np.zeros([nsub, nchan])
        channel_snrs = np.zeros([nsub, nchan])
        profile_fluxes = np.zeros([nsub, nchan]); profile_flux_errs = np.zeros([nsub, nchan])
        fluxes = np.zeros(nsub); flux_errs = np.zeros(nsub); flux_freqs = np.zeros(nsub)
        covariances = np.zeros([nsub, self.nfit, self.nfit])
        nu_fits_arr = list(np.zeros([nsub, 3])); nu_refs_arr = list(np.zeros([nsub, 3]))
        # everything that is the same arithmetic for every subint, for all of them at once
        okm = mask.astype(bool)
        okm[np.setdiff1d(np.arange(nsub), ok_isubs)] = False
        scales[okm] = res["scales"][okm]
        scale_errs[okm] = res["scale_errs"][okm]
        channel_snrs[okm] = res["channel_snrs"][okm]
        fmax = np.where(okm, freqs, -np.inf).max(axis=1)
        fmin = np.where(okm, freqs, np.inf).min(axis=1)
        nu_fits_rows = _nu_fit_guesses(d, mask) if nu_fits_in is None else nu_fits_in   # pptoas.py:400-407
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
            if print_flux:                                  # pptoas.py:554-577
                okc = np.nonzero(okm[isub])[0]
                means = np.asarray(models[table_of[isub]])[okc].mean(axis=1)
                profile_fluxes[isub, okc] = means * scales[isub, okc]
                profile_flux_errs[isub, okc] = abs(means) * scale_errs[isub, okc]
                fluxes[isub], flux_errs[isub] = weighted_mean(profile_fluxes[isub, okc],
                                                             profile_flux_errs[isub, okc])
                flux_freqs[isub], _ = weighted_mean(freqs[isub, okc], profile_flux_errs[isub, okc])
            nu_refs_arr[isub] = list(nu_out)
            nu_fits_arr[isub] = list(nu_fits_rows[isub])
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
            else:                                           # pptoas.py:596-600
                for ii, a_ in enumerate(ifit):
                    for jj, b_ in enumerate(ifit):
                        if a_ < self.nfit and b_ < self.nfit:
                            covariances[isub][a_, b_] = cm[ii, jj]
            snr, gof = res["snr"][isub], res["red_chi2"][isub]
            toa_flags = {}                                  # pptoas.py:604-651
            DM_out, DM_err_out = (DM, DM_err) if flags[1] else (None, None)
            if flags[2]:
                toa_flags['gm'], toa_flags['gm_err'] = GM, GM_err
            if flags[3]:                                    # pptoas.py:611-624
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
            toa_flags.update(be=d.backend, fe=d.frontend, f=fe_be, nbin=nbin, nch=nchan, nchx=int(nok[isub]),
                             bw=fmax[isub] - fmin[isub], chbw=chbw, subint=int(isub), tobs=subtimes[isub],
                             fratio=fmax[isub] / fmin[isub], tmplt=tmplt, snr=snr)
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
            toa_flags.update(addtnl_toa_flags)
            self.TOA_list.append(TOA(d.filename, nu_out[0], TOA_mjd, TOA_err,
                                     d.telescope, d.telescope_code, DM_out, DM_err_out,
                                     toa_flags))
        return dict(phis=phis, phi_errs=phi_errs, TOAs=TOAs, TOA_errs=TOA_errs, DMs=DMs, DM_errs=DM_errs,
                    GMs=GMs, GM_errs=GM_errs, scales=scales, scale_errs=scale_errs, channel_snrs=channel_snrs,
                    profile_fluxes=profile_fluxes, profile_flux_errs=profile_flux_errs, fluxes=fluxes,
                    flux_errs=flux_errs, flux_freqs=flux_freqs, covariances=covariances, nu_fits=nu_fits_arr,
                    nu_refs=nu_refs_arr)

    def _archive_arrays(self, d, res, DMs, DM_errs, method):
        """The per-archive result arrays taken from the fit as they are, and the Delta-DM mean (pptoas.py:665-682)."""
        nsub = int(d.nsub)
        ok_isubs = np.asarray(d.ok_isubs, dtype=int)
        taus = np.zeros(nsub); tau_errs = np.zeros(nsub)
        alphas = np.zeros(nsub); alpha_errs = np.zeros(nsub)
        nfevals = np.zeros(nsub, dtype="int"); rcs = np.zeros(nsub, dtype="int")
        snrs = np.zeros(nsub); red_chi2s = np.zeros(nsub)
        taus[ok_isubs], tau_errs[ok_isubs] = res["params"][ok_isubs, 3], res["param_errs"][ok_isubs, 3]
        alphas[ok_isubs], alpha_errs[ok_isubs] = res["params"][ok_isubs, 4], res["param_errs"][ok_isubs, 4]
        nfevals[ok_isubs] = res["nfeval"][ok_isubs]
        # pptoaslib.py:1017
        rcs[ok_isubs] = [pplib.scipy_return_code(c, method) for c in res["return_code"][ok_isubs]]
        snrs[ok_isubs] = res["snr"][ok_isubs]
        red_chi2s[ok_isubs] = res["red_chi2"][ok_isubs]
        DM0 = float(d.DM) if self.DM0 is None else self.DM0
        DeltaDMs = DMs - DM0
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
        return dict(taus=taus, tau_errs=tau_errs, alphas=alphas, alpha_errs=alpha_errs, nfevals=nfevals, rcs=rcs,
                    snrs=snrs, red_chi2s=red_chi2s, DM0s=DM0, DeltaDM_means=DeltaDM_mean,
                    DeltaDM_errs=DeltaDM_var ** 0.5)

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
        for _, d in self._archives_to_fit(datafile, tscrunch, quiet):
            nsub, nchan, nbin = int(d.nsub), int(d.nchan), int(d.nbin)
            ok_isubs = np.asarray(d.ok_isubs, dtype=int)
            freqs = np.asarray(d.freqs, dtype=np.float64)
            Ps = np.asarray(d.Ps, dtype=np.float64)
            _, table_of, models = self._model_tables_of(d, False, add_instrumental_response, by_period=False)
            model_of = [models[t] for t in table_of]
            pl = get_plan(nchan, nbin)
            fit_start = time.time()
            profs = _f32(np.asarray(d.subints)[ok_isubs, 0]).reshape(len(ok_isubs) * nchan, nbin)
            noise = np.ascontiguousarray(np.asarray(d.noise_stds)[ok_isubs, 0], dtype=np.float64)
            okmask = _chan_mask(nsub, nchan, d.ok_ichans, ok_isubs)[ok_isubs].astype(bool) & (noise > 0)
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
            out = _archive_entries(d)
            out.update(phis=phis, phi_errs=phi_errs, TOAs=TOAs, TOA_errs=TOA_errs, taus=taus, tau_errs=tau_errs,
                       scales=scales, scale_errs=scale_errs, channel_snrs=channel_snrs, profile_fluxes=profile_fluxes,
                       profile_flux_errs=profile_flux_errs, channel_red_chi2s=channel_red_chi2s,
                       fit_durations=fit_duration)
            self._append_archive(out)
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
