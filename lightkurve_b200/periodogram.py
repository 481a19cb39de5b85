"""Periodogram classes: the mirror of /root/reference/src/lightkurve/periodogram.py on the hot path.

``LombScarglePeriodogram.from_lightcurve`` (:636-989) and
``BoxLeastSquaresPeriodogram.from_lightcurve`` (:1042-1192) keep the reference's keyword
handling, defaults, frequency/period grid construction, warnings and error strings; the two
places where the reference calls astropy (``LombScargle(...).power`` :961-964 and
``BoxLeastSquares(...).power`` :1161-1169) are single C-ABI calls into the CUDA kernels
(``lkb_ls_power`` with the :969-975 rescale fused as its epilogue, and ``lkb_bls_power``).
"""
import copy
import logging
import math
import warnings

import numpy as np

from . import units as u
from .units import Quantity, Time
from .utils import LightkurveWarning, validate_method

log = logging.getLogger(__name__)

__all__ = ["Periodogram", "SNRPeriodogram", "LombScarglePeriodogram", "BoxLeastSquaresPeriodogram"]

_PER_DAY = 1 / u.day          # built once: the single-light-curve call is latency-bound (BASELINE config 1)


def _is_regular(frequency):
    """astropy implementations.main._is_regular (used at periodogram.py:933)."""
    frequency = np.asarray(getattr(frequency, "value", frequency))
    if frequency.ndim != 1:
        return False
    if len(frequency) == 1:
        return True
    d = np.diff(frequency)
    return bool(np.allclose(d[0], d))


class Periodogram(object):
    """Generic power spectrum container (periodogram.py:33-586, without plotting/table export)."""

    frequency = None
    power = None

    def __init__(self, frequency, power, nyquist=None, label=None, targetid=None, default_view="frequency",
                 meta={}):
        if not isinstance(frequency, Quantity):
            raise ValueError("frequency must be an `astropy.units.Quantity` object.")
        if not isinstance(power, Quantity):
            raise ValueError("power must be an `astropy.units.Quantity` object.")
        if not frequency.unit.is_equivalent(u.Hz):
            raise ValueError("Frequency must be in units of 1/time.")
        if frequency.shape[0] <= 1:
            raise ValueError("frequency and power must have a length greater than 1.")
        if frequency.shape != power.shape:
            raise ValueError("frequency and power must have the same length.")
        self.frequency = frequency
        self.power = power
        self.nyquist = nyquist
        self.label = label
        self.targetid = targetid
        self.default_view = self._validate_view(default_view)
        self.meta = meta

    def _validate_view(self, view):
        if view is None and hasattr(self, "default_view"):
            view = self.default_view
        return validate_method(view, ["frequency", "period"])

    def _is_evenly_spaced(self):
        freqdiff = np.diff(self.frequency.value)
        return bool(np.allclose(freqdiff[0], freqdiff))

    @property
    def period(self):
        """The array of periods, i.e. 1/frequency."""
        return 1.0 / self.frequency

    @property
    def max_power(self):
        return np.nanmax(self.power)

    @property
    def frequency_at_max_power(self):
        return self.frequency[np.nanargmax(self.power.value)]

    @property
    def period_at_max_power(self):
        return 1.0 / self.frequency_at_max_power

    def copy(self):
        return copy.deepcopy(self)

    def __repr__(self):
        return "Periodogram(ID: {})".format(self.label)

    def __getitem__(self, key):
        copy_self = self.copy()
        copy_self.frequency = self.frequency[key]
        copy_self.power = self.power[key]
        return copy_self

    def _arith(self, other, op):
        copy_self = self.copy()
        copy_self.power = op(copy_self.power, other)
        return copy_self

    def __add__(self, other):
        return self._arith(other, lambda a, b: a + b)

    __radd__ = __add__

    def __sub__(self, other):
        return self._arith(other, lambda a, b: a - b)

    def __rsub__(self, other):
        return self._arith(other, lambda a, b: b - a)

    def __mul__(self, other):
        return self._arith(other, lambda a, b: a * b)

    __rmul__ = __mul__

    def __truediv__(self, other):
        return self._arith(other, lambda a, b: a / b)

    def __rtruediv__(self, other):
        return self._arith(other, lambda a, b: b / a)

    def bin(self, binsize=10, method="mean"):
        """Bins the power spectrum (periodogram.py:142-180)."""
        if binsize < 1:
            raise ValueError("binsize must be larger than or equal to 1")
        method = validate_method(method, ["mean", "median"])
        m = int(len(self.power) / binsize)
        fr = self.frequency.value[: m * binsize].reshape((m, binsize))
        pw = self.power.value[: m * binsize].reshape((m, binsize))
        if method == "mean":
            binned_freq, binned_power = fr.mean(1), pw.mean(1)
        else:
            binned_freq, binned_power = np.nanmedian(fr, axis=1), np.nanmedian(pw, axis=1)
        binned_pg = self.copy()
        binned_pg.frequency = Quantity(binned_freq, self.frequency.unit)
        binned_pg.power = Quantity(binned_power, self.power.unit)
        return binned_pg

    def smooth(self, method="boxkernel", filter_width=0.1):
        """Smooths the power spectrum (periodogram.py:182-284)."""
        method = validate_method(method, ["boxkernel", "logmedian"])
        if method == "boxkernel":
            if getattr(filter_width, "value", filter_width) <= 0.0:
                raise ValueError("the `filter_width` parameter must be "
                                 "larger than 0 for the 'boxkernel' method.")
            try:
                filter_width = Quantity(filter_width, self.frequency.unit)
            except u.UnitConversionError:
                raise ValueError("the `filter_width` parameter must have " "frequency units.")
            if not self._is_evenly_spaced():
                raise ValueError("the 'boxkernel' method requires the periodogram "
                                 "to have a grid of evenly spaced frequencies.")
            fs = np.mean(np.diff(self.frequency.value))
            width = int(math.ceil(float(filter_width.value) / fs))
            # astropy Box1DKernel(width) has an odd number of taps; convolve(): zero fill, normalised
            ntaps = width if width % 2 == 1 else width + 1
            kernel = np.ones(ntaps)
            if width % 2 == 0:
                kernel[0] = kernel[-1] = 0.5
            kernel /= kernel.sum()
            full = np.convolve(self.power.value, kernel, mode="full")      # zero-filled boundaries
            start = (ntaps - 1) // 2
            smooth_power = full[start:start + len(self.power)]
            smooth_pg = self.copy()
            smooth_pg.power = Quantity(smooth_power, self.power.unit)
            return smooth_pg
        if isinstance(filter_width, Quantity) or u.is_quantity(filter_width):
            raise ValueError("the 'logmedian' method requires a dimensionless "
                             "value for `filter_width` in log10(frequency) space.")
        # moving log-median on the GPU (exact medians per window; lkb_pg_logmedian)
        from . import engine
        bkg = engine.pg_logmedian(self.frequency.value, self.power.value, float(filter_width))
        smooth_pg = self.copy()
        smooth_pg.power = Quantity(bkg, self.power.unit)
        return smooth_pg

    def flatten(self, method="logmedian", filter_width=0.01, return_trend=False):
        """Signal-to-noise spectrum (periodogram.py:381-429)."""
        bkg = self.smooth(method=method, filter_width=filter_width)
        snr_pg = self / bkg.power
        snr = SNRPeriodogram(snr_pg.frequency, snr_pg.power, nyquist=self.nyquist, targetid=self.targetid,
                             label=self.label, meta=self.meta)
        if return_trend:
            return snr, bkg
        return snr

    def to_seismology(self, **kwargs):
        """`Seismology` object of this periodogram (periodogram.py:576-587); background-correct it first
        (`flatten()`), otherwise a LightkurveWarning is raised."""
        from .seismology import Seismology
        return Seismology(self)

    def plot(self, *args, **kwargs):
        raise NotImplementedError("plotting is outside the hot-path scope of lightkurve_b200")


class SNRPeriodogram(Periodogram):
    """Signal-to-noise spectrum (periodogram.py:589-619)."""

    def __repr__(self):
        return "SNRPeriodogram(ID: {})".format(self.label)


class LombScarglePeriodogram(Periodogram):
    """Power spectrum generated with the Lomb-Scargle method (periodogram.py:622-1018)."""

    def __init__(self, *args, **kwargs):
        self._LS_object = kwargs.pop("ls_obj", None)
        self.nterms = kwargs.pop("nterms", 1)
        self.ls_method = kwargs.pop("ls_method", "fastchi2")
        self._fit_data = kwargs.pop("fit_data", None)      # (time, flux) the model() fit needs
        super(LombScarglePeriodogram, self).__init__(*args, **kwargs)

    def __repr__(self):
        return "LombScarglePeriodogram(ID: {})".format(self.label)

    @staticmethod
    def _prepare(lc, minimum_frequency=None, maximum_frequency=None, minimum_period=None, maximum_period=None,
                 frequency=None, period=None, nterms=1, nyquist_factor=1, oversample_factor=None, freq_unit=None,
                 normalization="amplitude", ls_method="fast", **kwargs):
        """Everything from_lightcurve does BEFORE the astropy call (periodogram.py:784-958).
        Returns a dict with the cleaned light curve, the frequency grid (Quantity in freq_unit)
        and the bookkeeping the result object needs."""
        normalization = validate_method(normalization, ["psd", "amplitude"])
        if np.isnan(np.asarray(lc.flux.value)).any():
            lc = lc.remove_nans()
            log.debug("Lightcurve contains NaN values."
                      "These are removed before creating the periodogram.")
        if freq_unit is None:
            freq_unit = _PER_DAY if normalization == "amplitude" else u.microhertz
        freq_unit = u._as_unit(freq_unit)
        if oversample_factor is None:
            oversample_factor = 5.0 if normalization == "amplitude" else 1.0

        for old, new in (("min_period", "minimum_period"), ("max_period", "maximum_period"),
                         ("min_frequency", "minimum_frequency"), ("max_frequency", "maximum_frequency")):
            if old in kwargs:
                warnings.warn("`{}` keyword is deprecated, "
                              "please use `{}` instead.".format(old, new), LightkurveWarning)
                val = kwargs.pop(old, None)
                if new == "minimum_period":
                    minimum_period = val
                elif new == "maximum_period":
                    maximum_period = val
                elif new == "minimum_frequency":
                    minimum_frequency = val
                else:
                    maximum_frequency = val
        if kwargs:
            raise TypeError("unsupported LombScargle keyword(s) {}: the CUDA kernel implements the "
                            "reference's own call (dy=None, fit_mean=True, center_data=True)".format(sorted(kwargs)))

        if not all(b is None for b in [period, minimum_period, maximum_period]):
            default_view = "period"
        else:
            default_view = "frequency"
        if (not all(b is None for b in [period, minimum_period, maximum_period])) & (
                not all(b is None for b in [frequency, minimum_frequency, maximum_frequency])):
            raise ValueError("You have input keyword arguments for both frequency and period. "
                             "Please only use one.")

        time = lc.time.copy()
        tval = np.asarray(time.value, dtype=np.float64)
        nyquist = Quantity(0.5 * (1.0 / (np.median(np.diff(tval)))), _PER_DAY)
        fs = Quantity((1.0 / (tval[-1] - tval[0])) / oversample_factor, _PER_DAY)
        nyquist = nyquist.to(freq_unit)
        fs = fs.to(freq_unit)

        if (frequency is not None) & (any([a is not None for a in [minimum_frequency, maximum_frequency]])):
            log.warning("You have passed both a grid of frequencies "
                        "and min_frequency/maximum_frequency arguments; "
                        "the latter will be ignored.")
        if (period is not None) & (any([a is not None for a in [minimum_period, maximum_period]])):
            log.warning("You have passed a grid of periods "
                        "and minimum_period/maximum_period arguments; "
                        "the latter will be ignored.")

        def _inv(x):
            if u.is_quantity(x):
                return 1.0 / Quantity(x)
            return 1.0 / np.asarray(x, dtype=float) if np.ndim(x) else 1.0 / x

        if maximum_period is not None:
            minimum_frequency = _inv(maximum_period)
        if minimum_period is not None:
            maximum_frequency = _inv(minimum_period)
        if period is not None:
            frequency = _inv(period)

        grid_is_arange = frequency is None      # built below by np.arange: regular by construction
        if frequency is None:
            if minimum_frequency is not None:
                minimum_frequency = Quantity(minimum_frequency, freq_unit)
            if maximum_frequency is not None:
                maximum_frequency = Quantity(maximum_frequency, freq_unit)
            if (minimum_frequency is not None) & (maximum_frequency is not None):
                if minimum_frequency > maximum_frequency:
                    if default_view == "frequency":
                        raise ValueError("minimum_frequency cannot be larger than maximum_frequency")
                    if default_view == "period":
                        raise ValueError("minimum_period cannot be larger than maximum_period")
            if minimum_frequency is None:
                minimum_frequency = fs
            if maximum_frequency is None:
                maximum_frequency = nyquist * nyquist_factor
            frequency = np.arange(float(minimum_frequency.value), float(maximum_frequency.value), float(fs.value))
        frequency = Quantity(frequency, freq_unit)

        # ls_method="fastnifty" / "fastnifty_chi2" (periodogram.py:917-931): the reference needs the optional nifty-ls
        # package for these and downgrades to "fast" / "fastchi2" without it.  Here the non-uniform FFT is one of the
        # library's own kernel families (csrc/ls_nufft.cu), so the name is kept - no import, no downgrade.

        if not (grid_is_arange or _is_regular(frequency)) and \
                ls_method in ["fastchi2", "fast", "fastnifty_chi2", "fastnifty"]:
            oldmethod = ls_method
            ls_method = {"fastchi2": "chi2", "fast": "slow", "fastnifty_chi2": "chi2", "fastnifty": "slow"}[ls_method]
            log.warning("The requested periodogram is not evenly sampled in frequency.\n"
                        "Method has been changed from '{}' to '{}' to allow for this.".format(oldmethod, ls_method))

        if (nterms > 1) and (ls_method not in ["fastchi2", "chi2", "fastnifty_chi2"]):
            warnings.warn(
                "Building a Lomb Scargle Periodogram using the `slow` method. "
                "`nterms` has been set to >1, however this is not supported under the `{}` method. "
                "To run with higher nterms, set `ls_method` to either 'fastchi2', 'chi2', or 'fastnifty_chi2. "
                "Please refer to the `astropy.timeseries.periodogram.LombScargle` documentation.".format(ls_method),
                LightkurveWarning,
            )
            nterms = 1
        if nterms > 4:
            raise NotImplementedError("nterms > 4 is not supported by the CUDA chi2 kernel")
        if ls_method not in ("fast", "slow", "auto", "cython", "scipy", "chi2", "fastchi2", "fastnifty",
                             "fastnifty_chi2"):
            raise ValueError("unknown ls_method '{}'".format(ls_method))
        return dict(lc=lc, time=tval, frequency=frequency, freq_unit=freq_unit, fs=fs, nyquist=nyquist,
                    oversample_factor=oversample_factor, normalization=normalization, ls_method=ls_method,
                    nterms=nterms, default_view=default_view)

    @staticmethod
    def _finish(prep, power_values):
        lc, norm = prep["lc"], prep["normalization"]
        if norm == "psd":
            unit = lc.flux.unit ** 2 / prep["freq_unit"]
        else:
            unit = lc.flux.unit
        power = Quantity(np.asarray(power_values, dtype=np.float64), unit)
        return LombScarglePeriodogram(frequency=prep["frequency"], power=power, nyquist=prep["nyquist"],
                                      targetid=lc.meta.get("TARGETID"), label=lc.meta.get("LABEL"),
                                      default_view=prep["default_view"], ls_obj=None, nterms=prep["nterms"],
                                      ls_method=prep["ls_method"], meta=lc.meta,
                                      fit_data=(prep["time"], np.asarray(lc.flux.value, dtype=np.float64),
                                                lc.flux.unit, lc.time.format, lc.time.scale))

    @staticmethod
    def _norm_args(prep):
        """(normalization name, per-LC scale) for the kernel epilogue (periodogram.py:969-975)."""
        if prep["normalization"] == "psd":
            n = len(prep["time"])
            return "psd", 2.0 / (n * prep["oversample_factor"] * float(prep["fs"].value))
        return "amplitude", None

    @staticmethod
    def _engine_algo(ls_method):
        """Kernel family for a (validated) ``ls_method`` - the `method=` of ``LombScargle.power`` at
        periodogram.py:964: "slow" is the exact direct sums; "fastnifty" asks for the non-uniform FFT (the algorithm
        nifty-ls implements); everything else ("fast", "auto", "cython", "scipy") lets the library choose - the FFT
        path for large jobs on grids that allow it, the direct sums otherwise.  Both families evaluate the same
        floating-mean estimator to the parity tolerance (DESIGN.md section 2)."""
        return {"slow": "direct", "fastnifty": "nufft"}.get(ls_method, "auto")

    @staticmethod
    def _ragged_power(engine, times, fluxes, freq, norm, scales, ls_method):
        algo = LombScarglePeriodogram._engine_algo(ls_method)
        try:
            return engine.ls_power_ragged(times, fluxes, freq, norm, scales, algo=algo)
        except Exception as e:
            if algo != "nufft" or getattr(e, "status", None) != -5:       # LKB_E_UNSUPPORTED
                raise
            log.warning("ls_method='fastnifty': this light curve / grid does not qualify for the non-uniform FFT "
                        "kernels ({}); the direct sums are used instead.".format(e))
            return engine.ls_power_ragged(times, fluxes, freq, norm, scales, algo="direct")

    @staticmethod
    def from_lightcurve(lc, **kwargs):
        """Creates a Periodogram from a LightCurve using the Lomb-Scargle method.

        Same signature as the reference (periodogram.py:636-652).  The power is the generalised
        (floating-mean) Lomb-Scargle estimator of astropy's ``method="slow"``, evaluated either by exact
        direct sums or through a non-uniform FFT accurate to the parity tolerance (see ``_engine_algo``);
        the reference's default ``ls_method="fast"`` is astropy's coarser extirpolation + FFT approximation
        of the same quantity.  ``pg.ls_method`` records the requested/auto-switched name as in the reference.
        """
        from . import engine
        prep = LombScarglePeriodogram._prepare(lc, **kwargs)
        norm, scale = LombScarglePeriodogram._norm_args(prep)
        freq_day = np.asarray(prep["frequency"].to(_PER_DAY).value, dtype=np.float64)
        flux = np.asarray(prep["lc"].flux.value)
        if flux.dtype != np.float32:
            flux = flux.astype(np.float64)
        if prep["ls_method"] in ("chi2", "fastchi2", "fastnifty_chi2"):
            # multi-term fit (periodogram.py:948-964): dedicated kernel, any nterms in [1, 4]
            out = engine.ls_power_chi2([prep["time"]], [flux], freq_day, prep["nterms"], norm,
                                       None if scale is None else [scale])
        else:
            out = LombScarglePeriodogram._ragged_power(engine, [prep["time"]], [flux], freq_day, norm,
                                                       None if scale is None else [scale], prep["ls_method"])
        return LombScarglePeriodogram._finish(prep, out[0])

    def model(self, time, frequency=None):
        """Obtain the flux model for a given frequency and time (periodogram.py:991-1018): the
        maximum-likelihood offset + nterms-harmonic fit at `frequency` (default: frequency at max
        power), evaluated at `time`, returned as a normalized LightCurve like the reference does.
        The normal equations are accumulated and solved on the GPU (lkb_ls_power_chi2)."""
        from . import engine
        from .lightcurve import LightCurve
        if self._fit_data is None:
            raise ValueError("No `astropy` Lomb Scargle object exists.")
        if frequency is None:
            frequency = self.frequency_at_max_power
        t_lc, y_lc, flux_unit, tfmt, tscale = self._fit_data
        f_day = float(np.asarray(Quantity(frequency, self.frequency.unit).to(1 / u.day).value))
        _, theta = engine.ls_power_chi2([t_lc], [y_lc], np.array([f_day]), self.nterms, "psd_raw", return_theta=True)
        th = theta[0, 0]
        tv = np.asarray(getattr(time, "value", time), dtype=np.float64)
        trel = tv - t_lc[0]
        f = np.full(len(tv), th[0] + y_lc.mean())
        for i in range(1, self.nterms + 1):
            f += th[2 * i - 1] * np.sin(2 * np.pi * i * f_day * trel) + th[2 * i] * np.cos(2 * np.pi * i * f_day * trel)
        lc = LightCurve(time=Time(tv, tfmt, tscale), flux=Quantity(f, flux_unit),
                        meta={"FREQUENCY": frequency, "LABEL": "LS Model"})
        return lc.normalize()


class BoxLeastSquaresPeriodogram(Periodogram):
    """Power spectrum generated with the BoxLeastSquares method (periodogram.py:1021-1340)."""

    def __init__(self, *args, **kwargs):
        self.duration = kwargs.pop("duration", None)
        self.depth = kwargs.pop("depth", None)
        self.snr = kwargs.pop("snr", None)
        self._BLS_result = kwargs.pop("bls_result", None)
        self._BLS_object = kwargs.pop("bls_obj", None)
        self.transit_time = kwargs.pop("transit_time", None)
        self.time = kwargs.pop("time", None)
        self.flux = kwargs.pop("flux", None)
        self.time_unit = kwargs.pop("time_unit", None)
        super(BoxLeastSquaresPeriodogram, self).__init__(*args, **kwargs)

    def __repr__(self):
        return "BoxLeastSquaresPeriodogram(ID: {})".format(self.label)

    @staticmethod
    def autoperiod(time, duration, minimum_period=None, maximum_period=None, minimum_n_transit=3,
                   frequency_factor=1.0):
        """astropy BoxLeastSquares.autoperiod (closed form; called at periodogram.py:1163-1168)."""
        t = np.asarray(time, dtype=np.float64)
        duration = np.atleast_1d(np.asarray(duration, dtype=np.float64))
        baseline = t.max() - t.min()
        df = frequency_factor * duration.min() / baseline ** 2
        if minimum_period is None:
            minimum_period = 2.0 * duration.max()
        if maximum_period is None:
            if minimum_n_transit <= 1:
                raise ValueError("minimum number of transits must be greater than 1")
            maximum_period = baseline / (minimum_n_transit - 1)
        if maximum_period < minimum_period:
            minimum_period, maximum_period = maximum_period, minimum_period
        if minimum_period <= 0.0:
            raise ValueError("minimum period must be positive")
        minimum_frequency = 1.0 / maximum_period
        maximum_frequency = 1.0 / minimum_period
        nf = 1 + int(np.round((maximum_frequency - minimum_frequency) / df))
        return 1.0 / (maximum_frequency - df * np.arange(nf))

    @staticmethod
    def _prepare(lc, **kwargs):
        """Validation and grid construction of from_lightcurve (periodogram.py:1093-1168)."""
        lc = lc.remove_nans()
        flux_err = np.asarray(lc.flux_err.value, dtype=np.float64)
        dy = flux_err if np.isfinite(flux_err).all() else None

        duration = kwargs.pop("duration", [0.05, 0.10, 0.15, 0.20, 0.25, 0.33])
        duration = getattr(duration, "value", duration)
        if duration is not None and ~np.all(np.isfinite(duration)):
            raise ValueError("`duration` parameter contains illegal nan or inf value(s)")

        period = kwargs.pop("period", None)
        period = getattr(period, "value", period)
        minimum_period = kwargs.pop("minimum_period", None)
        maximum_period = kwargs.pop("maximum_period", None)
        minimum_period = getattr(minimum_period, "value", minimum_period)
        maximum_period = getattr(maximum_period, "value", maximum_period)
        if period is not None and ~np.all(np.isfinite(period)):
            raise ValueError("`period` parameter contains illegal nan or inf value(s)")
        tval = np.asarray(lc.time.value, dtype=np.float64)
        if minimum_period is None:
            if period is None:
                minimum_period = np.max([np.median(np.diff(tval)) * 4,
                                         np.max(duration) + np.median(np.diff(tval))])
            else:
                minimum_period = np.min(period)
        if maximum_period is None:
            if period is None:
                maximum_period = (np.max(tval) - np.min(tval)) / 3.0
            else:
                maximum_period = np.max(period)

        time_unit = kwargs.pop("time_unit", "day")
        if time_unit not in ("day", "d", "hour", "h", "minute", "min", "second", "s"):
            raise ValueError("{} is not a valid value for `time_unit`".format(time_unit))

        frequency_factor = kwargs.pop("frequency_factor", 10)
        df = frequency_factor * np.min(duration) / (np.max(tval) - np.min(tval)) ** 2
        npoints = int(((1 / minimum_period) - (1 / maximum_period)) / df)
        if npoints > 1e7:
            raise ValueError("`period` contains {} points."
                             "Periodogram is too large to evaluate. "
                             "Consider setting `frequency_factor` to a higher value."
                             "".format(np.round(npoints, 4)))
        elif npoints > 1e5:
            log.warning("`period` contains {} points."
                        "Periodogram is likely to be large, and slow to evaluate. "
                        "Consider setting `frequency_factor` to a higher value."
                        "".format(np.round(npoints, 4)))
        if period is None:
            period = BoxLeastSquaresPeriodogram.autoperiod(tval, duration, minimum_period=minimum_period,
                                                           maximum_period=maximum_period,
                                                           frequency_factor=frequency_factor)
        period = np.atleast_1d(np.asarray(period, dtype=np.float64))
        duration = np.atleast_1d(np.asarray(duration, dtype=np.float64))
        objective = kwargs.pop("objective", None) or "likelihood"
        validate_method(objective, ["likelihood", "snr"])
        # `bls_method` is the same keyword under a name that to_periodogram("bls", ...) can carry (its first argument
        # is already called `method`), as `ls_method` is for Lomb-Scargle
        method, bls_method = kwargs.pop("method", None), kwargs.pop("bls_method", None)
        method = method or bls_method or "fast"
        if method not in ("fast", "slow"):
            raise NotImplementedError("only astropy's methods 'fast' (binned) and 'slow' (exact) are implemented "
                                      "on the GPU")
        oversample = int(kwargs.pop("oversample", 10))
        if oversample < 1:
            raise ValueError("oversample must be an int greater than 0 (got {})".format(oversample))
        if kwargs:
            raise TypeError("unexpected keyword arguments {}".format(sorted(kwargs)))
        if np.min(period) <= np.max(duration):
            raise ValueError("The maximum transit duration must be shorter than the minimum period")
        flux, lc_dy = np.asarray(lc.flux.value, dtype=np.float64), dy
        if method == "slow" and np.any(np.diff(tval) < 0):
            # the exact search walks ascending times; its result does not depend on the cadence order (up to the
            # summation order of the sums)
            order = np.argsort(tval, kind="stable")
            tval, flux = tval[order], flux[order]
            dy = None if dy is None else dy[order]
        return dict(lc=lc, time=tval, flux=flux, dy=dy, period=period, duration=duration, objective=objective,
                    oversample=oversample, time_unit=time_unit, method=method, lc_dy=lc_dy)

    @staticmethod
    def _engine_kwargs(prep):
        """Keywords of engine.bls_power for a prepared call; `method` only for the exact search, so that the default
        binned search is requested exactly as by engines that know no other."""
        kw = dict(oversample=prep["oversample"], objective=prep["objective"])
        if prep["method"] != "fast":
            kw["method"] = prep["method"]
        return kw

    @staticmethod
    def _finish(prep, res, b=0):
        lc = prep["lc"]
        tu = u._as_unit(prep["time_unit"])
        period = Quantity(res["period"], tu)
        return BoxLeastSquaresPeriodogram(
            frequency=1.0 / period,
            power=Quantity(res["power"][b], u.dimensionless_unscaled),
            default_view="period",
            label=lc.meta.get("LABEL"),
            targetid=lc.meta.get("TARGETID"),
            transit_time=Time(res["transit_time"][b], lc.time.format, lc.time.scale),
            duration=Quantity(res["duration"][b], tu),
            depth=Quantity(res["depth"][b], lc.flux.unit),
            bls_result={k: res[k][b] for k in res if k not in ("period", "bins", "index")},
            snr=Quantity(res["depth_snr"][b], u.dimensionless_unscaled),
            bls_obj=None,
            time=lc.time,
            flux=lc.flux,
            time_unit=prep["time_unit"],
        )

    @staticmethod
    def from_lightcurve(lc, **kwargs):
        """Creates a Periodogram from a LightCurve using the Box Least Squares method
        (periodogram.py:1042-1192).  Keywords: duration, period, minimum_period, maximum_period,
        frequency_factor, time_unit, objective, oversample, method ("fast": astropy's binned search, K3; "slow": its
        exact unbinned search, K3s - the reported durations are then the trial durations themselves; through
        ``to_periodogram("bls", ...)`` spelled ``bls_method``).  Where astropy's method="slow" finds no box with
        positive depth at a period it raises; here that period gets power -inf."""
        from . import engine
        prep = BoxLeastSquaresPeriodogram._prepare(lc, **kwargs)
        res = engine.bls_power([prep["time"]], [prep["flux"]], None if prep["dy"] is None else [prep["dy"]],
                               prep["period"], prep["duration"], **BoxLeastSquaresPeriodogram._engine_kwargs(prep))
        pg = BoxLeastSquaresPeriodogram._finish(prep, res)
        pg._dy = prep["lc_dy"]
        return pg

    # -- follow-ups ------------------------------------------------------------------------
    def _defaults(self, period, duration, transit_time):
        if period is None:
            period = self.period_at_max_power
            log.warning("No period specified. Using period at max power")
        if duration is None:
            duration = self.duration_at_max_power
            log.warning("No duration specified. Using duration at max power")
        if transit_time is None:
            transit_time = self.transit_time_at_max_power
            log.warning("No transit time specified. Using transit time at max power")
        f = lambda x: float(np.asarray(getattr(x, "value", x)))
        return f(period), f(duration), f(transit_time)

    def compute_stats(self, period=None, duration=None, transit_time=None):
        """Computes commonly used vetting statistics for a transit model (periodogram.py:1194-1229):
        astropy ``BoxLeastSquares.compute_stats`` restated (depth, odd/even/half/phased depths,
        per-transit counts and log-likelihoods, harmonic amplitude / delta log-likelihood).
        A one-off O(N) vetting step for ONE candidate - evaluated on the host."""
        period, duration, transit_time = self._defaults(period, duration, transit_time)
        t_abs = np.asarray(self.time.value, dtype=np.float64)
        tstart = t_abs[0]
        t = t_abs - tstart
        transit_time = transit_time - tstart
        y = np.asarray(self.flux.value, dtype=np.float64)
        dy = getattr(self, "_dy", None)
        ivar = np.ones_like(y) if dy is None else 1.0 / np.asarray(dy, dtype=np.float64) ** 2

        def _compute_depth(m, y_out=None, var_out=None):
            if np.any(m) and (var_out is None or np.isfinite(var_out)):
                var_m = 1.0 / np.sum(ivar[m])
                y_m = np.sum(y[m] * ivar[m]) * var_m
                if y_out is None:
                    return y_m, var_m
                return y_out - y_m, np.sqrt(var_m + var_out)
            return 0.0, np.inf

        hp = 0.5 * period
        m_in = np.abs((t - transit_time + hp) % period - hp) < 0.5 * duration
        m_out = ~m_in
        m_odd = np.abs((t - transit_time) % (2 * period) - period) < 0.5 * duration
        m_even = np.abs((t - transit_time + period) % (2 * period) - period) < 0.5 * duration
        y_out, var_out = _compute_depth(m_out)
        depth = _compute_depth(m_in, y_out, var_out)
        depth_odd = _compute_depth(m_odd, y_out, var_out)
        depth_even = _compute_depth(m_even, y_out, var_out)
        y_in = y_out - depth[0]
        m_phase = np.abs((t - transit_time) % period - hp) < 0.5 * duration
        depth_phase = _compute_depth(m_phase, *_compute_depth((~m_phase) & m_out))
        m_half = np.abs((t - transit_time + 0.25 * period) % (0.5 * period) - 0.25 * period) < 0.5 * duration
        depth_half = _compute_depth(m_half, *_compute_depth(~m_half))

        if m_in.any():
            transit_id = np.round((t[m_in] - transit_time) / period).astype(int)
            transit_times = period * np.arange(transit_id.min(), transit_id.max() + 1) + transit_time
            unique_ids, unique_counts = np.unique(transit_id, return_counts=True)
            unique_ids = unique_ids - np.min(transit_id)
            transit_id = transit_id - np.min(transit_id)
            counts = np.zeros(np.max(transit_id) + 1, dtype=int)
            counts[unique_ids] = unique_counts
            ll = -0.5 * ivar[m_in] * ((y[m_in] - y_in) ** 2 - (y[m_in] - y_out) ** 2)
            lls = np.zeros(len(counts))
            for i in unique_ids:
                lls[i] = np.sum(ll[transit_id == i])
        else:
            transit_times, counts, lls = np.zeros(0), np.zeros(0, dtype=int), np.zeros(0)
        full_ll = -0.5 * np.sum(ivar[m_in] * (y[m_in] - y_in) ** 2)
        full_ll -= 0.5 * np.sum(ivar[m_out] * (y[m_out] - y_out) ** 2)
        A = np.vstack((np.sin(2 * np.pi * t / period), np.cos(2 * np.pi * t / period), np.ones_like(t))).T
        w = np.linalg.solve(np.dot(A.T, A * ivar[:, None]), np.dot(A.T, y * ivar))
        mod = np.dot(A, w)
        sin_ll = -0.5 * np.sum((y - mod) ** 2 * ivar)
        yu = self.flux.unit
        q = lambda pair: (Quantity(pair[0], yu), Quantity(pair[1], yu))
        return dict(
            transit_times=Time(tstart + transit_times, self.time.format, self.time.scale),
            per_transit_count=counts,
            per_transit_log_likelihood=lls,
            depth=q(depth),
            depth_phased=q(depth_phase),
            depth_half=q(depth_half),
            depth_odd=q(depth_odd),
            depth_even=q(depth_even),
            harmonic_amplitude=Quantity(np.sqrt(np.sum(w[:2] ** 2)), yu),
            harmonic_delta_log_likelihood=sin_ll - full_ll,
        )

    def get_transit_model(self, period=None, duration=None, transit_time=None):
        """Box transit model (periodogram.py:1231-1274; astropy BoxLeastSquares.model)."""
        from .lightcurve import LightCurve
        period, duration, transit_time = self._defaults(period, duration, transit_time)
        t = np.asarray(self.time.value, dtype=np.float64)
        y = np.asarray(self.flux.value, dtype=np.float64)
        dy = getattr(self, "_dy", None)
        ivar = np.ones_like(y) if dy is None else 1.0 / np.asarray(dy) ** 2
        hp = 0.5 * period
        m_in = np.abs((t - transit_time + hp) % period - hp) < 0.5 * duration
        m_out = ~m_in
        with np.errstate(divide="ignore", invalid="ignore"):
            y_in = np.sum(y[m_in] * ivar[m_in]) / np.sum(ivar[m_in])
            y_out = np.sum(y[m_out] * ivar[m_out]) / np.sum(ivar[m_out])
        y_model = y_out + np.zeros_like(t)
        y_model[m_in] = y_in
        return LightCurve(time=self.time, flux=Quantity(y_model, self.flux.unit), label="Transit Model Flux")

    def get_transit_mask(self, period=None, duration=None, transit_time=None):
        """True where there are transits (periodogram.py:1276-1296)."""
        model = self.get_transit_model(period=period, duration=duration, transit_time=transit_time)
        mv = np.asarray(model.flux.value)
        return mv != np.median(mv)

    @property
    def transit_time_at_max_power(self):
        return self.transit_time[np.nanargmax(self.power.value)]

    @property
    def duration_at_max_power(self):
        return self.duration[np.nanargmax(self.power.value)]

    @property
    def depth_at_max_power(self):
        return self.depth[np.nanargmax(self.power.value)]

    def flatten(self, **kwargs):
        raise NotImplementedError("`flatten` is not implemented for `BoxLeastSquaresPeriodogram`.")

    def smooth(self, **kwargs):
        raise NotImplementedError("`smooth` is not implemented for `BoxLeastSquaresPeriodogram`. ")
