"""`LightCurveCollection`: /root/reference/src/lightkurve/collections.py:18-276 (list semantics)
plus the batch methods the reference lacks (SURVEY.md F6): ``to_periodogram`` and ``flatten``
over the whole collection in ONE kernel launch sequence.  Their contract is "identical to
``[lc.method(...) for lc in collection]``" - the per-light-curve preparation code is literally
the same functions (``LombScarglePeriodogram._prepare`` etc.); only the device call is batched.
"""
import numpy as np

from .lightcurve import LightCurve

__all__ = ["Collection", "LightCurveCollection"]


class Collection(object):
    """List-like container with numpy-style indexing (collections.py:18-142)."""

    def __init__(self, data):
        if data is not None:
            self.data = [item for item in data]
        else:
            self.data = []

    def __len__(self):
        return len(self.data)

    def __getitem__(self, index_or_mask):
        if isinstance(index_or_mask, (int, np.integer, slice)):
            res = self.data[index_or_mask]
            return type(self)(res) if isinstance(index_or_mask, slice) else res
        if all(isinstance(i, (bool, np.bool_)) for i in index_or_mask):
            if len(index_or_mask) != len(self.data):
                raise IndexError("boolean mask length does not match the collection")
            return type(self)([self.data[i] for i in np.nonzero(index_or_mask)[0]])
        return type(self)([self.data[i] for i in index_or_mask])

    def __setitem__(self, index, obj):
        self.data[index] = obj

    def append(self, obj):
        self.data.append(obj)

    def __iter__(self):
        return iter(self.data)

    def __repr__(self):
        return "{} of {} objects".format(type(self).__name__, len(self.data))


class LightCurveCollection(Collection):
    """Collection of LightCurve objects (collections.py:145-276)."""

    def __init__(self, lightcurves):
        super().__init__(lightcurves)
        for lc in self.data:
            if not isinstance(lc, LightCurve):
                raise TypeError("LightCurveCollection needs LightCurve objects")

    # ---- batched hot path (new API; == per-LC loop) -----------------------------------------
    def to_periodogram(self, method="lombscargle", **kwargs):
        """Batched ``LightCurve.to_periodogram``: returns a list of Periodogram objects."""
        from .periodogram import LombScarglePeriodogram, BoxLeastSquaresPeriodogram
        from .utils import validate_method
        from . import engine
        from . import units as u
        method = validate_method(method.replace(" ", ""), ["ls", "bls", "lombscargle", "boxleastsquares"])
        if len(self.data) == 0:
            return []
        if method in ("bls", "boxleastsquares"):
            preps = [BoxLeastSquaresPeriodogram._prepare(lc, **dict(kwargs)) for lc in self.data]
            p0 = preps[0]
            same = all(np.array_equal(p["period"], p0["period"]) and np.array_equal(p["duration"], p0["duration"])
                       and (p["dy"] is None) == (p0["dy"] is None) for p in preps)
            if not same:
                return [lc.to_periodogram(method, **dict(kwargs)) for lc in self.data]
            res = engine.bls_power([p["time"] for p in preps], [p["flux"] for p in preps],
                                   None if p0["dy"] is None else [p["dy"] for p in preps], p0["period"],
                                   p0["duration"], **BoxLeastSquaresPeriodogram._engine_kwargs(p0))
            out = []
            for b, p in enumerate(preps):
                pg = BoxLeastSquaresPeriodogram._finish(p, res, b)
                pg._dy = p["lc_dy"]
                out.append(pg)
            return out
        preps = [LombScarglePeriodogram._prepare(lc, **dict(kwargs)) for lc in self.data]
        p0 = preps[0]
        norm, _ = LombScarglePeriodogram._norm_args(p0)
        freqs = [np.asarray(p["frequency"].to(1 / u.day).value, dtype=np.float64) for p in preps]
        scales = [LombScarglePeriodogram._norm_args(p)[1] for p in preps]
        shared_t = all(len(p["time"]) == len(p0["time"]) and np.array_equal(p["time"], p0["time"]) for p in preps)
        shared_f = all(len(f) == len(freqs[0]) and np.array_equal(f, freqs[0]) for f in freqs)
        if p0["ls_method"] in ("chi2", "fastchi2", "fastnifty_chi2"):
            fl = [np.asarray(p["lc"].flux.value) for p in preps]
            fl = [f if f.dtype == np.float32 else f.astype(np.float64) for f in fl]
            powers = engine.ls_power_chi2([p["time"] for p in preps], fl, freqs[0] if shared_f else freqs,
                                          p0["nterms"], norm, None if norm != "psd" else scales)
        elif shared_t and shared_f and len(preps) > 1:
            Y = np.stack([np.asarray(p["lc"].flux.value) for p in preps])
            if Y.dtype != np.float32:
                Y = Y.astype(np.float64)
            algo = {"direct": "simt"}.get(LombScarglePeriodogram._engine_algo(p0["ls_method"]),
                                          LombScarglePeriodogram._engine_algo(p0["ls_method"]))
            try:
                powers = engine.ls_power_shared(p0["time"], Y, freqs[0], norm, scales[0], algo=algo)
            except Exception as e:
                if algo != "nufft" or getattr(e, "status", None) != -5:          # LKB_E_UNSUPPORTED
                    raise
                powers = engine.ls_power_shared(p0["time"], Y, freqs[0], norm, scales[0], algo="auto")
        else:
            fl = [np.asarray(p["lc"].flux.value) for p in preps]
            fl = [f if f.dtype == np.float32 else f.astype(np.float64) for f in fl]
            powers = LombScarglePeriodogram._ragged_power(engine, [p["time"] for p in preps], fl,
                                                          freqs[0] if shared_f else freqs, norm,
                                                          None if norm != "psd" else scales, p0["ls_method"])
        return [LombScarglePeriodogram._finish(p, powers[b]) for b, p in enumerate(preps)]

    def flatten(self, window_length=101, polyorder=2, return_trend=False, break_tolerance=5, niters=3, sigma=3,
                mask=None):
        """Batched ``LightCurve.flatten``; `mask` is None or a list of per-LC boolean masks."""
        from . import engine
        if len(self.data) == 0:
            return LightCurveCollection([])
        if polyorder >= window_length:
            polyorder = window_length - 1
        times = [np.asarray(lc.time.value, dtype=np.float64) for lc in self.data]
        fluxes = [np.asarray(lc.flux.value, dtype=np.float64) for lc in self.data]
        errs = [np.asarray(lc.flux_err.value, dtype=np.float64) for lc in self.data]
        masks = None
        if mask is not None:
            masks = [np.zeros(len(t), bool) if m is None else np.asarray(m, dtype=bool) for t, m in zip(times, mask)]
        flat, flat_err, trend = engine.flatten(times, fluxes, errs, masks, window_length=window_length,
                                               polyorder=polyorder, break_tolerance=break_tolerance, niters=niters,
                                               sigma=sigma)
        flats, trends = [], []
        for b, lc in enumerate(self.data):
            dt = lc.flux.dtype if lc.flux.dtype == np.float32 else np.float64
            r = lc._wrap_flatten(flat[b].astype(dt), flat_err[b].astype(dt), trend[b].astype(dt), return_trend)
            if return_trend:
                flats.append(r[0])
                trends.append(r[1])
            else:
                flats.append(r)
        if return_trend:
            return LightCurveCollection(flats), LightCurveCollection(trends)
        return LightCurveCollection(flats)

    def stitch(self, corrector_func=lambda x: x.normalize()):
        """Concatenate the light curves (collections.py:196-230)."""
        from .units import Quantity, Time
        lcs = [corrector_func(lc) for lc in self.data]
        first = lcs[0]
        new = first.copy()
        new.time = Time(np.concatenate([np.asarray(lc.time.value) for lc in lcs]), first.time.format, first.time.scale)
        new.flux = Quantity(np.concatenate([np.asarray(lc.flux.to(first.flux.unit).value) for lc in lcs]),
                            first.flux.unit)
        new.flux_err = Quantity(np.concatenate([np.asarray(lc.flux_err.to(first.flux.unit).value) for lc in lcs]),
                                first.flux.unit)
        return new
