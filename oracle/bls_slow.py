"""Oracle: Box Least Squares ``method="slow"`` as lightkurve reaches it (TEST INFRASTRUCTURE ONLY).

lightkurve passes every extra keyword of ``to_periodogram("bls", ...)`` to astropy's
``BoxLeastSquares.power(period, duration, **kwargs)`` (lightkurve ``periodogram.py:1169``), so
``method="slow"`` selects astropy's exact, unbinned search ``timeseries/periodograms/bls/methods.py::_bls_slow_one``.

PROVENANCE: the loop below is RECALLED from upstream astropy, not read from it - astropy is not
installed where this project is developed and tested (the same standing as SURVEY.md Appendix A.1-A.4).
``tests/test_bls_slow_oracle.py::test_literal_matches_astropy`` pins it wherever astropy imports.
The inputs go through the prologue of ``core.py power()`` (``oracle.bls._prepare``): x = t - min(t),
y - median(y), ivar = 1/dy^2 (ones without errors).

Difference to astropy: a period where no (duration, t0) box has depth > 0 makes astropy fail (it
unpacks a ``None``); here it gets power -inf, depth = depth_err = snr = log_likelihood = duration = 0,
transit_time = min(t), the values K3 leaves for a period without a box, and best index (-1, -1, 0).
"""
import numpy as np

from .bls import RESULT_FIELDS, _prepare, _validate


def _empty_result(P):
    return {k: np.zeros(P) for k in RESULT_FIELDS}, np.tile(np.array([-1, -1, 0], np.int32), (P, 1))


def _finish(out, index, period, t_ref, return_index):
    out["transit_time"] = out["transit_time"] + t_ref
    out["period"] = period
    if return_index:
        out["index"] = index
    return out


def bls_power_slow_numpy(t, y, dy, period, duration, oversample=10, objective="likelihood", return_index=False):
    """Literal restatement of astropy's ``_bls_slow_one`` loop (one O(N) numpy pass per (period, duration, t0)).
    ``index`` [P, 3] = (duration index, t0 index, number of in-box cadences) of the winning box."""
    period, duration = _validate(period, duration)
    x, yc, ivar, t_ref = _prepare(t, y, dy)
    use_likelihood = objective == "likelihood"
    P = len(period)
    out, index = _empty_result(P)
    for p, per in enumerate(period):
        best = -np.inf
        hp = 0.5 * per
        min_t = np.min(x)
        for k, dur in enumerate(duration):
            d_phase = dur / oversample
            phase = np.arange(0, per + d_phase, d_phase)
            for i, t0 in enumerate(phase):
                m_in = np.abs((x - min_t - t0 + hp) % per - hp) < 0.5 * dur
                m_out = ~m_in
                with np.errstate(divide="ignore", invalid="ignore"):
                    ivar_in = np.sum(ivar[m_in])
                    ivar_out = np.sum(ivar[m_out])
                    y_in = np.sum(yc[m_in] * ivar[m_in]) / ivar_in
                    y_out = np.sum(yc[m_out] * ivar[m_out]) / ivar_out
                    depth = y_out - y_in
                    depth_err = np.sqrt(1.0 / ivar_in + 1.0 / ivar_out)
                    snr = depth / depth_err
                    loglike = -0.5 * np.sum((y_in - yc[m_in]) ** 2 * ivar[m_in])
                    loglike += 0.5 * np.sum((y_out - yc[m_in]) ** 2 * ivar[m_in])
                obj = loglike if use_likelihood else snr
                if depth > 0 and obj > best:
                    best = obj
                    out["power"][p] = obj
                    out["depth"][p] = depth
                    out["depth_err"][p] = depth_err
                    out["duration"][p] = dur
                    out["transit_time"][p] = (t0 + min_t) % per
                    out["depth_snr"][p] = snr
                    out["log_likelihood"][p] = loglike
                    index[p] = (k, i, int(np.count_nonzero(m_in)))
        if best == -np.inf:
            out["power"][p] = -np.inf
    return _finish(out, index, period, t_ref, return_index)


def objective_at_slow(t, y, dy, period, dur, t0_index, oversample=10, objective="likelihood", return_count=False):
    """Objective of ONE box (trial duration `dur`, epoch t0 = t0_index * dur / oversample) at ONE period, in the
    literal oracle's arithmetic.  The parity tests use it to recognise boxes that tie with the oracle's winner."""
    x, yc, ivar, _ = _prepare(t, y, dy)
    per, dur = np.float64(period), np.float64(dur)
    d_phase = dur / oversample
    t0 = np.arange(0, per + d_phase, d_phase)[t0_index]
    hp = 0.5 * per
    m_in = np.abs((x - np.min(x) - t0 + hp) % per - hp) < 0.5 * dur
    m_out = ~m_in
    with np.errstate(divide="ignore", invalid="ignore"):
        ivar_in, ivar_out = np.sum(ivar[m_in]), np.sum(ivar[m_out])
        y_in = np.sum(yc[m_in] * ivar[m_in]) / ivar_in
        y_out = np.sum(yc[m_out] * ivar[m_out]) / ivar_out
        if objective == "snr":
            val = (y_out - y_in) / np.sqrt(1.0 / ivar_in + 1.0 / ivar_out)
        else:
            val = -0.5 * np.sum((y_in - yc[m_in]) ** 2 * ivar[m_in])
            val += 0.5 * np.sum((y_out - yc[m_in]) ** 2 * ivar[m_in])
    if return_count:
        return val, int(np.count_nonzero(m_in))
    return val


def _in_box(xv, t0, hp, per, half):
    """The literal predicate, elementwise (x - min(x) = x since min(x) = 0)."""
    return np.abs((xv - t0 + hp) % per - hp) < half


def bls_power_slow_vec(t, y, dy, period, duration, oversample=10, objective="likelihood", return_index=False):
    """The same search, vectorised over (t0, cycle): for medium sizes (a few 1e4 cadences x a few 100 periods).

    For each box and each cycle c (window centre xc = t0 + c P) the in-box cadences of ascending times form one run;
    its ends are found by binary search with a margin of 1e-9 (P + baseline) days on either side of each window end,
    and every cadence inside a margin is decided by the literal predicate.  The run's sums are differences of prefix
    sums, added over the cycles in increasing order (so boxes with the same member cadences get bitwise equal sums).
    Raises AssertionError if a margin holds members that are not contiguous with the run."""
    period, duration = _validate(period, duration)
    x, yc, ivar, t_ref = _prepare(t, y, dy)
    order = np.argsort(x, kind="stable")
    x, yc, ivar = x[order], yc[order], ivar[order]
    n = len(x)
    x_max = x[-1]
    cy = np.concatenate([[0.0], np.cumsum(yc * ivar)])
    ci = np.concatenate([[0.0], np.cumsum(ivar)])
    sum_y, sum_ivar = np.sum(yc * ivar), np.sum(ivar)
    use_snr = objective == "snr"
    P = len(period)
    out, index = _empty_result(P)
    for p, per in enumerate(period):
        best = -np.inf
        hp = 0.5 * per
        margin = 1e-9 * (per + x_max)
        for k, dur in enumerate(duration):
            d_phase = dur / oversample
            t0 = np.arange(0, per + d_phase, d_phase)
            half = 0.5 * dur
            c = np.arange(np.floor((-hp - t0[-1]) / per) - 1, np.ceil((x_max + hp) / per) + 2)
            xc = t0[:, None] + c[None, :] * per
            T0 = np.broadcast_to(t0[:, None], xc.shape)
            lo_out = np.searchsorted(x, xc - half - margin, "left")
            lo_in = np.searchsorted(x, xc - half + margin, "left")
            hi_in = np.searchsorted(x, xc + half - margin, "left")
            hi_out = np.searchsorted(x, xc + half + margin, "left")
            # lower margin: out ... out in ... in  -> the run starts at the first member
            lo = lo_in.copy()
            found = np.zeros(xc.shape, bool)
            for j in range(int(np.max(lo_in - lo_out, initial=0))):
                idx = lo_out + j
                valid = idx < lo_in
                pv = valid & _in_box(x[np.minimum(idx, n - 1)], T0, hp, per, half)
                assert not np.any(found & valid & ~pv), "members of a lower margin are not contiguous"
                lo = np.where(pv & ~found, idx, lo)
                found |= pv
            # upper margin: in ... in out ... out
            hi = hi_in.copy()
            open_ = np.ones(xc.shape, bool)
            for j in range(int(np.max(hi_out - hi_in, initial=0))):
                idx = hi_in + j
                valid = idx < hi_out
                pv = valid & _in_box(x[np.minimum(idx, n - 1)], T0, hp, per, half)
                assert not np.any(~open_ & pv), "members of an upper margin are not contiguous"
                hi = np.where(pv & open_, idx + 1, hi)
                open_ &= ~(valid & ~pv)
            s_y = np.zeros(len(t0))
            s_i = np.zeros(len(t0))
            for j in range(xc.shape[1]):               # cycles in increasing order, like the kernel
                s_y += cy[hi[:, j]] - cy[lo[:, j]]
                s_i += ci[hi[:, j]] - ci[lo[:, j]]
            cnt = np.sum(hi - lo, axis=1)
            yw_out, i_out = sum_y - s_y, sum_ivar - s_i
            full = cnt == n
            yw_out[full] = 0.0
            i_out[full] = 0.0
            with np.errstate(divide="ignore", invalid="ignore"):
                depth = yw_out / i_out - s_y / s_i
                depth_err = np.sqrt(1.0 / s_i + 1.0 / i_out)
                snr = depth / depth_err
                ll = 0.5 * s_i * depth * depth
            obj = np.where(depth > 0, snr if use_snr else ll, -np.inf)
            i = int(np.argmax(obj))                     # first maximum
            if obj[i] > best:
                best = obj[i]
                out["power"][p] = obj[i]
                out["depth"][p] = depth[i]
                out["depth_err"][p] = depth_err[i]
                out["duration"][p] = dur
                out["transit_time"][p] = t0[i] % per
                out["depth_snr"][p] = snr[i]
                out["log_likelihood"][p] = ll[i]
                index[p] = (k, i, cnt[i])
        if best == -np.inf:
            out["power"][p] = -np.inf
    return _finish(out, index, period, t_ref, return_index)
