"""Batched host-side entry points over the C ABI (``include/lkb200.h``).

Every function takes either host ``numpy`` arrays (the library stages them through
its device workspace; the call is synchronous) or CUDA ``torch`` tensors (raw device
pointers are handed over; the call is asynchronous on the current torch stream).
PyTorch is only the allocator / stream provider here - no torch op is on the
compute path.  No CPU fallback exists: without the built library or without a GPU
these functions raise.
"""
import numpy as np

from . import _lib as L

_NORMS = {"psd_raw": L.LS_NORM_PSD_RAW, "psd": L.LS_NORM_PSD_SCALE, "amplitude": L.LS_NORM_AMPLITUDE}
_ALGOS = {"auto": L.LS_ALGO_AUTO, "simt": L.LS_ALGO_SIMT, "tcgen05": L.LS_ALGO_TCGEN05, "nufft": L.LS_ALGO_NUFFT}


def _is_torch(x):
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda")


def _stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def device_count():
    return L.load().lkb_device_count()


def init(device=0):
    """Bind this process to one GPU (one process per GPU, like torch.distributed ranks)."""
    L.check(L.load().lkb_init(int(device)))


def shutdown():
    L.check(L.load().lkb_shutdown())


def launch_count():
    return int(L.load().lkb_launch_count())


def ls_last_algo():
    """Kernel family the most recent Lomb-Scargle call ran: "simt" (direct sums), "tcgen05" or "nufft"."""
    return {L.LS_ALGO_SIMT: "simt", L.LS_ALGO_TCGEN05: "tcgen05", L.LS_ALGO_NUFFT: "nufft"}.get(
        int(L.load().lkb_ls_last_algo()), "none")


def ls_last_escalated():
    """Light curves of the most recent shared-grid NUFFT call that took the double-precision pass (lkb200.h)."""
    return int(L.load().lkb_ls_last_escalated())


def profile_enable(on=True):
    """Record CUDA events around the dominant kernel of each subsequent call (see lkb200.h)."""
    L.check(L.load().lkb_profile_enable(1 if on else 0))


def profile_read(max_n=512):
    """Durations [ms] of the dominant kernels launched since profile_enable / the last read."""
    buf = np.zeros(max_n, dtype=np.float64)
    n = L.load().lkb_profile_read(L.ptr(buf), max_n)
    if n < 0:
        L.check(n)
    return buf[:n].copy()


# workspace slot numbers (enum Slot in csrc/common.cuh) for the diagnostic read-back
WS_SLOTS = {name: i for i, name in enumerate(
    ["A", "B", "C", "D", "E", "F", "G", "H", "I", "J", "K", "L", "M", "N", "O", "P"]
    + ["IN%d" % i for i in range(8)] + ["OUT%d" % i for i in range(8)] + ["X%d" % i for i in range(8)] + ["Y%d" % i for i in range(8)])}


def ws_read(slot, count, dtype, offset_bytes=0):
    """Diagnostic: `count` items of `dtype` from workspace slot `slot` ("A".."P", "IN0".., "OUT0"..) as left by
    the last call (device synchronised first)."""
    out = np.empty(count, dtype=dtype)
    L.check(L.load().lkb_ws_read(WS_SLOTS[slot], int(offset_bytes), int(out.nbytes), L.ptr(out)))
    return out


def sm_count():
    return int(L.load().lkb_sm_count())


def _csr(arrays, dtype=np.float64):
    lens = [len(a) for a in arrays]
    offsets = np.zeros(len(arrays) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    cat = np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=dtype) for a in arrays])) if arrays else \
        np.zeros(0, dtype)
    return cat, offsets


def _y_dtype_code(dt):
    if dt == np.float32:
        return L.DTYPE_F32
    if dt == np.float64:
        return L.DTYPE_F64
    raise TypeError("flux must be float32 or float64")


# --------------------------------------------------------------------------------------
# Lomb-Scargle
# --------------------------------------------------------------------------------------
_RAGGED_ALGOS = {"auto": L.LS_ALGO_AUTO, "direct": L.LS_ALGO_SIMT, "simt": L.LS_ALGO_SIMT, "nufft": L.LS_ALGO_NUFFT}


def ls_power_ragged(times, fluxes, frequency, normalization="amplitude", norm_scale=None, algo="auto"):
    """K1.  `times`/`fluxes`: lists of 1-D arrays (one per light curve, no NaNs).
    `frequency`: one 1-D grid shared by all light curves, or a list of per-LC grids.
    `algo`: "auto" (the NUFFT kernels for a large job on one shared regular grid with sorted times, else the direct
    sums), "direct" (always the exact direct sums - astropy method="slow") or "nufft" (raises when the grid or the
    times do not qualify - the reference's ls_method="fastnifty").
    Returns a [B, F] float32 array (shared grid) or a list of float32 arrays."""
    lib = L.load()
    B = len(times)
    if B == 0:
        return []
    if algo not in _RAGGED_ALGOS:
        raise ValueError("algo must be one of %s" % sorted(_RAGGED_ALGOS))
    t, offsets = _csr(times)
    ydt = np.float32 if all(np.asarray(f).dtype == np.float32 for f in fluxes) else np.float64
    y, yoff = _csr(fluxes, ydt)
    if not np.array_equal(offsets, yoff):
        raise ValueError("time and flux lengths differ")
    per_lc = isinstance(frequency, (list, tuple))
    if per_lc:
        freq, foff = _csr(frequency)
        F = 0
        out = np.empty(int(foff[-1]), dtype=np.float32)
    else:
        freq = np.ascontiguousarray(frequency, dtype=np.float64)
        foff = None
        F = len(freq)
        out = np.empty((B, F), dtype=np.float32)
    ns = None if norm_scale is None else np.ascontiguousarray(np.broadcast_to(norm_scale, (B,)), dtype=np.float64)
    L.check(lib.lkb_ls_power_ex(L.ptr(t), L.ptr(y), _y_dtype_code(ydt), L.ptr(offsets), B, L.ptr(freq), L.ptr(foff), F,
                                _NORMS[normalization], L.ptr(ns), L.ptr(out), L.MEM_HOST, None, _RAGGED_ALGOS[algo]))
    if per_lc:
        return [out[foff[b]:foff[b + 1]] for b in range(B)]
    return out


def ls_power_ragged_device(t_cat, y_cat, offsets, frequency, normalization="amplitude", norm_scale=None, algo="auto",
                           out=None):
    """K1 with DEVICE-resident inputs: `t_cat` (float64) and `y_cat` (float32 / float64) are CUDA torch tensors
    holding the light curves back to back, `offsets` the int64 [B + 1] CSR boundaries (host metadata, numpy),
    `frequency` a CUDA float64 tensor [F] shared by all light curves, `norm_scale` None or a CUDA float64 [B].
    Returns a CUDA float32 [B, F] tensor (`out` if given).  The kernels run on the current torch stream; the call
    synchronises that stream for its metadata read-backs."""
    import torch
    lib = L.load()
    if algo not in _RAGGED_ALGOS:
        raise ValueError("algo must be one of %s" % sorted(_RAGGED_ALGOS))
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    B = len(offsets) - 1
    if B <= 0:
        raise ValueError("empty batch")
    for name, x in (("t_cat", t_cat), ("y_cat", y_cat), ("frequency", frequency)):
        if not (_is_torch(x) and x.is_cuda and x.is_contiguous() and x.dim() == 1):
            raise ValueError("%s must be a contiguous one-dimensional CUDA tensor" % name)
    if t_cat.dtype != torch.float64 or frequency.dtype != torch.float64:
        raise TypeError("t_cat and frequency must be float64")
    if y_cat.dtype not in (torch.float32, torch.float64):
        raise TypeError("flux must be float32 or float64, not %s" % (y_cat.dtype,))
    if offsets[0] != 0 or np.any(np.diff(offsets) < 0) or t_cat.numel() != offsets[-1] or y_cat.numel() != offsets[-1]:
        raise ValueError("offsets do not describe t_cat / y_cat")
    F = frequency.numel()
    if out is None:
        out = torch.empty((B, F), dtype=torch.float32, device=y_cat.device)
    elif not (_is_torch(out) and out.is_cuda and out.dtype == torch.float32 and tuple(out.shape) == (B, F)
              and out.is_contiguous()):
        raise ValueError("`out` must be a contiguous CUDA float32 tensor of shape (%d, %d)" % (B, F))
    if norm_scale is not None and not (_is_torch(norm_scale) and norm_scale.is_cuda and
                                       norm_scale.dtype == torch.float64 and norm_scale.numel() == B):
        raise ValueError("norm_scale must be a CUDA float64 tensor with one entry per light curve")
    ycode = L.DTYPE_F32 if y_cat.dtype == torch.float32 else L.DTYPE_F64
    L.check(lib.lkb_ls_power_ex(L.ptr(t_cat), L.ptr(y_cat), ycode, L.ptr(offsets), B, L.ptr(frequency), None, F,
                                _NORMS[normalization], L.ptr(norm_scale), L.ptr(out), L.MEM_DEVICE, _stream_ptr(),
                                _RAGGED_ALGOS[algo]))
    return out


def ls_power_chi2(times, fluxes, frequency, nterms=1, normalization="amplitude", norm_scale=None,
                  return_theta=False):
    """K1n.  Multi-term periodogram (astropy method="chi2"/"fastchi2", nterms in [1, 4]); same
    arguments as ls_power_ragged.  With return_theta also returns the 2*nterms+1 fitted parameters
    per (light curve, frequency): [offset, sin 1, cos 1, sin 2, cos 2, ...]."""
    lib = L.load()
    B = len(times)
    if B == 0:
        return []
    t, offsets = _csr(times)
    ydt = np.float32 if all(np.asarray(f).dtype == np.float32 for f in fluxes) else np.float64
    y, yoff = _csr(fluxes, ydt)
    if not np.array_equal(offsets, yoff):
        raise ValueError("time and flux lengths differ")
    M = 2 * int(nterms) + 1
    per_lc = isinstance(frequency, (list, tuple))
    if per_lc:
        freq, foff = _csr(frequency)
        F = 0
        out = np.empty(int(foff[-1]), dtype=np.float32)
        theta = np.empty((int(foff[-1]), M), dtype=np.float64) if return_theta else None
    else:
        freq = np.ascontiguousarray(frequency, dtype=np.float64)
        foff = None
        F = len(freq)
        out = np.empty((B, F), dtype=np.float32)
        theta = np.empty((B, F, M), dtype=np.float64) if return_theta else None
    ns = None if norm_scale is None else np.ascontiguousarray(np.broadcast_to(norm_scale, (B,)), dtype=np.float64)
    L.check(lib.lkb_ls_power_chi2(L.ptr(t), L.ptr(y), _y_dtype_code(ydt), L.ptr(offsets), B, L.ptr(freq), L.ptr(foff),
                                  F, int(nterms), _NORMS[normalization], L.ptr(ns), L.ptr(out), L.ptr(theta),
                                  L.MEM_HOST, None))
    if per_lc:
        out = [out[foff[b]:foff[b + 1]] for b in range(B)]
        if return_theta:
            theta = [theta[foff[b]:foff[b + 1]] for b in range(B)]
    return (out, theta) if return_theta else out


def ls_power_shared(t, Y, frequency, normalization="amplitude", norm_scale=None, algo="auto", out=None):
    """K2.  One cadence grid `t` [N] shared by the batch `Y` [B, N]; `frequency` [F].
    numpy in -> numpy out (host mode); CUDA torch tensors in -> torch tensor out (device mode: the kernels are
    enqueued on the current torch stream, but the call itself synchronises that stream once for a small metadata
    read-back, and the library's grow-only workspaces are shared by all calls - use ONE stream per process).
    `algo`: "auto" (the spread + FFT path of DESIGN.md K2n when the grid is regular with integer f0/df,
    df * baseline <= 1 and the times ascend; else the tcgen05 tensor path when the shape allows; else the CUDA-core
    contraction), "simt", "tcgen05", or "nufft" (raises for grids / times it does not support)."""
    lib = L.load()
    if algo not in _ALGOS:
        raise ValueError("algo must be one of %s" % sorted(_ALGOS))
    if _is_torch(Y):
        import torch
        if not (_is_torch(t) and _is_torch(frequency) and Y.is_cuda and t.is_cuda and frequency.is_cuda):
            raise ValueError("device mode needs CUDA tensors for t, Y and frequency")
        if Y.dim() != 2 or t.dim() != 1 or frequency.dim() != 1:
            raise ValueError("Y must be [B, N], t [N] and frequency [F]")
        B, N = Y.shape
        F = frequency.numel()
        if t.numel() != N:
            raise ValueError("t has %d cadences but Y has %d columns" % (t.numel(), N))
        if t.dtype != torch.float64 or frequency.dtype != torch.float64:
            raise TypeError("t and frequency must be float64")
        if Y.dtype not in (torch.float32, torch.float64):
            raise TypeError("flux must be float32 or float64, not %s" % (Y.dtype,))
        if not (Y.is_contiguous() and t.is_contiguous() and frequency.is_contiguous()):
            raise ValueError("t, Y and frequency must be contiguous")
        ycode = L.DTYPE_F32 if Y.dtype == torch.float32 else L.DTYPE_F64
        if out is None:
            out = torch.empty((B, F), dtype=torch.float32, device=Y.device)
        elif not (_is_torch(out) and out.is_cuda and out.device == Y.device and out.dtype == torch.float32
                  and tuple(out.shape) == (B, F) and out.is_contiguous()):
            raise ValueError("`out` must be a contiguous CUDA float32 tensor of shape (%d, %d) on %s" % (B, F, Y.device))
        ns = None
        if norm_scale is not None:
            ns = torch.tensor([float(norm_scale)], dtype=torch.float64, device=Y.device)
        L.check(lib.lkb_ls_power_shared(L.ptr(t), L.ptr(Y), ycode, int(B), int(N), L.ptr(frequency), int(F),
                                        _NORMS[normalization], L.ptr(ns), L.ptr(out), L.MEM_DEVICE, _stream_ptr(),
                                        _ALGOS[algo]))
        return out
    t = np.ascontiguousarray(t, dtype=np.float64)
    Y = np.ascontiguousarray(Y)
    if Y.dtype not in (np.float32, np.float64):
        Y = Y.astype(np.float64)
    if Y.ndim != 2 or t.ndim != 1:
        raise ValueError("Y must be [B, N] and t [N]")
    B, N = Y.shape
    if t.shape != (N,):
        raise ValueError("t has %d cadences but Y has %d columns" % (len(t), N))
    freq = np.ascontiguousarray(frequency, dtype=np.float64)
    if freq.ndim != 1:
        raise ValueError("frequency must be one-dimensional")
    if out is None:
        out = np.empty((B, len(freq)), dtype=np.float32)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.shape == (B, len(freq))
              and out.flags.c_contiguous and out.flags.writeable):
        raise ValueError("`out` must be a writeable C-contiguous float32 array of shape (%d, %d)" % (B, len(freq)))
    ns = None if norm_scale is None else np.array([float(norm_scale)], dtype=np.float64)
    L.check(lib.lkb_ls_power_shared(L.ptr(t), L.ptr(Y), _y_dtype_code(Y.dtype), B, N, L.ptr(freq), len(freq),
                                    _NORMS[normalization], L.ptr(ns), L.ptr(out), L.MEM_HOST, None, _ALGOS[algo]))
    return out


# --------------------------------------------------------------------------------------
# Box Least Squares
# --------------------------------------------------------------------------------------
BLS_FIELDS = ("power", "depth", "depth_err", "duration", "transit_time", "depth_snr", "log_likelihood")


def bls_power(times, fluxes, flux_errs, period, duration, oversample=10, objective="likelihood",
              return_bins=False, method="fast"):
    """K3 (method="fast", astropy's binned search) or K3s (method="slow", astropy's exact unbinned search; the times
    of every light curve must be ascending).  Lists of per-LC arrays (flux_errs: list or None => unit weights), one
    shared period grid [P] and duration grid [D].  Returns dict of [B, P] float64 arrays; with `return_bins`, also
    "bins" [B, P, 2] = (start bin, duration in bins) for "fast" or "index" [B, P, 3] = (duration index, t0 index,
    number of in-box cadences) for "slow"."""
    if method not in ("fast", "slow"):
        raise ValueError("method must be 'fast' or 'slow' (got %r)" % (method,))
    lib = L.load()
    B = len(times)
    t, offsets = _csr(times)
    y, yoff = _csr(fluxes)
    if not np.array_equal(offsets, yoff):
        raise ValueError("time and flux lengths differ")
    dy = None
    if flux_errs is not None:
        dy, doff = _csr(flux_errs)
        if not np.array_equal(offsets, doff):
            raise ValueError("time and flux_err lengths differ")
    period = np.ascontiguousarray(np.atleast_1d(period), dtype=np.float64)
    duration = np.ascontiguousarray(np.atleast_1d(duration), dtype=np.float64)
    P, D = len(period), len(duration)
    outs = [np.empty((B, P), dtype=np.float64) for _ in range(7)]
    if method == "slow":
        index = np.empty((B, P, 3), dtype=np.int32) if return_bins else None
        L.check(lib.lkb_bls_power_slow(L.ptr(t), L.ptr(y), L.ptr(dy), L.ptr(offsets), B, L.ptr(period), P,
                                       L.ptr(duration), D, int(oversample),
                                       L.BLS_SNR if objective == "snr" else L.BLS_LIKELIHOOD,
                                       *[L.ptr(o) for o in outs], L.ptr(index), L.MEM_HOST, None))
    else:
        bins = np.empty((B, P, 2), dtype=np.int32) if return_bins else None
        L.check(lib.lkb_bls_power(L.ptr(t), L.ptr(y), L.ptr(dy), L.ptr(offsets), B, L.ptr(period), P, L.ptr(duration),
                                  D, int(oversample), L.BLS_SNR if objective == "snr" else L.BLS_LIKELIHOOD,
                                  *[L.ptr(o) for o in outs], L.ptr(bins), L.MEM_HOST, None))
    res = dict(zip(BLS_FIELDS, outs))
    res["period"] = period
    if return_bins:
        if method == "slow":
            res["index"] = index
        else:
            res["bins"] = bins
    return res


def bls_bin_index(t_rel, min_t, period, bin_duration):
    lib = L.load()
    t_rel = np.ascontiguousarray(t_rel, dtype=np.float64)
    out = np.empty(len(t_rel), dtype=np.int32)
    L.check(lib.lkb_bls_bin_index(L.ptr(t_rel), len(t_rel), float(min_t), float(period), float(bin_duration),
                                  L.ptr(out), L.MEM_HOST, None))
    return out


# --------------------------------------------------------------------------------------
# flatten
# --------------------------------------------------------------------------------------
def flatten_csr(t, f, fe, exclude, offsets, window_length=101, polyorder=2, break_tolerance=5, niters=3, sigma=3,
                flat=None, flat_err=None, trend=None):
    """K4 on already concatenated host arrays (CSR `offsets` [B + 1]): `t`, `f`, `fe` (or None) float64 [total],
    `exclude` uint8 [total] or None (1 = leave the cadence out of the fit).  Output arrays may be passed in (e.g.
    page-locked buffers).  Returns (flat, flat_err, trend) float64 [total]."""
    lib = L.load()
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    B = len(offsets) - 1
    total = int(offsets[-1])
    for name, a in (("t", t), ("f", f), ("fe", fe)):
        if a is not None and not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.shape == (total,)
                                  and a.flags.c_contiguous):
            raise ValueError("%s must be a C-contiguous float64 array of %d cadences" % (name, total))
    if exclude is not None and not (isinstance(exclude, np.ndarray) and exclude.dtype == np.uint8
                                    and exclude.shape == (total,) and exclude.flags.c_contiguous):
        raise ValueError("exclude must be a C-contiguous uint8 array of %d cadences" % total)
    outs = []
    for name, a in (("flat", flat), ("flat_err", flat_err), ("trend", trend)):
        if a is None:
            a = np.empty(total, dtype=np.float64)
        elif not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.shape == (total,) and a.flags.c_contiguous
                  and a.flags.writeable):
            raise ValueError("%s must be a writeable C-contiguous float64 array of %d cadences" % (name, total))
        outs.append(a)
    flat, flat_err, trend = outs
    bt = np.nan if break_tolerance is None else float(break_tolerance)
    L.check(lib.lkb_flatten(L.ptr(t), L.ptr(f), L.ptr(fe), L.ptr(exclude), L.ptr(offsets), B, int(window_length),
                            int(polyorder), bt, int(niters), float(sigma), L.ptr(flat), L.ptr(flat_err),
                            L.ptr(trend), L.MEM_HOST, None))
    return flat, flat_err, trend


def flatten(times, fluxes, flux_errs=None, masks=None, window_length=101, polyorder=2, break_tolerance=5,
            niters=3, sigma=3):
    """K4.  Lists of per-LC arrays.  `masks`: list of bool arrays, True = exclude (lightkurve
    semantics) or None.  Returns (flat, flat_err, trend) as lists of float64 arrays."""
    B = len(times)
    t, offsets = _csr(times)
    f, foff = _csr(fluxes)
    if not np.array_equal(offsets, foff):
        raise ValueError("time and flux lengths differ")
    fe = None
    if flux_errs is not None:
        fe, eoff = _csr(flux_errs)
        if not np.array_equal(offsets, eoff):
            raise ValueError("time and flux_err lengths differ")
    ex = None
    if masks is not None:
        if len(masks) != B or any(len(m) != len(tt) for m, tt in zip(masks, times)):
            raise ValueError("time and mask lengths differ")
        ex = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=bool) for m in masks]).astype(np.uint8))
    flat, flat_err, trend = flatten_csr(t, f, fe, ex, offsets, window_length, polyorder, break_tolerance, niters, sigma)
    sp = lambda a: [a[offsets[b]:offsets[b + 1]] for b in range(B)]
    return sp(flat), sp(flat_err), sp(trend)


# --------------------------------------------------------------------------------------
# regression
# --------------------------------------------------------------------------------------
def regress(X, Y, flux_err=None, cadence_mask=None, prior_mu=None, prior_sigma=None, sigma=5, niters=5,
            return_cov=False):
    """K5.  X [N, K] (shared) or [B, N, K]; Y [B, N]; flux_err [B, N] or None (ones);
    cadence_mask bool [B, N] or None.  Returns dict(coefficients [B,K], model [B,N]
    (median-subtracted), outlier_mask bool [B,N], status int32 [B])."""
    lib = L.load()
    X = np.ascontiguousarray(X, dtype=np.float64)
    Y = np.ascontiguousarray(np.atleast_2d(Y), dtype=np.float64)
    B, N = Y.shape
    batched = X.ndim == 3
    K = X.shape[-1]
    if X.shape[-2] != N or (batched and X.shape[0] != B):
        raise ValueError("X shape %s does not match Y shape %s" % (X.shape, Y.shape))
    fe = None if flux_err is None else np.ascontiguousarray(np.broadcast_to(flux_err, Y.shape), dtype=np.float64)
    cm = None if cadence_mask is None else \
        np.ascontiguousarray(np.broadcast_to(np.asarray(cadence_mask, dtype=bool), Y.shape).astype(np.uint8))
    pm = None if prior_mu is None else np.ascontiguousarray(prior_mu, dtype=np.float64)
    ps = None if prior_sigma is None else np.ascontiguousarray(prior_sigma, dtype=np.float64)
    coeff = np.empty((B, K), dtype=np.float64)
    model = np.empty((B, N), dtype=np.float64)
    om = np.empty((B, N), dtype=np.uint8)
    status = np.empty(B, dtype=np.int32)
    cov = np.empty((B, K, K), dtype=np.float64) if return_cov else None
    L.check(lib.lkb_regress(L.ptr(X), 1 if batched else 0, L.ptr(Y), L.ptr(fe), L.ptr(cm), L.ptr(pm), L.ptr(ps),
                            B, N, K, float(sigma), int(niters), L.ptr(coeff), L.ptr(model), L.ptr(om),
                            L.ptr(status), L.ptr(cov), L.MEM_HOST, None))
    out = dict(coefficients=coeff, model=model, outlier_mask=om.astype(bool), status=status)
    if return_cov:
        out["covariance"] = cov
    return out


def nanmedian_std(arrays):
    """K6.  np.nanmedian and np.nanstd of each array."""
    lib = L.load()
    x, offsets = _csr(arrays)
    B = len(arrays)
    med = np.empty(B, dtype=np.float64)
    sd = np.empty(B, dtype=np.float64)
    L.check(lib.lkb_nanmedian_std(L.ptr(x), L.ptr(offsets), B, L.ptr(med), L.ptr(sd), L.MEM_HOST, None))
    return med, sd


def logmedian_windows(frequency, filter_width):
    """Half-open bin ranges of the reference's moving log10-frequency window (periodogram.py:267-277) for an
    ASCENDING frequency grid: window w = { i : |log10 f_i - x0_w| < filter_width }, x0 advancing by
    filter_width / 2 from log10 f_0 (the same fp64 accumulation).  Empty windows are kept (they add nothing)."""
    logf = np.log10(np.asarray(frequency, dtype=np.float64))
    F = len(logf)
    x0s = []
    x0 = logf[0]
    while x0 < logf[-1]:
        x0s.append(x0)
        x0 += 0.5 * filter_width
    x0s = np.asarray(x0s, dtype=np.float64)
    lo = np.searchsorted(logf, x0s - filter_width, side="right")
    hi = np.searchsorted(logf, x0s + filter_width, side="left")
    # the reference's expression is |logf - x0| < w in fp64: settle the edge bins with exactly that
    inside = lambda i, c: np.abs(logf[np.clip(i, 0, F - 1)] - c) < filter_width
    for _ in range(3):
        grow = (lo > 0) & inside(lo - 1, x0s)
        lo = np.where(grow, lo - 1, lo)
        shrink = (lo < hi) & ~inside(lo, x0s)
        lo = np.where(shrink, lo + 1, lo)
        grow = (hi < F) & inside(hi, x0s)
        hi = np.where(grow, hi + 1, hi)
        shrink = (hi > lo) & ~inside(hi - 1, x0s)
        hi = np.where(shrink, hi - 1, hi)
    return lo.astype(np.int32), np.maximum(hi, lo).astype(np.int32)


def pg_logmedian(frequency, power, filter_width):
    """Background of B periodograms on one frequency grid (Periodogram.smooth(method="logmedian")).
    power [B, F] (or [F]); returns the same shape, fp64."""
    lib = L.load()
    freq = np.asarray(frequency, dtype=np.float64)
    p = np.asarray(power, dtype=np.float64)
    one = p.ndim == 1
    p = np.ascontiguousarray(np.atleast_2d(p))
    B, F = p.shape
    if len(freq) != F:
        raise ValueError("frequency and power must have the same length")
    order = None
    if F > 1 and not np.all(np.diff(freq) >= 0):
        order = np.argsort(freq, kind="stable")
        freq, p = freq[order], np.ascontiguousarray(p[:, order])
    lo, hi = logmedian_windows(freq, filter_width)
    out = np.empty((B, F), dtype=np.float64)
    if len(lo) == 0:
        out[:] = np.nan
    else:
        lo, hi = np.ascontiguousarray(lo), np.ascontiguousarray(hi)
        L.check(lib.lkb_pg_logmedian(L.ptr(p), B, F, L.ptr(lo), L.ptr(hi), len(lo), (8.0 / 9.0) ** 3, L.ptr(out),
                                     L.MEM_HOST, None))
    if order is not None:
        inv = np.empty_like(order)
        inv[order] = np.arange(F)
        out = out[:, inv]
    return out[0] if one else out


# --------------------------------------------------------------------------------------
# multi-GPU exchange step (SURVEY.md 8e): NCCL all-gather through the C ABI
# --------------------------------------------------------------------------------------
def nccl_version():
    """NCCL_VERSION_CODE of the library the C ABI bound at run time (0: none could be loaded)."""
    return int(L.load().lkb_nccl_version())


def nccl_unique_id():
    """128-byte NCCL id (bytes).  Rank 0 creates it; the host program carries it to the other ranks."""
    buf = np.zeros(L.NCCL_ID_BYTES, dtype=np.uint8)
    L.check(L.load().lkb_nccl_unique_id(L.ptr(buf)))
    return buf.tobytes()


def nccl_init(rank, world_size, unique_id):
    """Collective: every rank calls this with the SAME id after ``init(device)``."""
    buf = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy()
    if buf.size != L.NCCL_ID_BYTES:
        raise ValueError("an NCCL unique id has %d bytes, got %d" % (L.NCCL_ID_BYTES, buf.size))
    L.check(L.load().lkb_nccl_init(int(rank), int(world_size), L.ptr(buf)))


def nccl_shutdown():
    L.check(L.load().lkb_nccl_shutdown())


def nccl_rank_world():
    lib = L.load()
    return int(lib.lkb_nccl_rank()), int(lib.lkb_nccl_world_size())


def allgather_f32(local, out=None):
    """One ncclAllGather of a contiguous CUDA float32 torch tensor `local` ([n, ...], same shape on every
    rank) into `out` ([world * n, ...], rank-major), asynchronous on the current torch stream."""
    import torch
    lib = L.load()
    world = int(lib.lkb_nccl_world_size())
    if world <= 0:
        raise ValueError("allgather_f32: no communicator (call engine.nccl_init on every rank first)")
    if not (_is_torch(local) and local.is_cuda and local.dtype == torch.float32 and local.is_contiguous()):
        raise TypeError("allgather_f32 needs a contiguous CUDA float32 tensor")
    shape = (world * local.shape[0],) + tuple(local.shape[1:])
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=local.device)
    elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous():
        raise ValueError("allgather_f32: `out` must be a contiguous CUDA float32 tensor of shape %r" % (shape,))
    L.check(lib.lkb_allgather_f32(L.ptr(local), int(local.numel()), L.ptr(out), _stream_ptr()))
    return out
