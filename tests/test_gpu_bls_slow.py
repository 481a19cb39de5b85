"""K3s on the B200: BLS method="slow" (lightkurve_b200/csrc/bls_slow.cu) against the literal restatement of astropy's
loop and, at config-3 scale, against the vectorised oracle (oracle/bls_slow.py)."""
import numpy as np
import pytest

from lightkurve_b200 import LightCurve, LightCurveCollection
from lightkurve_b200.periodogram import BoxLeastSquaresPeriodogram
from lightkurve_b200 import _lib as L
from oracle import bls_slow as osl
from test_bls_slow_emulated import check_against_literal

pytestmark = pytest.mark.gpu

FIELDS = ("power", "depth", "depth_err", "duration", "transit_time", "depth_snr", "log_likelihood")


def _lc(rng, n, per0, dep, dur0, dt=2.0 / 1440, gaps=((0.45, 0.55),), err=None):
    t = 1325.0 + np.arange(int(n * 1.3)) * dt
    keep = np.ones(len(t), bool)
    for g0, g1 in gaps:
        keep[int(g0 * len(t)):int(g1 * len(t))] = False
    t = t[keep][:n]
    y = 1 + 5e-4 * rng.normal(size=len(t))
    if dep:
        y[np.abs((t - t[0] - 0.37 + 0.5 * per0) % per0 - 0.5 * per0) < 0.5 * dur0] -= dep
    dy = None if err is None else err * rng.uniform(0.8, 1.2, len(t))
    return t, y, dy


@pytest.mark.parametrize("objective,with_err", [("likelihood", False), ("likelihood", True), ("snr", False),
                                                ("snr", True)])
def test_k3s_ragged_batches_vs_literal(engine, objective, with_err):
    rng = np.random.default_rng(100 + 2 * with_err + (objective == "snr"))
    err = 5e-4 if with_err else None
    lcs = [_lc(rng, 1100, 0.9, 4e-3, 0.06, err=err),
           _lc(rng, 1500, 0.8, 2e-3, 0.1, gaps=((0.2, 0.25), (0.6, 0.7)), err=err),
           _lc(rng, 700, 0.0, 0.0, 0.0, err=err),
           _lc(rng, 1800, 1.2, 6e-3, 0.12, gaps=(), err=err)]
    times, fluxes, errs = (list(v) for v in zip(*lcs))
    period = np.exp(np.linspace(np.log(0.3), np.log(1.6), 23))
    duration = [0.04, 0.07, 0.11, 0.15]
    res = engine.bls_power(times, fluxes, errs if with_err else None, period, duration, objective=objective,
                           return_bins=True, method="slow")
    for b in range(len(times)):
        check_against_literal(times[b], fluxes[b], errs[b] if with_err else None, period, duration, res, b,
                              objective=objective)


def test_k3s_no_positive_depth(engine):
    """A constant light curve (every box has depth 0) next to a normal one: power -inf and the documented outputs."""
    rng = np.random.default_rng(3)
    t1 = np.arange(300) * 0.01
    t2, y2, _ = _lc(rng, 800, 0.5, 3e-3, 0.05)
    period = np.array([0.3, 0.5, 0.7])
    res = engine.bls_power([t1, t2], [np.ones(300), y2], None, period, [0.05], return_bins=True, method="slow")
    assert np.all(res["power"][0] == -np.inf) and np.all(res["index"][0] == [-1, -1, 0])
    assert np.all(res["duration"][0] == 0) and np.all(res["depth"][0] == 0)
    np.testing.assert_array_equal(res["transit_time"][0], t1[0])
    check_against_literal(t2, y2, None, period, [0.05], res, 1)


def test_k3s_device_mem_matches_host_mem(engine):
    import torch
    rng = np.random.default_rng(8)
    lcs = [_lc(rng, 1200, 0.7, 3e-3, 0.08, err=5e-4), _lc(rng, 900, 0.0, 0.0, 0.0, err=5e-4)]
    times, fluxes, errs = (list(v) for v in zip(*lcs))
    period = np.exp(np.linspace(np.log(0.3), np.log(1.5), 40))
    duration = np.array([0.05, 0.1])
    host = engine.bls_power(times, fluxes, errs, period, duration, return_bins=True, method="slow")
    off = np.zeros(3, np.int64)
    np.cumsum([len(t) for t in times], out=off[1:])
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.concatenate(v)).to(dev) for k, v in (("t", times), ("y", fluxes), ("dy", errs))}
    d_per, d_dur = torch.from_numpy(period).to(dev), torch.from_numpy(duration).to(dev)
    outs = [torch.empty((2, len(period)), dtype=torch.float64, device=dev) for _ in FIELDS]
    idx = torch.empty((2, len(period), 3), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    L.check(L.load().lkb_bls_power_slow(L.ptr(d["t"]), L.ptr(d["y"]), L.ptr(d["dy"]), L.ptr(off), 2, L.ptr(d_per),
                                        len(period), L.ptr(d_dur), len(duration), 10, L.BLS_LIKELIHOOD,
                                        *[L.ptr(o) for o in outs], L.ptr(idx), L.MEM_DEVICE, st))
    torch.cuda.synchronize()
    for k, o in zip(FIELDS, outs):
        np.testing.assert_array_equal(o.cpu().numpy(), host[k], err_msg=k)
    np.testing.assert_array_equal(idx.cpu().numpy(), host["index"])


def test_k3s_unsorted_times_are_refused(engine):
    rng = np.random.default_rng(4)
    t, y, _ = _lc(rng, 500, 0.5, 3e-3, 0.05)
    t = t.copy()
    t[[100, 101]] = t[[101, 100]]
    with pytest.raises(L.EngineError, match="ascending"):
        engine.bls_power([t], [y], None, [0.5, 0.7], [0.05], method="slow")
    with pytest.raises(ValueError, match="method"):
        engine.bls_power([t], [y], None, [0.5, 0.7], [0.05], method="brute")


def test_k3s_config3_sliver_vs_vectorised_oracle(engine):
    """4 TESS-like light curves x 20 000 cadences x 200 of config 3's periods x its 10 durations (bench.py's
    make_bls_workload), against the vectorised oracle; tie rule in the literal oracle's arithmetic."""
    import bench
    t, fluxes, errs, period_full, duration = bench.make_bls_workload(1003, B=4, N=20000, P=50000)
    period = period_full[::250]
    res = engine.bls_power([t] * 4, fluxes, errs, period, duration, return_bins=True, method="slow")
    n_tied = 0
    for b in range(4):
        ref = osl.bls_power_slow_vec(t, fluxes[b], errs[b], period, duration, return_index=True)
        got_idx = res["index"][b]
        diff = np.flatnonzero(np.any(got_idx != ref["index"], axis=1))
        for p in diff:
            k, i, cnt = (int(v) for v in got_idx[p])
            val, c = osl.objective_at_slow(t, fluxes[b], errs[b], period[p], duration[k], i, return_count=True)
            assert abs(val - ref["power"][p]) <= 1e-10 * abs(ref["power"][p]), (b, p, got_idx[p], ref["index"][p])
            assert c == cnt
        n_tied += len(diff)
        same = np.all(got_idx == ref["index"], axis=1)
        floor = 1e-12 * np.max(ref["power"])
        for f in FIELDS:
            np.testing.assert_allclose(res[f][b][same], ref[f][same], rtol=1e-9,
                                       atol=floor if f in ("power", "log_likelihood", "depth_snr") else 0, err_msg=f)
        np.testing.assert_allclose(res["power"][b], ref["power"], rtol=1e-9, atol=floor)
    assert n_tied <= 0.02 * 4 * len(period)


def _shim_lc(rng, n=3000, per0=1.1, dep=2e-3, dur0=0.1):
    t, y, dy = _lc(rng, n, per0, dep, dur0, err=5e-4)
    return LightCurve(time=t, flux=y, flux_err=dy)


def test_k3s_shim_to_periodogram(engine):
    rng = np.random.default_rng(17)
    lc = _shim_lc(rng)
    period = np.exp(np.linspace(np.log(0.5), np.log(1.6), 80))
    duration = [0.05, 0.1, 0.15]
    pg = lc.to_periodogram("bls", period=period, duration=duration, bls_method="slow")
    direct = BoxLeastSquaresPeriodogram.from_lightcurve(lc, period=period, duration=duration, method="slow")
    np.testing.assert_array_equal(direct.power.value, pg.power.value)
    ref = osl.bls_power_slow_vec(lc.time.value, lc.flux.value, lc.flux_err.value, period, duration)
    np.testing.assert_allclose(pg.power.value, ref["power"], rtol=1e-9, atol=1e-12 * np.max(ref["power"]))
    assert abs(pg.period_at_max_power.value - 1.1) < 0.02
    assert pg.duration_at_max_power.value == 0.1
    # the follow-ups work on the slow result as on the fast one
    stats = pg.compute_stats()
    assert np.isfinite(stats["depth"][0])
    assert pg.get_transit_mask().sum() > 0
    # method="fast" is unchanged and still the default
    fast = lc.to_periodogram("bls", period=period, duration=duration)
    np.testing.assert_array_equal(fast.power.value,
                                  lc.to_periodogram("bls", period=period, duration=duration,
                                                    bls_method="fast").power.value)
    with pytest.raises(NotImplementedError):
        lc.to_periodogram("bls", period=period, duration=duration, bls_method="brute")


def test_k3s_shim_unsorted_input(engine):
    rng = np.random.default_rng(18)
    lc = _shim_lc(rng, n=2000)
    perm = rng.permutation(len(lc.time.value))
    t, y, dy = lc.time.value, lc.flux.value, lc.flux_err.value
    lc_shuffled = LightCurve(time=t[perm], flux=y[perm], flux_err=dy[perm])
    period = np.exp(np.linspace(np.log(0.5), np.log(1.6), 50))
    duration = [0.05, 0.1]
    a = lc.to_periodogram("bls", period=period, duration=duration, bls_method="slow")
    b = lc_shuffled.to_periodogram("bls", period=period, duration=duration, bls_method="slow")
    np.testing.assert_allclose(b.power.value, a.power.value, rtol=1e-9)
    np.testing.assert_allclose(b.transit_time.value, a.transit_time.value, rtol=1e-12)
    # the follow-ups use the light curve's own cadence order
    args = dict(period=a.period_at_max_power.value, duration=a.duration_at_max_power.value,
                transit_time=a.transit_time_at_max_power.value)
    np.testing.assert_allclose(b.compute_stats(**args)["depth"], a.compute_stats(**args)["depth"], rtol=1e-9)


def test_k3s_collection_equals_loop(engine):
    rng = np.random.default_rng(19)
    lcs = [_shim_lc(rng, n=n, per0=p0) for n, p0 in ((2000, 0.9), (2600, 1.2), (1500, 0.7))]
    period = np.exp(np.linspace(np.log(0.5), np.log(1.6), 40))
    duration = [0.05, 0.1]
    many = LightCurveCollection(lcs).to_periodogram("bls", period=period, duration=duration, bls_method="slow")
    for lc, pg in zip(lcs, many):
        one = lc.to_periodogram("bls", period=period, duration=duration, bls_method="slow")
        np.testing.assert_array_equal(pg.power.value, one.power.value)
        np.testing.assert_array_equal(pg.duration.value, one.duration.value)
        np.testing.assert_array_equal(pg.transit_time.value, one.transit_time.value)
