"""The CPU truth of BLS method="slow" (oracle/bls_slow.py): hand-checkable answers, literal vs vectorised oracle,
transit recovery next to the binned search, and - wherever astropy imports - astropy itself."""
import numpy as np
import pytest

from oracle import bls as obls
from oracle import bls_slow as osl


def test_known_answer_one_box():
    """20 unit-weight cadences at x = 0..19, three of them (x = 9, 10, 11) 1 lower.  Period 20, duration 3.5,
    oversample 7 (d_phase = 0.5): the box centred on t0 = 10 holds exactly the three low cadences (|x - 10| < 1.75)."""
    t = 100.0 + np.arange(20.0)
    y = np.zeros(20)
    y[9:12] = -1.0
    r = osl.bls_power_slow_numpy(t, y, None, [20.0], [3.5], oversample=7, return_index=True)
    # median(y) = 0; y_in = -1, y_out = 0; depth 1; ivar_in 3, ivar_out 17; loglike = 0.5 * 3 * 1 = 1.5
    assert list(r["index"][0]) == [0, 20, 3]
    assert r["power"][0] == pytest.approx(1.5, rel=1e-15)
    assert r["depth"][0] == 1.0
    assert r["depth_err"][0] == pytest.approx(np.sqrt(1 / 3 + 1 / 17), rel=1e-15)
    assert r["duration"][0] == 3.5
    assert r["transit_time"][0] == 110.0
    rs = osl.bls_power_slow_numpy(t, y, None, [20.0], [3.5], oversample=7, objective="snr", return_index=True)
    assert rs["power"][0] == pytest.approx(1.0 / np.sqrt(1 / 3 + 1 / 17), rel=1e-15)
    # the neighbouring epoch t0 = 9.5 (i = 19) holds x = 8 .. 11: four cadences, one of them not low
    assert osl.objective_at_slow(t, y, None, 20.0, 3.5, 19, oversample=7, return_count=True)[1] == 4


def test_known_answer_wraps_and_transit_time():
    """A box at phase 0 wraps around the period: at P = 5 the low cadences x = 0, 5, ..., 20 are the members of the
    box at t0 = 0 and of the boxes at t0 = 4.8 and 5.4 (past the period end); the three tie and the first wins."""
    t = np.arange(21.0)
    y = np.zeros(21)
    y[::5] = -2.0
    r = osl.bls_power_slow_numpy(t, y, None, [5.0], [1.2], oversample=2, return_index=True)
    k, i, cnt = r["index"][0]
    assert (k, i, cnt) == (0, 0, 5)
    assert r["transit_time"][0] == 0.0 and r["depth"][0] == 2.0
    d_phase = 1.2 / 2
    last = len(np.arange(0, 5.0 + d_phase, d_phase)) - 1
    assert osl.objective_at_slow(t, y, None, 5.0, 1.2, last, oversample=2) == r["power"][0]


def test_no_positive_depth_gives_minus_inf():
    t = np.arange(50.0)
    y = np.ones(50)
    r = osl.bls_power_slow_numpy(t, y, None, [4.0, 7.0], [1.0], return_index=True)
    assert np.all(r["power"] == -np.inf) and np.all(r["index"] == [-1, -1, 0])
    v = osl.bls_power_slow_vec(t, y, None, [4.0, 7.0], [1.0], return_index=True)
    assert np.all(v["power"] == -np.inf) and np.all(v["index"] == [-1, -1, 0])


def _lc(rng, n=1500, per0=0.9, dep=3e-3, dur0=0.08, dt=2.0 / 1440, err=None):
    t = 1325.0 + np.arange(int(n * 1.1)) * dt
    t = np.concatenate([t[: n // 2], t[n // 2 + int(0.1 * n):]])[:n]
    y = 1 + 5e-4 * rng.normal(size=n)
    y[np.abs((t - t[0] - 0.31 + 0.5 * per0) % per0 - 0.5 * per0) < 0.5 * dur0] -= dep
    return t, y, (None if err is None else err * rng.uniform(0.8, 1.2, n))


@pytest.mark.parametrize("objective,err,oversample", [("likelihood", None, 10), ("snr", 5e-4, 10),
                                                      ("likelihood", 5e-4, 4)])
def test_literal_and_vectorised_oracles_agree(objective, err, oversample):
    rng = np.random.default_rng(7)
    t, y, dy = _lc(rng, err=err)
    period = np.exp(np.linspace(np.log(0.3), np.log(1.4), 17))
    duration = [0.05, 0.09, 0.13]
    a = osl.bls_power_slow_numpy(t, y, dy, period, duration, oversample, objective, return_index=True)
    b = osl.bls_power_slow_vec(t, y, dy, period, duration, oversample, objective, return_index=True)
    np.testing.assert_array_equal(a["index"], b["index"])
    for f in obls.RESULT_FIELDS:
        np.testing.assert_allclose(b[f], a[f], rtol=1e-9, atol=1e-12 * np.max(np.abs(a["power"])), err_msg=f)


def test_vectorised_oracle_on_an_aligned_grid():
    """Cadences and window ends on one binary grid: many cadences sit exactly on a window end, where only the
    literal predicate decides."""
    rng = np.random.default_rng(3)
    t = 0.0078125 * np.arange(900)
    y = 1 + 1e-3 * rng.normal(size=len(t))
    y[(t % 1.25) < 0.125] -= 4e-3
    period = np.array([0.5, 0.625, 1.0, 1.25, 1.5, 2.5])
    duration = [0.25, 0.125, 0.0625]
    a = osl.bls_power_slow_numpy(t, y, None, period, duration, 4, return_index=True)
    b = osl.bls_power_slow_vec(t, y, None, period, duration, 4, return_index=True)
    np.testing.assert_array_equal(a["index"], b["index"])
    np.testing.assert_allclose(b["power"], a["power"], rtol=1e-9)


def test_injected_transit_found_by_slow_and_fast():
    rng = np.random.default_rng(21)
    t, y, dy = _lc(rng, n=2500, per0=1.1, dep=2e-3, dur0=0.1, err=5e-4)
    period = np.exp(np.linspace(np.log(0.5), np.log(1.6), 60))
    duration = [0.05, 0.1, 0.15]
    s = osl.bls_power_slow_vec(t, y, dy, period, duration)
    f = obls.bls_power_numpy(t, y, dy, period, duration)
    ps, pf = int(np.argmax(s["power"])), int(np.argmax(f["power"]))
    assert abs(period[ps] - 1.1) < 0.02 and abs(period[pf] - 1.1) < 0.02
    assert s["duration"][ps] == 0.1
    assert s["depth"][ps] == pytest.approx(2e-3, rel=0.1)
    phase = ((s["transit_time"][ps] - t[0] - 0.31) / period[ps] + 0.5) % 1.0 - 0.5
    assert abs(phase) < 0.03


def test_numpy_arange_is_the_kernels_t0_grid():
    """K3s builds t0_i = i * d_phase for i < ceil((P + d_phase) / d_phase); that is np.arange(0, P + d_phase, d_phase)
    bit for bit."""
    rng = np.random.default_rng(0)
    for _ in range(3000):
        per, dur, os_ = rng.uniform(0.1, 30), rng.uniform(0.01, 0.5), int(rng.integers(1, 20))
        d_phase = np.float64(dur) / os_
        ar = np.arange(0, per + d_phase, d_phase)
        n = int(np.ceil((per + d_phase) / d_phase))
        assert len(ar) == n
        np.testing.assert_array_equal(ar, np.arange(n) * d_phase)


def test_literal_matches_astropy():
    """The pin of the recalled method="slow" semantics: astropy's own search where astropy is installed."""
    bls_mod = pytest.importorskip("astropy.timeseries")
    rng = np.random.default_rng(4)
    t, y, dy = _lc(rng, n=700, err=5e-4)
    period = np.exp(np.linspace(np.log(0.35), np.log(1.2), 9))
    duration = [0.05, 0.1]
    for objective in ("likelihood", "snr"):
        ref = bls_mod.BoxLeastSquares(t, y, dy).power(period, duration, objective=objective, method="slow",
                                                      oversample=10)
        mine = osl.bls_power_slow_numpy(t, y, dy, period, duration, 10, objective)
        for f in ("power", "depth", "depth_err", "duration", "transit_time", "depth_snr", "log_likelihood"):
            np.testing.assert_allclose(mine[f], np.asarray(getattr(ref, f)), rtol=1e-9, err_msg=f)
