"""K3s (lightkurve_b200/csrc/bls_slow.cu: prologue, lookup tables, exact-membership search, host orchestration)
executed on the CPU through tests/native/cuda_emu.h and compared with the literal restatement of astropy's
method="slow" loop (oracle/bls_slow.py).  Leaves only hardware-side behaviour to the GPU tests."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import bls_slow as osl

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"
c_vp, c_int, c_i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
FIELDS = ("power", "depth", "depth_err", "duration", "transit_time", "depth_snr", "log_likelihood")
MEM_HOST, MEM_DEVICE = 0, 1


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if shutil.which("g++") is None or not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA headers")
    out = str(tmp_path_factory.mktemp("emu") / "libbls_slow_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-pthread", "-I" + CUDA_INC, "-Wno-attributes", "-shared", "-fPIC",
                           "-Wl,-Bsymbolic", "-o", out, os.path.join(HERE, "native", "bls_slow_emu_driver.cpp")])
    lib = ctypes.CDLL(out)
    lib.emu_bls_power_slow.argtypes = [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_vp, c_int, c_int, c_int] + \
        [c_vp] * 8 + [c_int]
    lib.emu_bls_power_slow.restype = c_int
    lib.emu_last_error.restype = ctypes.c_char_p
    return lib


def _run(emu, times, fluxes, errs, period, duration, oversample=10, objective="likelihood", mem=MEM_HOST):
    B = len(times)
    off = np.zeros(B + 1, np.int64)
    np.cumsum([len(t) for t in times], out=off[1:])
    t = np.ascontiguousarray(np.concatenate(times), dtype=np.float64)
    y = np.ascontiguousarray(np.concatenate(fluxes), dtype=np.float64)
    dy = None if errs is None else np.ascontiguousarray(np.concatenate(errs), dtype=np.float64)
    period = np.ascontiguousarray(period, dtype=np.float64)
    duration = np.ascontiguousarray(duration, dtype=np.float64)
    P = len(period)
    outs = [np.full((B, P), -7.0) for _ in FIELDS]
    index = np.full((B, P, 3), -7, np.int32)
    rc = emu.emu_bls_power_slow(t.ctypes.data, y.ctypes.data, None if dy is None else dy.ctypes.data, off.ctypes.data,
                                B, period.ctypes.data, P, duration.ctypes.data, len(duration), oversample,
                                1 if objective == "snr" else 0, *[o.ctypes.data for o in outs], index.ctypes.data, mem)
    res = dict(zip(FIELDS, outs))
    res["index"] = index
    return rc, res


def _lc(rng, n, per0, dep, dur0, dt=2.0 / 1440, gap=(0.45, 0.55), err=None):
    t = 1325.0 + np.arange(int(n * 1.15)) * dt
    g0, g1 = int(gap[0] * len(t)), int(gap[1] * len(t))
    t = np.concatenate([t[:g0], t[g1:]])[:n]
    y = 1 + 5e-4 * rng.normal(size=n)
    y[np.abs((t - t[0] - 0.37 + 0.5 * per0) % per0 - 0.5 * per0) < 0.5 * dur0] -= dep
    dy = None if err is None else err * rng.uniform(0.8, 1.2, n)
    return t, y, dy


def check_against_literal(t, y, dy, period, duration, res, b, oversample=10, objective="likelihood"):
    """The parity rule of K3s: best index identical except where the literal oracle's objective_at_slow shows an exact
    tie (1e-10 relative), the in-box count of the chosen box exact, values rtol 1e-9 with a floor of 1e-12 x max power."""
    ref = osl.bls_power_slow_numpy(t, y, dy, period, duration, oversample, objective, return_index=True)
    got_idx, ref_idx = res["index"][b], ref["index"]
    fin = np.isfinite(ref["power"])
    floor = 1e-12 * np.max(np.abs(ref["power"][fin])) if fin.any() else 0.0
    np.testing.assert_array_equal(np.isfinite(res["power"][b]), fin)
    for p in np.flatnonzero(np.any(got_idx != ref_idx, axis=1)):
        k, i, cnt = (int(v) for v in got_idx[p])
        assert k >= 0, "period %d: no box found, oracle has %s" % (p, ref_idx[p])
        val, c = osl.objective_at_slow(t, y, dy, period[p], duration[k], i, oversample, objective, return_count=True)
        assert abs(val - ref["power"][p]) <= 1e-10 * abs(ref["power"][p]), \
            "period %d: box %s is not a tie of the oracle's %s" % (p, got_idx[p], ref_idx[p])
        assert c == cnt, "period %d: in-box count %d, the oracle counts %d" % (p, cnt, c)
    same = np.all(got_idx == ref_idx, axis=1)
    for f in FIELDS:
        g, r = res[f][b][same & fin], ref[f][same & fin]
        np.testing.assert_allclose(g, r, rtol=1e-9, atol=floor if f in ("power", "log_likelihood", "depth_snr") else 0,
                                   err_msg=f)
    return ref


@pytest.mark.parametrize("objective,with_err", [("likelihood", False), ("snr", True), ("likelihood", True)])
def test_k3s_ragged_batch_on_the_emulator(emu, objective, with_err):
    rng = np.random.default_rng(11 if with_err else 12)
    lcs = [_lc(rng, 900, 0.9, 4e-3, 0.06, err=5e-4 if with_err else None),
           _lc(rng, 1300, 0.8, 3e-3, 0.1, err=5e-4 if with_err else None),
           _lc(rng, 600, 0.7, 0.0, 0.1, err=5e-4 if with_err else None)]     # no transit
    times, fluxes, errs = (list(v) for v in zip(*lcs))
    period = np.exp(np.linspace(np.log(0.35), np.log(1.5), 13))
    duration = [0.04, 0.07, 0.11]
    rc, res = _run(emu, times, fluxes, errs if with_err else None, period, duration, objective=objective)
    assert rc == 0, emu.emu_last_error()
    for b in range(3):
        check_against_literal(times[b], fluxes[b], errs[b] if with_err else None, period, duration, res, b,
                              objective=objective)
    # the injected periods are found with their own duration
    for b, (per0, dur0) in enumerate(((0.9, 0.06), (0.8, 0.1))):
        p = int(np.argmax(res["power"][b]))
        assert abs(period[p] - per0) < 0.05 and abs(res["duration"][b][p] - dur0) <= 0.03


def test_k3s_aligned_grid_and_oversample_on_the_emulator(emu):
    """Cadences on an exact binary grid: window ends fall on cadences, so the exact predicate decides in the walks;
    oversample 3 and durations given in descending order."""
    rng = np.random.default_rng(5)
    t = 0.0078125 * np.arange(700)                 # 2^-7 d
    y = 1 + 1e-3 * rng.normal(size=len(t))
    y[(t % 1.25) < 0.125] -= 5e-3
    period = np.array([0.5, 0.625, 1.0, 1.25, 1.5, 2.5])
    duration = [0.25, 0.125, 0.0625]
    rc, res = _run(emu, [t], [y], None, period, duration, oversample=3)
    assert rc == 0, emu.emu_last_error()
    check_against_literal(t, y, None, period, duration, res, 0, oversample=3)


def test_k3s_no_positive_depth_and_device_mem_on_the_emulator(emu):
    """A constant light curve: every box has depth 0, so no period has a box with depth > 0 => power -inf and the
    documented outputs; the same through the device-buffer path (no staging)."""
    t = np.arange(200) * 0.01
    y = np.ones_like(t)
    period = np.array([0.3, 0.5])
    duration = [0.05]
    for mem in (MEM_HOST, MEM_DEVICE):
        rc, res = _run(emu, [t], [y], None, period, duration, mem=mem)
        assert rc == 0, emu.emu_last_error()
        assert np.all(res["power"][0] == -np.inf)
        assert np.all(res["index"][0] == [-1, -1, 0])
        assert np.all(res["duration"][0] == 0) and np.all(res["depth"][0] == 0)
        np.testing.assert_array_equal(res["transit_time"][0], t[0])


def test_k3s_rejects_unsorted_times_on_the_emulator(emu):
    rng = np.random.default_rng(2)
    t = np.sort(rng.uniform(0, 5, 300))
    t[[10, 11]] = t[[11, 10]]
    rc, _ = _run(emu, [t], [1 + 1e-3 * rng.normal(size=300)], None, np.array([1.0, 1.5]), [0.1])
    assert rc == -5 and b"ascending" in emu.emu_last_error()
    rc, _ = _run(emu, [t], [np.ones(300)], None, np.array([0.1]), [0.1])
    assert rc == -1 and b"shorter than the minimum period" in emu.emu_last_error()
