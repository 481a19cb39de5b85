"""The persistent row transform kernel (nufft_v2.cuh: v2_ring) on the CPU emulator, with the CTA count forced
(LKB_NUFFT_RING_CTAS) so that the ring's corner cases all occur: a CTA with more tiles than buffers and a tile count
that is not a multiple of 3 (the ring wraps and the mbarrier parities flip), CTAs with a single tile, and a group
without any tile.  Every such run must give the same bits as a run with one tile per CTA - the split of tiles over CTAs
and groups changes where a tile is computed, never how."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"
c_vp, c_i64, c_int, c_dbl = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double

# B = 7 light curves at 2^15 fine-grid cells (A = 32): 2 row groups per light curve -> 14 tiles.  1 CTA: tiles 0 .. 13
# (the ring wraps four times, parities 0, 1, 0); 4 CTAs: 4 + 4 + 3 + 3; 13 CTAs: one CTA with 2 tiles and twelve with a
# single tile, whose second group has none.
CTAS = [1, 4, 13]
ONE_TILE_EACH = 64


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if shutil.which("g++") is None or not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA headers")
    out = str(tmp_path_factory.mktemp("emu_ring") / "libnufft_emu.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-pthread", "-I" + CUDA_INC, "-Wno-attributes", "-shared", "-fPIC",
                           "-Wl,-Bsymbolic", "-o", out, os.path.join(HERE, "native", "nufft_emu_driver.cpp")])
    lib = ctypes.CDLL(out)
    lib.emu_nufft_shared.argtypes = [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_dbl, c_dbl, c_vp, c_vp,
                                     c_i64, c_int, c_dbl, c_vp]
    lib.emu_nufft_ragged.argtypes = [c_vp, c_vp, c_vp, c_vp, c_int, c_i64, c_i64, c_vp, c_vp, c_i64, c_dbl, c_dbl, c_int,
                                     c_vp, c_vp]
    lib.emu_last_error.restype = ctypes.c_char_p
    return lib


def test_shared_grid_ring_split_is_bitwise_invariant(emu, monkeypatch):
    rng = np.random.default_rng(31)
    B, N, F, oversample = 7, 500, 7000, 5.0
    trel = np.sort(rng.uniform(0, 30.0, N))
    trel -= trel[0]
    df = 1.0 / (oversample * trel[-1])
    freq = df * (1 + np.arange(F))
    Npad = 512
    yc = np.zeros((B, Npad), np.float32)
    yc[:, :N] = (10 ** rng.uniform(-4, -2, (B, 1)) * np.sin(2 * np.pi * rng.uniform(0.2, 3, (B, 1)) * trel)
                 + 1e-4 * rng.normal(size=(B, N)))
    yc[:, :N] -= yc[:, :N].mean(axis=1, keepdims=True)
    ysum = yc.astype(np.float64).sum(axis=1).astype(np.float32)
    absmax = np.abs(yc).max(axis=1).astype(np.float32)
    rot, rot2 = np.zeros((F, 4), np.float32), np.zeros((F, 2), np.float32)

    def run(ctas):
        monkeypatch.setenv("LKB_NUFFT_RING_CTAS", str(ctas))
        power = np.zeros((B, F), np.float32)
        rc = emu.emu_nufft_shared(trel.ctypes.data, N, yc.ctypes.data, Npad, ysum.ctypes.data, absmax.ctypes.data, B,
                                  freq.ctypes.data, F, df, df, rot.ctypes.data, rot2.ctypes.data, 0, 2, 1.0,
                                  power.ctypes.data)
        assert rc == 0, emu.emu_last_error()
        return power

    ref = run(ONE_TILE_EACH)
    assert np.all(np.isfinite(ref)) and ref.max() > 0
    for ctas in CTAS:
        np.testing.assert_array_equal(run(ctas), ref, err_msg="%d CTAs" % ctas)


def test_ragged_ring_split_is_bitwise_invariant(emu, monkeypatch):
    """The ragged path's row transforms (the kernel's write-out mode) through the same ring."""
    rng = np.random.default_rng(32)
    ns = [300, 77, 512]
    B, F = len(ns), 3500
    off, poff = np.zeros(B + 1, np.int64), np.zeros(B + 1, np.int64)
    for b, n in enumerate(ns):
        off[b + 1] = off[b] + n
        poff[b + 1] = poff[b] + ((n + 3) // 4) * 4
    ptotal = int(poff[-1])
    tt, yy = np.zeros(ptotal + 4), np.zeros(ptotal + 4, np.float32)
    span, ysum = np.zeros(B), np.zeros(B)
    for b, n in enumerate(ns):
        t = np.sort(rng.uniform(0, 25.0 * rng.uniform(0.4, 1.0), n))
        y = 1e-3 * np.sin(2 * np.pi * 0.9 * t) + 1e-4 * rng.normal(size=n)
        tt[poff[b]:poff[b] + n] = t - t[0]
        yy[poff[b]:poff[b] + n] = (y - y.mean()).astype(np.float32)
        span[b] = tt[poff[b]:poff[b] + n].max()
        ysum[b] = yy[poff[b]:poff[b] + n].astype(np.float64).sum()
    df = 1.0 / (5.0 * 25.0)
    scale = np.ones(B)

    def run(ctas):
        monkeypatch.setenv("LKB_NUFFT_RING_CTAS", str(ctas))
        power = np.zeros((B, F), np.float32)
        rc = emu.emu_nufft_ragged(tt.ctypes.data, yy.ctypes.data, off.ctypes.data, poff.ctypes.data, B, ptotal,
                                  max(ns), span.ctypes.data, ysum.ctypes.data, F, df, df, 1, scale.ctypes.data,
                                  power.ctypes.data)
        assert rc == 0, emu.emu_last_error()
        return power

    ref = run(ONE_TILE_EACH)
    assert np.all(np.isfinite(ref)) and ref.max() > 0
    for ctas in (1, 2):
        np.testing.assert_array_equal(run(ctas), ref, err_msg="%d CTAs" % ctas)
