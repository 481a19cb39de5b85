"""Throughput of BLS method="slow" (K3s) next to method="fast" (K3) on config 3's workload.

Workload: bench.py's make_bls_workload (256 TESS light curves x 20 000 cadences x 50 000 periods x 10 durations,
oversample 10, objective likelihood), inputs and outputs device-resident (the C ABI with LKB_MEM_DEVICE).  The two
searches run alternately in one process, after a warm-up of each, and every call is timed with CUDA events.
Reported: (light curve, period) pairs / s of each, and for K3s the table lookups / s, where the lookups per pair are
counted from the shapes by `slow_lookups_per_pair` (2 per (t0, cycle) box end).  CPU leg: the literal oracle
(oracle/bls_slow.py) on a few periods of one light curve, extrapolated to the workload and labelled as such.
The card's name and power limit are read with nvidia-smi in the same run.  Output: one JSON file under profiles/
(or --out).

    python tools/bls_slow_bench.py [--rounds 3] [--periods 50000] [--out profiles/bls_slow_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FIELDS = ("power", "depth", "depth_err", "duration", "transit_time", "depth_snr", "log_likelihood")


def slow_lookups_per_pair(period, duration, x_max, oversample=10):
    """Table lookups K3s makes per (light curve, period), averaged over the grid: for every duration, every
    t0_i = i d / oversample (i < ceil((P + d/oversample) / (d/oversample))) and every cycle of the kernel's range
    [floor((-P/2 - t0) / P), ceil((x_max + P/2 - t0) / P)], two lookups (one per window end)."""
    total = 0.0
    for d in duration:
        dp = d / oversample
        for P in period:
            n_t0 = int(np.ceil((P + dp) / dp))
            t0 = np.arange(n_t0) * dp
            cyc = np.ceil((x_max + 0.5 * P - t0) / P) - np.floor((-0.5 * P - t0) / P) + 1
            total += 2.0 * cyc.sum()
    return total / len(period)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, plim = (s.strip() for s in out[0].split(","))
        return {"name": name, "power_limit": plim}
    except Exception as e:                                          # pragma: no cover
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="timed calls of each search (alternating)")
    ap.add_argument("--lcs", type=int, default=256)
    ap.add_argument("--periods", type=int, default=50000)
    ap.add_argument("--cpu-periods", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bls_slow_bench.json"))
    args = ap.parse_args()

    import torch
    from bench import make_bls_workload
    from lightkurve_b200 import _lib as L, engine
    from oracle import bls_slow as osl

    if engine.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    engine.init(0)
    info = card()
    B, N, P = args.lcs, 20000, args.periods
    t, fluxes, errs, period, duration = make_bls_workload(1003, B, N, P)
    dev = torch.device("cuda:0")
    d_t = torch.from_numpy(np.tile(t, B)).to(dev)
    d_y = torch.from_numpy(np.concatenate(fluxes)).to(dev)
    d_dy = torch.from_numpy(np.concatenate(errs)).to(dev)
    d_per = torch.from_numpy(period).to(dev)
    d_dur = torch.from_numpy(duration).to(dev)
    off = np.arange(B + 1, dtype=np.int64) * N
    outs = {m: [torch.empty((B, P), dtype=torch.float64, device=dev) for _ in FIELDS] for m in ("fast", "slow")}
    bins = torch.empty((B, P, 2), dtype=torch.int32, device=dev)
    index = torch.empty((B, P, 3), dtype=torch.int32, device=dev)
    lib = L.load()
    st = torch.cuda.current_stream().cuda_stream

    def call(method):
        o = [L.ptr(x) for x in outs[method]]
        if method == "fast":
            rc = lib.lkb_bls_power(L.ptr(d_t), L.ptr(d_y), L.ptr(d_dy), L.ptr(off), B, L.ptr(d_per), P, L.ptr(d_dur),
                                   len(duration), 10, L.BLS_LIKELIHOOD, *o, L.ptr(bins), L.MEM_DEVICE, st)
        else:
            rc = lib.lkb_bls_power_slow(L.ptr(d_t), L.ptr(d_y), L.ptr(d_dy), L.ptr(off), B, L.ptr(d_per), P,
                                        L.ptr(d_dur), len(duration), 10, L.BLS_LIKELIHOOD, *o, L.ptr(index),
                                        L.MEM_DEVICE, st)
        L.check(rc)

    for m in ("fast", "slow"):                                       # warm-up (workspace growth, module load)
        call(m)
    torch.cuda.synchronize()
    ms = {"fast": [], "slow": []}
    for _ in range(args.rounds):
        for m in ("fast", "slow"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call(m)
            e1.record()
            torch.cuda.synchronize()
            ms[m].append(e0.elapsed_time(e1))

    pairs = float(B) * P
    x_max = float(t[-1] - t[0])
    lpp = slow_lookups_per_pair(period, duration, x_max)
    res = {"card": info, "workload": "config 3: %d TESS LC x %d cadences x %d periods x %d durations, oversample 10, "
                                     "objective likelihood, device-resident" % (B, N, P, len(duration)),
           "timing": "CUDA events around each whole C-ABI call (prologue, tables, search), %d alternating rounds after "
                     "one warm-up call of each" % args.rounds}
    for m in ("fast", "slow"):
        med = float(np.median(ms[m]))
        res[m] = {"ms": ms[m], "ms_median": med, "lc_period_pairs_per_s": pairs / (med * 1e-3)}
    res["slow"]["lookups_per_pair"] = lpp
    res["slow"]["lookups_per_s"] = lpp * pairs / (res["slow"]["ms_median"] * 1e-3)
    res["slow_over_fast_time"] = res["slow"]["ms_median"] / res["fast"]["ms_median"]

    # parity on a sample: the GPU's slow result against the vectorised oracle, first light curve, 20 periods
    sub = np.arange(0, P, max(1, P // 20))
    p_gpu = outs["slow"][0][0].cpu().numpy()[sub]
    ref = osl.bls_power_slow_vec(t, fluxes[0], errs[0], period[sub], duration)
    res["parity_on_sample"] = bool(np.allclose(p_gpu, ref["power"], rtol=1e-9, atol=1e-12 * np.max(ref["power"])))

    # CPU leg: the literal oracle, one light curve x a few periods, extrapolated (NOT a measurement of the full job)
    cpu_sub = period[:: max(1, P // args.cpu_periods)][: args.cpu_periods]
    t0 = time.perf_counter()
    osl.bls_power_slow_numpy(t, fluxes[0], errs[0], cpu_sub, duration)
    secs = time.perf_counter() - t0
    # the literal loop's cost is one O(N) pass per (duration, t0): scale by the number of boxes
    boxes = lambda pers: sum(np.ceil((pers + d / 10) / (d / 10)).sum() for d in duration)
    full_s = secs * B * boxes(period) / boxes(cpu_sub)
    res["cpu_literal_oracle"] = {"measured": "%d periods of one light curve in %.1f s (one numpy process)"
                                             % (len(cpu_sub), secs),
                                 "extrapolated_full_job_s": full_s,
                                 "extrapolated_lc_period_pairs_per_s": pairs / full_s,
                                 "note": "extrapolated from the sample by the number of (duration, t0) boxes, "
                                         "not run at full size"}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
