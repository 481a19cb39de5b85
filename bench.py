#!/usr/bin/env python
"""bench.py - the headline benchmark of the hot path (BASELINE.json: Lomb-Scargle throughput in
frequency-bins x cadences / s; config[1] at N=1: 1024 Kepler long-cadence light curves (65 000
cadences, shared time grid) x 1e5 frequencies).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels via the C ABI)
  python bench.py ... --dump-outputs DIR                   # also write the last step's power rows (rank 0, a
                                                           #   fixed row sample) to DIR/power.npy
  python bench.py --impl reference ...                     # the reference's CPU algorithm (oracle port
                                                           #   of astropy LombScargle method="fast")
For N > 1 launch with torchrun (one rank per GPU): the batch is sharded BY TARGET, every rank
processes its own 1024 light curves (weak scaling) and one NCCL all-gather reassembles the power
array (the only collective of the path, SURVEY.md 8e).

One JSON line on stdout (rank 0).  A "step" = one pass of lkb_ls_power_shared over the batch.
  value   : whole-job F*N*B_total / time, inputs resident in HBM (CUDA events, max over ranks)
  e2e     : same metric through the same C-ABI call with HOST buffers: pinned H2D of the flux
            matrix and D2H of the power array inside the timed region
  roofline: tensor roofline of the dominant kernel (ls_tcg_kernel): algorithmic flops 4*F*N*B per
            launch / CUDA-event duration of that kernel, vs MEASURED_PEAKS.json bf16 sustained
  cpu_baseline: the oracle port of the reference default (astropy "fast" extirpolation+FFT),
            timed on a bounded sample of the same workload on this box's host cores.
  secondary.bls: the other half of BASELINE.json's metric ("BLS periods/s"): configs[2] (256 TESS light
            curves x 20 000 cadences x 50 000 periods x 10 durations per GPU) with its own value / e2e /
            roofline / cpu_baseline objects (``secondary_bls``); ``--no-secondary`` skips it.
  secondary.ls_nufft (N = 1 only): the opt-in NUFFT Lomb-Scargle path (algo="nufft", DESIGN.md K2n) on the same
            workload - ms/step and bin*cadence/s of its variants plus a parity check against the default path, measured
            in a CHILD PROCESS after the headline timing (a fault there cannot touch the reported numbers).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLS_WARP_INSTR_PER_PAIR = 33450.0      # ncu smsp__inst_executed.sum / (light curves x periods), config-3 grid (run 4)
METRIC = "lombscargle_freqbins_x_cadences_per_s"
UNIT = "bin*cadence/s"

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(B=1024, N=65000, F=100000, desc="1024 Kepler LC (65000 cadences, shared grid) x 1e5 frequencies"),
    # BASELINE.json configs[4]: ragged collection sharded by target over the ranks (strong scaling), all-gather of power
    "c5": dict(B=16384, F=20000, desc="16384 irregularly sampled LC (2000..20000 cadences) x 20000 frequencies, sharded by "
                                      "target over the ranks, all-gather of the power rows"),
    # reduced shapes for debugging only (never the reported number)
    "c2_small": dict(B=256, N=8192, F=4096, desc="DEBUG 256 x 8192 x 4096"),
    "c5_small": dict(B=512, F=20000, desc="DEBUG 512 ragged LC x 20000 frequencies"),
}


def make_workload(name, seed):
    """SURVEY.md 8(d) config C2: Kepler grid t = 131.5 + c*0.0204336 d, c = 71 500 consecutive cadence
    numbers with ~9 % deleted in 18 contiguous gaps -> N cadences shared by the batch; flux = 1 + up to
    3 sinusoids (A~LogU(1e-4,1e-2), f~U(0.05,20)/d) + N(0, sigma_b), fp32; F regular frequencies,
    f0 = df = 1/(5*baseline); amplitude normalisation."""
    w = WORKLOADS[name]
    B, N, F = w["B"], w["N"], w["F"]
    rng = np.random.default_rng(seed)
    ntot = int(round(N * 1.1))
    keep = np.ones(ntot, bool)
    ndel = ntot - N
    cuts = np.sort(rng.choice(ntot - ndel // 18 - 2, 18, replace=False))
    for i, c in enumerate(cuts):
        keep[c:c + ndel // 18 + (1 if i < ndel % 18 else 0)] = False
    idx = np.flatnonzero(keep)
    if len(idx) > N:
        idx = idx[:N]
    elif len(idx) < N:                          # overlapping gaps: top up with the first deleted cadences
        extra = np.flatnonzero(~keep)[:N - len(idx)]
        idx = np.sort(np.concatenate([idx, extra]))
    t = 131.5 + idx * 0.0204336
    Y = np.ones((B, N), dtype=np.float32)
    chunk = 64
    for b0 in range(0, B, chunk):
        nb = min(chunk, B - b0)
        acc = np.zeros((nb, N))
        for _ in range(3):
            A = 10 ** rng.uniform(-4, -2, (nb, 1))
            f = rng.uniform(0.05, 20, (nb, 1))
            ph = rng.uniform(0, 2 * np.pi, (nb, 1))
            acc += A * np.sin(2 * np.pi * f * t[None, :] + ph)
        sig = 10 ** rng.uniform(np.log10(5e-5), -3, (nb, 1))
        acc += sig * rng.standard_normal((nb, N))
        Y[b0:b0 + nb] = (1.0 + acc).astype(np.float32)
    df = 1.0 / (5.0 * (t[-1] - t[0]))
    freq = df * (1 + np.arange(F))
    return t, Y, freq


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, device_index, period_s=0.005):
        self.dev = device_index
        self.period = period_s
        self.sm, self.reasons, self.power = [], set(), []
        self.sm_max = None
        self._stop = threading.Event()
        self.th = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.dev)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:                                    # pragma: no cover
            self.err = "nvml unavailable: %r" % (e,)
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, v in bits.items():
                    if r & v:
                        self.reasons.add(k)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception as e:                                # pragma: no cover
                self.err = repr(e)
                break
            time.sleep(self.period)

    def stop(self):
        self._stop.set()
        if self.th is not None:
            self.th.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
               "reasons": sorted(self.reasons), "samples": len(self.sm),
               "power_w_max": max(self.power) if self.power else None}
        if self.err:
            out["error"] = self.err
        return out


def _cpu_ls_worker(args):
    from oracle import ls as ols
    t, y, f0, df, nf = args
    p = ols.ls_fast_psd(t, y.astype(np.float64), f0, df, nf)
    return float(np.sqrt(p[-1]))


def _cpu_worker_init():
    """One BLAS/OpenMP thread per worker process (the pool provides the parallelism)."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass


def cpu_reference_rate(t, Y, freq, n_lc, procs, pool=None):
    """Reference CPU path (oracle port of astropy LombScargle(...).power(method='fast'), the
    lightkurve default) on `n_lc` light curves of the workload, `procs` worker processes.
    Returns (bin*cadence/s equivalent, seconds)."""
    f0, df, nf = float(freq[0]), float(freq[1] - freq[0]), len(freq)
    jobs = [(t, Y[i % len(Y)], f0, df, nf) for i in range(n_lc)]
    t0 = time.perf_counter()
    if procs <= 1 or pool is None:
        for j in jobs:
            _cpu_ls_worker(j)
    else:
        pool.map(_cpu_ls_worker, jobs, chunksize=1)
    dt = time.perf_counter() - t0
    return len(freq) * len(t) * n_lc / dt, dt


_REF = {}           # workload of the reference arm: set before the worker pool forks, so jobs carry only an index


def _ref_index_worker(i):
    t, Y, f0, df, nf, real = _REF["t"], _REF["Y"], _REF["f0"], _REF["df"], _REF["nf"], _REF["real"]
    y = Y[i % len(Y)]
    return _real_reference_worker((t, y, f0, f0 + df * nf)) if real else _cpu_ls_worker((t, y, f0, df, nf))


def _real_reference_worker(args):
    """One light curve through the REAL reference (lightkurve + astropy), if they are importable on this box."""
    import lightkurve as lk
    t, y, fmin, fmax = args
    lc = lk.LightCurve(time=t, flux=y)
    pg = lc.to_periodogram("lombscargle", minimum_frequency=fmin, maximum_frequency=fmax, oversample_factor=5,
                           normalization="amplitude", ls_method="fast")
    return float(pg.power.value[-1])


def _have_real_reference():
    try:
        import astropy  # noqa: F401
        import lightkurve  # noqa: F401
        return True
    except Exception:
        return False


def run_reference(args, rank):
    """--impl reference: the reference's own CPU algorithm on the box's host cores (rank 0 only).  The REAL lightkurve +
    astropy call chain when importable (kind "reference"); else the oracle's restatement of astropy's default method
    "fast" (kind "port" - astropy is in neither this image nor its wheelhouse).  Every step takes the next `n_lc`
    DISTINCT light curves of the full 1024-curve workload; value = the median step; 1-core and all-core rates."""
    if rank != 0:
        return
    name = args.workload if args.workload in ("c2", "c2_small") else "c2"
    w = WORKLOADS[name]
    from multiprocessing import get_context
    t, Y, freq = make_workload(name, args.seed)
    cores = _cores()
    real = _have_real_reference()
    n_lc = min(w["B"], max(cores, 8))
    f0, df, nf = float(freq[0]), float(freq[1] - freq[0]), len(freq)
    _REF.update(t=t, Y=Y, f0=f0, df=df, nf=nf, real=real)
    fn, job = _ref_index_worker, (lambda i: i)
    pool = get_context("fork").Pool(cores, initializer=_cpu_worker_init) if cores > 1 else None

    def step(k, n):
        jobs = [job(k * n + i) for i in range(n)]
        t0 = time.perf_counter()
        if pool is None:
            for j in jobs:
                fn(j)
        else:
            pool.map(fn, jobs, chunksize=1)
        return time.perf_counter() - t0

    for k in range(args.warmup):
        step(k, min(n_lc, cores))
    secs = [step(args.warmup + k, n_lc) for k in range(args.steps)]
    t0 = time.perf_counter()
    for i in range(2):
        fn(job(i))
    one_core = 2 * nf * len(t) / (time.perf_counter() - t0)
    if pool is not None:
        pool.close()
        pool.join()
    med = float(np.median(secs))
    val = nf * len(t) * n_lc / med
    how = ("lightkurve.LightCurve.to_periodogram(ls_method='fast') on astropy" if real else
           "astropy 'fast' (extirpolation + FFT) restated in oracle/ls.py")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * med,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: %s; CPU sample = %d distinct light curves per step" % (name, w["desc"], n_lc)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "reference" if real else "port",
                         "value_1core": one_core,
                         "sample": "%d distinct light curves of the %d-LC workload per step (median of %d steps; "
                                   "min %.0f / max %.0f ms), %s, pool of %d single-threaded processes; "
                                   "value = F*N*n/time (the FFT method does far less than F*N work)" %
                                   (n_lc, w["B"], args.steps, 1e3 * min(secs), 1e3 * max(secs), how, cores)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def make_workload_sample(name, seed, n_lc=16):
    """Same generator, but only the first `n_lc` light curves (the CPU legs never need the full batch)."""
    w = dict(WORKLOADS[name])
    full_B = w["B"]
    WORKLOADS["_sample"] = dict(w, B=min(n_lc, full_B))
    try:
        return make_workload("_sample", seed)
    finally:
        del WORKLOADS["_sample"]


def make_bls_workload(seed, B=256, N=20000, P=50000):
    """SURVEY.md 8(d) config C3 (BASELINE.json configs[2]): TESS 2-min sector t = 1325 + n/720 d with a 1-d
    mid-sector gap, N cadences; flux = 1 + N(0, 5e-4) with a box transit (P~U(1,8) d, depth~LogU(5e-4,1e-2),
    duration~U(0.05,0.3) d) in 75 % of the light curves; flux_err = 5e-4; 10 durations linspace(0.05, 0.33);
    P periods uniform in frequency between 1/9.26 and 1/0.3314 per day."""
    rng = np.random.default_rng(seed)
    t = 1325 + np.arange(N + 720) / 720.0
    t = np.concatenate([t[: N // 2], t[N // 2 + 720:]])[:N]
    fluxes, errs = [], []
    for b in range(B):
        y = 1 + 5e-4 * rng.normal(size=N)
        per0, dep, dur0 = rng.uniform(1, 8), 10 ** rng.uniform(np.log10(5e-4), -2), rng.uniform(0.05, 0.3)
        if b % 4 != 3:
            y[np.abs((t - t[0] - 0.7 + 0.5 * per0) % per0 - 0.5 * per0) < 0.5 * dur0] -= dep
        fluxes.append(y)
        errs.append(np.full(N, 5e-4))
    duration = np.linspace(0.05, 0.33, 10)
    period = 1.0 / np.linspace(1 / 0.3314, 1 / 9.26, P)
    return t, fluxes, errs, period, duration


def secondary_bls(engine, torch, dist, rank, world, dev, steps=2, cpu_baseline=True):
    """Second half of BASELINE.json's metric ("BLS periods/s"): configs[2] (256 TESS light curves x 20 000
    cadences x 50 000 trial periods x 10 durations per GPU; weak scaling by target, no collective - every
    (light curve, period) is independent and the 7 result arrays stay with the rank that owns the target).
    value = (light curve, period) pairs / s from the library's CUDA events around the search kernels (inputs
    resident), e2e = the same through the host-buffer C-ABI call (H2D of t/y/dy, D2H of the 7 [B, P] arrays)."""
    B, N, P = 256, 20000, 50000
    t, fluxes, errs, period, duration = make_bls_workload(1003 + rank, B, N, P)
    times = [t] * B
    engine.bls_power(times, fluxes, errs, period, duration)                     # warm-up (workspace growth)
    engine.profile_enable(True)
    l0 = engine.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = engine.bls_power(times, fluxes, errs, period, duration)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    launches = engine.launch_count() - l0
    kms = engine.profile_read()
    engine.profile_enable(False)
    tm = torch.tensor([float(np.mean(kms)), 1e3 * wall / steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    k_ms, e2e_ms = (float(x) for x in tm.tolist())
    pairs = float(B) * P * world
    out = {"metric": "bls_lc_period_pairs_per_s", "unit": "(LC,period)/s", "value": pairs / (k_ms * 1e-3),
           "ms_per_step": k_ms, "steps": steps, "n_gpus": world, "scaling": "weak", "dtype": "f64 sums, int32 bins",
           "config": {"workload": "c3: %d TESS LC (%d cadences) x %d periods x %d durations per GPU, oversample 10, "
                                  "objective likelihood" % (B, N, P, len(duration))},
           "e2e": {"value": pairs / (e2e_ms * 1e-3), "unit": "(LC,period)/s", "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": int(3 * 8 * B * N) * world, "d2h_bytes_per_step": int(7 * 8 * B * P) * world},
           "gpu_launches": int(launches),
           # K3 keeps the light curve on chip (DRAM 0.01 %, profiles/r01_bls_kernel_v2_boundary.md): the bound is
           # instruction issue.  33 450 warp instructions per (light curve, period), measured with ncu over ALL period
           # chunks of this workload's grid (profiles/r02_bls_instructions.csv); peak = SMs x 4 schedulers x max clock.
           "roofline": {"bound": "issue", "unit": "warp-instructions/s",
                        "achieved": BLS_WARP_INSTR_PER_PAIR * B * P / (k_ms * 1e-3),
                        "warp_instructions_per_pair": BLS_WARP_INSTR_PER_PAIR,
                        "compulsory_bytes_per_step": int(3 * 8 * B * N + 7 * 8 * B * P),
                        "effective_gbs_of_24N_plus_56": B * P * (24.0 * N + 56) / (k_ms * 1e-3) / 1e9,
                        "note": "issue-slot roofline (the SURVEY 8(d) streaming figure (24 N + 56) B per pair is kept as "
                                "effective_gbs...: the kernel never streams the light curve from HBM)"}}
    if rank == 0:
        pk = float(engine.sm_count()) * 4.0 * float(_peaks().get("sm_max_mhz", 1965.0)) * 1e6
        out["roofline"]["peak"] = pk
        out["roofline"]["frac"] = out["roofline"]["achieved"] / pk
        out["roofline"]["peak_source"] = "SM count x 4 warp schedulers x sm_max_mhz of MEASURED_PEAKS.json"
        if cpu_baseline:
            out.update(_bls_cpu_leg(t, fluxes, errs, period, duration, res, P))
    return out


def _bls_cpu_leg(t, fluxes, errs, period, duration, res, P, n_lc=4, budget_s=15.0):
    """CPU leg of the BLS line: astropy's bls.c restated in oracle/bls_c.c (OpenMP over periods, all host
    cores) on `n_lc` light curves x every `stride`-th period (stride chosen from a short probe so that the
    sample costs about `budget_s` seconds at most), plus a parity check of the GPU result on that sample."""
    try:
        from oracle import bls as obls
        t0 = time.perf_counter()
        obls.bls_power_c(t, fluxes[0], errs[0], period[::50], duration)
        rate = len(period[::50]) / (time.perf_counter() - t0)
        stride = max(1, int(np.ceil(n_lc * P / max(1.0, rate * budget_s))))
        sub = period[::stride]
        t0 = time.perf_counter()
        refs = [obls.bls_power_c(t, fluxes[b], errs[b], sub, duration) for b in range(n_lc)]
        secs = time.perf_counter() - t0
        ok = all(bool(np.allclose(res["power"][b][::stride], refs[b]["power"], rtol=1e-9, atol=0))
                 for b in range(n_lc))
        try:
            cores = len(os.sched_getaffinity(0))
        except Exception:
            cores = os.cpu_count() or 1
        return {"cpu_baseline": {"value": n_lc * len(sub) / secs, "unit": "(LC,period)/s", "cores": cores,
                                 "kind": "port",
                                 "sample": "%d of the 256 light curves x %d of the %d periods (every %d-th; %.2f s), "
                                           "astropy bls.c restated in oracle/bls_c.c, OpenMP over periods"
                                           % (n_lc, len(sub), P, stride, secs)},
                "parity_on_sample": ok}
    except Exception as e:                                                      # pragma: no cover
        return {"cpu_baseline": {"error": repr(e)}}



def make_c5_workload(seed, B=16384, F=20000, only=None):
    """SURVEY.md 8(d) config C5 (BASELINE.json configs[4]): per light curve N_b ~ round(LogU(2000, 20000)) cadences of a
    TESS-like 2-min grid over 27.8 d after a seeded random deletion, U(-20 s, 20 s) jitter (irregular: no shared grid);
    flux = 1 + sinusoid + noise, fp32; one common regular frequency grid of F bins up to 50 / d (f0 = df).
    `only` (index array): generate the flux of these light curves only (the others keep their times - the sharding
    needs every length - and get a zero-length placeholder flux)."""
    rng = np.random.default_rng(seed)
    grid = 1325 + np.arange(int(27.8 * 720)) / 720.0
    ns = np.minimum(len(grid), np.round(10 ** rng.uniform(np.log10(2000), np.log10(20000), B)).astype(int))
    want = np.ones(B, bool) if only is None else np.isin(np.arange(B), only)
    times, fluxes = [], []
    for b in range(B):
        r = np.random.default_rng([seed, b])
        if not want[b]:
            times.append(np.empty(int(ns[b]), dtype=np.float64))       # length only
            fluxes.append(np.empty(0, dtype=np.float32))
            continue
        keep = np.sort(r.choice(len(grid), int(ns[b]), replace=False))
        t = grid[keep] + r.uniform(-20, 20, int(ns[b])) / 86400.0
        times.append(t)
        fluxes.append((1 + 10 ** r.uniform(-4, -2) * np.sin(2 * np.pi * r.uniform(0.05, 20) * t + r.uniform(0, 6.28))
                       + 10 ** r.uniform(np.log10(5e-5), -3) * r.standard_normal(int(ns[b]))).astype(np.float32))
    freq = np.linspace(50.0 / F, 50.0, F)
    return times, fluxes, freq


def make_c4_workload(seed, B, N=65000, K=151):
    """SURVEY.md 8(d) config C4 (BASELINE.json configs[3]): Kepler-like shared grid of N cadences; X = K - 1 orthonormalised
    seeded random-walk "CBVs" + a constant column; flux = 1 + X w_b + slow trend + N(0, sigma) + 0.3 % outliers at
    8 sigma; flux_err ~ sigma U(0.8, 1.2)."""
    rng = np.random.default_rng(seed)
    keep = np.sort(rng.choice(71500, N, replace=False))
    tt = 131.5 + keep * 0.0204336
    X = np.cumsum(rng.normal(size=(N, K - 1)), axis=0)
    X, _ = np.linalg.qr(X - X.mean(0))
    X = np.hstack([X * np.sqrt(N), np.ones((N, 1))])
    W = rng.normal(size=(B, K)) * 1e-3
    slow = np.cumsum(rng.normal(size=N)) * 1e-5
    Y = np.empty((B, N))
    FE = np.empty((B, N))
    for b0 in range(0, B, 256):
        nb = min(256, B - b0)
        Y[b0:b0 + nb] = 1 + W[b0:b0 + nb] @ X.T + slow[None, :] + 3e-4 * rng.standard_normal((nb, N))
        FE[b0:b0 + nb] = 3e-4 * rng.uniform(0.8, 1.2, (nb, N))
    out = rng.integers(0, N, (B, N // 300))
    Y[np.arange(B)[:, None], out] += 8 * 3e-4
    return tt, X, Y, FE


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def power_sample(power, max_bytes=48 << 20, seed=0):
    """Host copy of a fixed, seeded sample of the rows of a [B, F] float32 power tensor: every row when they fit in
    `max_bytes`, else as many distinct rows (in ascending order) as do.  Same B, F and seed: same rows."""
    import torch
    B, F = power.shape
    n = min(B, max(1, max_bytes // (4 * F)))
    rows = np.arange(B) if n == B else np.sort(np.random.default_rng(seed).choice(B, n, replace=False))
    return power.index_select(0, torch.as_tensor(rows, device=power.device)).cpu().numpy()


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _max_over_ranks(torch, dist, world, dev, vals):
    tm = torch.tensor([float(v) for v in vals], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    return [float(x) for x in tm.tolist()]


def c5_step_stats(engine, torch, dist, rank, world, dev, times, fluxes, freq, steps, warmup, chunks=4,
                  sample_power=False):
    """Device-resident sharded ragged Lomb-Scargle (lightkurve_b200.dist.ShardedLombScargle): per step compute of this
    rank's shard + the pipelined all-gathers + restoring the target order.  Returns ms (device events, max over
    ranks) for the resident step and for the end-to-end step (pinned H2D of the shard, the step, D2H of the whole
    gathered power array on every rank); with `sample_power`, also `power_sample` of the last resident step's output."""
    from lightkurve_b200.dist import ShardedLombScargle
    job = ShardedLombScargle(times, fluxes, freq, "amplitude", chunks=chunks, device=dev)
    job.upload()
    h_out = torch.empty((job.n_total, job.F), dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(n):
            fn()
        ev1.record()
        barrier()
        return ev0.elapsed_time(ev1) / n

    def step_e2e():
        job.upload()
        out = job.run()
        h_out.copy_(out, non_blocking=True)

    last = {}

    def step_resident():
        last["power"] = job.run()

    for _ in range(warmup):
        job.run()
    engine.profile_enable(True)
    l0 = engine.launch_count()
    ms_res = timed(step_resident, steps)
    launches = (engine.launch_count() - l0) // max(1, steps)
    kms = engine.profile_read()
    engine.profile_enable(False)
    sample = power_sample(last["power"]) if sample_power else None
    step_e2e()
    ms_e2e = timed(step_e2e, steps)
    k_ms = float(np.sum(kms)) / max(1, steps) if len(kms) else float("nan")      # all pieces of one step
    ms_res, ms_e2e, k_ms = _max_over_ranks(torch, dist, world, dev, [ms_res, ms_e2e, k_ms])
    mine = job.shards[rank]
    return dict(ms=ms_res, ms_e2e=ms_e2e, kernel_ms=k_ms, launches=int(launches), family=engine.ls_last_algo(),
                h2d=job.h2d_bytes, d2h=int(job.n_total) * job.F * 4, n_local=len(mine), job=job, power_sample=sample)


def _ragged_cpu_leg(times, fluxes, freq, n_lc=48, budget_s=12.0):
    """Reference default (astropy 'fast' restated in oracle/ls.py) on a sample of the ragged light curves, 1 core."""
    from oracle import ls as ols
    f0, df, nf = float(freq[0]), float(freq[1] - freq[0]), len(freq)
    idx = [i for i in range(len(times)) if len(fluxes[i]) == len(times[i])][:n_lc]
    t0 = time.perf_counter()
    units = 0
    done = 0
    for i in idx:
        ols.ls_fast_psd(times[i], fluxes[i].astype(np.float64), f0, df, nf)
        units += nf * len(times[i])
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    secs = time.perf_counter() - t0
    return {"value": units / secs, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d of the light curves (%.1f s), astropy method='fast' (lightkurve default) restated in oracle/ls.py, "
                      "1 process; equivalent bin*cadence/s = F*sum(N)/time" % (done, secs)}


def _nufft_fine_log2(kmax_plus_1):
    """log2 of the NUFFT fine grid (ls_nufft.cu: fine_log2): the smallest power of two with an upsampling factor of at
    least LKB_NUFFT_SIGMA (default 2) over the highest mode."""
    smin = min(2.0, max(1.25, float(os.environ.get("LKB_NUFFT_SIGMA", "2"))))
    return max(4, int(np.ceil(np.log2(2.0 * smin * kmax_plus_1))))


def _ragged_roofline(F, units, k_ms, family, n_local, clocks_mhz=None):
    """K1's bounds (DESIGN.md): the direct kernel is issue/MUFU-bound (SURVEY 8d: 2.3e12 units/s at 1965 MHz); the
    NUFFT family is an HBM/L2 sweep of the fine grids."""
    pk = _peaks()
    hbm = float(pk.get("hbm_gbs", 6589.3))
    if family == "nufft":
        p = _nufft_fine_log2(1 + F)
        M, M2 = 2 ** p, 2 ** (p + 1)
        npairs = (n_local + 1) // 2
        # per pair: flux grid T written + read, pruned modes written + read (<= M / 2), the same on the 2x finer grid
        nbytes = npairs * 8.0 * (2.5 * M + 2.5 * M2) + 4.0 * n_local * F
        return {"bound": "hbm", "unit": "GB/s", "achieved": nbytes / (k_ms * 1e-3) / 1e9, "peak": hbm,
                "frac": nbytes / (k_ms * 1e-3) / 1e9 / hbm, "traffic": None, "kernel_ms": k_ms,
                "kernel": "nufft2_spread_ragged + cols + rows (flux and window grids) + nufft_finish_ragged",
                "note": "algorithmic bytes per pair of light curves: column transforms written + read and the kept modes "
                        "written + read on the flux grid (2^%d cells) and the window grid (2^%d), + power; spread reads "
                        "(cadence tables, flux) not counted" % (p, p + 1)}
    ceil_units = 2.3e12
    return {"bound": "issue", "unit": "bin*cadence/s", "achieved": units / (k_ms * 1e-3), "peak": ceil_units,
            "frac": units / (k_ms * 1e-3) / ceil_units, "traffic": None, "kernel_ms": k_ms, "kernel": "ls_direct_kernel",
            "note": "SURVEY 8(d) K1 ceiling: 2 MUFU + ~12 FMA-pipe slots per bin x cadence at 1965 MHz"}


def secondary_ls_ragged(engine, torch, dist, rank, world, dev, steps=3, cpu_baseline=True):
    """BASELINE.json configs[4] share: every rank takes 2048 of the ragged light curves (16384 / 8; at --gpus 8 this IS
    config 5 with the all-gathers inside the step), F = 20000."""
    B = 2048 * world
    times, fluxes, freq = make_c5_workload(1005, B=B)
    st = c5_step_stats(engine, torch, dist, rank, world, dev, times, fluxes, freq, steps, warmup=2)
    units = float(len(freq)) * float(sum(len(t) for t in times))
    mine = st["job"].shards[rank]
    units_local = float(len(freq)) * float(sum(len(times[i]) for i in mine))
    out = {"metric": METRIC, "unit": UNIT, "value": units / (st["ms"] * 1e-3), "ms_per_step": st["ms"], "steps": steps,
           "n_gpus": world, "scaling": "weak", "dtype": "f32 spreading + FFT, f64 tables" if st["family"] == "nufft"
           else "f32 sums flushed to f64, fixed-point phases",
           "config": {"workload": "c5 share: %d ragged LC per GPU (2000..20000 cadences) x %d frequencies, sharded by "
                                  "target, %d pipelined all-gather(s) of the power rows per step" %
                                  (2048, len(freq), st["job"].chunks if world > 1 else 0), "kernel_family": st["family"]},
           "e2e": {"value": units / (st["ms_e2e"] * 1e-3), "unit": UNIT, "ms_per_step": st["ms_e2e"],
                   "h2d_bytes_per_step": st["h2d"] * world, "d2h_bytes_per_step": st["d2h"] * world},
           "gpu_launches": st["launches"],
           "roofline": _ragged_roofline(len(freq), units_local, st["kernel_ms"], st["family"], st["n_local"])}
    if rank == 0 and cpu_baseline:
        out["cpu_baseline"] = _ragged_cpu_leg(times, fluxes, freq)
    return out


def secondary_flatten(engine, torch, dist, rank, world, dev, cpu_baseline=True, B=4096):
    """BASELINE.json configs[3], first half: LightCurve.flatten(window_length=401) of 4096 Kepler-length light curves
    per GPU (weak scaling by target; no collective).  value = light curves / s from the library's CUDA events around
    the flatten kernel; e2e = the host-buffer C-ABI call (page-locked in/out arrays: 6.4 GB up, 6.4 GB down)."""
    N = 65000
    tt, _, Y, FE = make_c4_workload(1004 + rank, B, N, K=3)
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    t_cat = pin(np.tile(tt, B))
    f_cat = pin(Y.reshape(-1))
    fe_cat = pin(FE.reshape(-1))
    offsets = np.arange(B + 1, dtype=np.int64) * N
    outs = [pin(np.empty(B * N)) for _ in range(3)]
    call = lambda: engine.flatten_csr(t_cat, f_cat, fe_cat, None, offsets, window_length=401, flat=outs[0],
                                      flat_err=outs[1], trend=outs[2])
    call()                                                                       # warm-up (workspace growth)
    engine.profile_enable(True)
    l0 = engine.launch_count()
    t0 = time.perf_counter()
    call()
    wall = time.perf_counter() - t0
    launches = engine.launch_count() - l0
    kms = engine.profile_read()
    engine.profile_enable(False)
    k_ms, e2e_ms = _max_over_ranks(torch, dist, world, dev, [float(np.sum(kms)), 1e3 * wall])
    hbm = float(_peaks().get("hbm_gbs", 6589.3))
    nbytes = 63.0 * N * B
    out = {"metric": "flatten_light_curves_per_s", "unit": "LC/s", "value": B * world / (k_ms * 1e-3), "ms_per_step": k_ms,
           "steps": 1, "n_gpus": world, "scaling": "weak", "dtype": "f64",
           "config": {"workload": "c4a: flatten(window_length=401, polyorder=2, niters=3, sigma=3) of %d LC x %d cadences "
                                  "per GPU" % (B, N)},
           "e2e": {"value": B * world / (e2e_ms * 1e-3), "unit": "LC/s", "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": int(3 * 8 * B * N) * world, "d2h_bytes_per_step": int(3 * 8 * B * N) * world},
           "gpu_launches": int(launches),
           "roofline": {"bound": "hbm", "unit": "GB/s", "achieved": nbytes / (k_ms * 1e-3) / 1e9, "peak": hbm,
                        "frac": nbytes / (k_ms * 1e-3) / 1e9 / hbm, "traffic": None, "kernel_ms": k_ms,
                        "note": "SURVEY 8(d) algorithmic bytes 63*N per light curve"}}
    if rank == 0 and cpu_baseline:
        from oracle import detrend as odet
        n_lc, t0 = 0, time.perf_counter()
        ok = True
        while n_lc < 16 and time.perf_counter() - t0 < 12.0:
            rf, _, rt = odet.flatten(tt, Y[n_lc], FE[n_lc], window_length=401)
            ok = ok and bool(np.allclose(outs[2][n_lc * N:(n_lc + 1) * N], rt, rtol=1e-5, atol=0))
            n_lc += 1
        secs = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n_lc / secs, "unit": "LC/s", "cores": 1, "kind": "reference",
                               "sample": "%d of the %d light curves (%.1f s): the reference's own flatten body on the real "
                                         "scipy.signal.savgol_filter / scipy.interpolate.interp1d (oracle/detrend.py), "
                                         "1 core" % (n_lc, B, secs)}
        out["parity_on_sample"] = ok
    return out


def secondary_regress(engine, torch, dist, rank, world, dev, cpu_baseline=True, B=4096):
    """BASELINE.json configs[3], second half: RegressionCorrector.correct (sigma = 5, niters = 5) of 4096 light curves
    against one shared design matrix of 150 CBV-like regressors + constant (K = 151)."""
    N, K = 65000, 151
    tt, X, Y, FE = make_c4_workload(1004 + rank, B, N, K)
    call = lambda: engine.regress(X, Y, FE, None, np.zeros(K), np.full(K, np.inf), sigma=5, niters=5)
    engine.regress(X, Y[:64], FE[:64], None, np.zeros(K), np.full(K, np.inf), sigma=5, niters=5)      # warm-up (kernels)
    call()               # warm-up at full size: the workspace pool grows to its final ~20 GB here (cudaMalloc inside a
    #                      timed call cost 0.17 s on a fresh box: 470 instead of 298 ms)
    engine.profile_enable(True)
    l0 = engine.launch_count()
    t0 = time.perf_counter()
    res = call()
    wall = time.perf_counter() - t0
    launches = engine.launch_count() - l0
    kms = engine.profile_read()
    engine.profile_enable(False)
    # the library records two intervals per call: the first Gram pass (the roofline kernel) and everything after it
    k_ms, dev_ms, e2e_ms = _max_over_ranks(torch, dist, world, dev, [float(kms[0]) if len(kms) else 0.0,
                                                                     float(np.sum(kms)), 1e3 * wall])
    pk = _peaks()
    flops = float(B) * N * K * K                      # symmetric half of X^T W X, once (later iterations downdate)
    out = {"metric": "regression_light_curves_per_s", "unit": "LC/s", "value": B * world / (dev_ms * 1e-3),
           "ms_per_step": dev_ms, "steps": 1, "n_gpus": world, "scaling": "weak",
           "dtype": "split-f16 tcgen05 Gram + f64 refinement (DMMA right-hand sides, LU)",
           "config": {"workload": "c4b: RegressionCorrector.correct(sigma=5, niters=5), %d LC x %d cadences, shared "
                                  "design matrix K = %d, per-cadence flux_err" % (B, N, K)},
           "e2e": {"value": B * world / (e2e_ms * 1e-3), "unit": "LC/s", "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": int(8 * (2 * B * N + N * K)) * world,
                   "d2h_bytes_per_step": int(8 * B * (N + K) + B * N) * world},
           "gpu_launches": int(launches),
           "roofline": {"bound": "tensor", "unit": "TFLOP/s", "achieved": flops / (k_ms * 1e-3) / 1e12,
                        "peak": float(pk.get("bf16_tflops_sustained", 1370.0)),
                        "frac": flops / (k_ms * 1e-3) / 1e12 / float(pk.get("bf16_tflops_sustained", 1370.0)),
                        "traffic": None, "kernel_ms": k_ms,
                        "kernel": "regress_tc_gram: rt_gram_kernel (tcgen05, split-f16 operands, f32 TMEM accumulators) + "
                                  "operand preparation + the DMMA right-hand side",
                        "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (dense 16-bit tensor-core rate; the "
                                        "kernel issues 3 f16 MMAs per algorithmic product: hi*hi, hi*lo, lo*hi)")
                                       if pk else "fallback 1370 TF/s (B200_PROFILING.md)",
                        "note": "algorithmic flops N*K^2 per light curve (symmetric half of X^T W X, first iteration; "
                                "later iterations downdate the clipped rows on the FP64 tensor cores); round 1's FP64 DMMA "
                                "Gram ran at 16 TF/s of a measured 37.1 TF/s FP64 peak"}}
    if rank == 0 and cpu_baseline:
        from oracle import detrend as odet
        n_lc, t0 = 0, time.perf_counter()
        ok = True
        while n_lc < 8 and time.perf_counter() - t0 < 15.0:
            ref = odet.regress(X, Y[n_lc], FE[n_lc], None, np.zeros(K), np.full(K, np.inf), sigma=5, niters=5)
            ok = ok and bool(np.array_equal(res["outlier_mask"][n_lc], ref["outlier_mask"])) and \
                bool(np.allclose(res["coefficients"][n_lc], ref["coefficients"], rtol=1e-6, atol=1e-9))
            n_lc += 1
        secs = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n_lc / secs, "unit": "LC/s", "cores": _cores(), "kind": "reference",
                               "sample": "%d of the %d light curves (%.1f s): the reference's correct() loop on the real "
                                         "numpy.linalg.solve / BLAS (oracle/detrend.py), BLAS threads = all cores"
                                         % (n_lc, B, secs)}
        out["parity_on_sample"] = ok
    return out


def run_c5(args, engine, torch, dist, rank, world, local_rank, dev):
    """--workload c5: BASELINE.json configs[4] as a STRONG-scaling job - the same 16384 light curves whatever the
    number of ranks; every rank computes its shard and pipelined all-gathers reassemble [16384, 20000] everywhere."""
    w = WORKLOADS[args.workload]
    B, F = w["B"], w["F"]
    lens_only = make_c5_workload(args.seed + 3, B=B, F=F, only=np.zeros(0, int))[0]
    from lightkurve_b200.dist import shard_by_length
    mine = shard_by_length([len(t) for t in lens_only], world)[rank]
    times, fluxes, freq = make_c5_workload(args.seed + 3, B=B, F=F, only=mine)
    for i in range(B):                       # the other ranks' light curves: lengths only (never uploaded here)
        if len(fluxes[i]) != len(times[i]):
            fluxes[i] = np.empty(len(times[i]), dtype=np.float32)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    st = c5_step_stats(engine, torch, dist, rank, world, dev, times, fluxes, freq, args.steps, args.warmup,
                       chunks=args.chunks if args.chunks > 0 else 4, sample_power=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop() if sampler else None
    units = float(F) * float(sum(len(t) for t in times))
    if rank != 0:
        return
    units_local = float(F) * float(sum(len(times[i]) for i in mine))
    cpu = None
    if not args.no_cpu_baseline:
        cpu = _ragged_cpu_leg([times[i] for i in mine], [fluxes[i] for i in mine], freq)
    line = {"metric": METRIC, "value": units / (st["ms"] * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": st["ms"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 spreading + FFT, f64 tables" if st["family"] == "nufft" else "f32/f64 direct sums",
            "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, w["desc"]), "light_curves": B, "frequencies": F,
                       "cadences_total": int(sum(len(t) for t in times)), "normalization": "amplitude",
                       "kernel_family": st["family"], "pieces": st["job"].chunks,
                       "sharding": "by target (sorted by length, round-robin), %d rank(s); per step %d asynchronous "
                                   "all-gather(s) of [%d x %d] fp32 blocks overlapped with the next piece's kernels" %
                                   (world, st["job"].chunks if world > 1 else 0, world * (st["job"].bounds[0][1]), F),
                       "l2": "the fine grids of one piece exceed the 126 MB L2"},
            "e2e": {"value": units / (st["ms_e2e"] * 1e-3), "unit": UNIT, "ms_per_step": st["ms_e2e"],
                    "h2d_bytes_per_step": st["h2d"] * world, "d2h_bytes_per_step": st["d2h"] * world,
                    "note": "pinned H2D of every rank's shard, the step, D2H of the whole [B, F] power array on every rank"},
            "gpu_launches": st["launches"],
            "roofline": _ragged_roofline(F, units_local, st["kernel_ms"], st["family"], st["n_local"]),
            "cpu_baseline": cpu, "clocks": clocks}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"power": st["power_sample"]})
    print(json.dumps(line), flush=True)

def nufft_leg_child(args):
    """Child process of the `secondary.ls_nufft` leg: the opt-in NUFFT Lomb-Scargle path (DESIGN.md K2n) on the same
    configs[1] workload, device-resident, CUDA-event timed, with a parity check against the default path on a sample
    of light curves.  Runs in its own process so that a fault of the not-yet-hardware-validated path cannot touch
    the headline measurement.  Prints one JSON line."""
    import torch
    from lightkurve_b200 import engine
    torch.cuda.set_device(0)
    engine.init(0)
    w = WORKLOADS[args.workload]
    B, N, F = w["B"], w["N"], w["F"]
    t, Y, freq = make_workload(args.workload, args.seed)
    dev = torch.device("cuda", 0)
    d_t, d_f, d_Y = torch.tensor(t, device=dev), torch.tensor(freq, device=dev), torch.tensor(Y, device=dev)
    d_ref = torch.empty((B, F), dtype=torch.float32, device=dev)
    engine.ls_power_shared(d_t, d_Y, d_f, "amplitude", algo="auto", out=d_ref)
    torch.cuda.synchronize()
    ref = d_ref[:: max(1, B // 16)].cpu().numpy().astype(np.float64)
    out = {"workload": "%s: %s" % (args.workload, w["desc"]), "modes": {}}
    modes = {"global passes": {}, "global passes, twiddle chain": {"LKB_NUFFT_TWIDDLE_CHAIN": "1"},
             "four-step smem, chain": {"LKB_NUFFT_TWIDDLE_CHAIN": "1", "LKB_NUFFT_FFT": "smem"},
             "four-step fused spread, chain": {"LKB_NUFFT_TWIDDLE_CHAIN": "1", "LKB_NUFFT_FFT": "fused"}}
    d_P = torch.empty((B, F), dtype=torch.float32, device=dev)
    for name, env in modes.items():
        for k in ("LKB_NUFFT_TWIDDLE_CHAIN", "LKB_NUFFT_FFT"):
            os.environ.pop(k, None)
        os.environ.update(env)
        try:
            os.environ["LKB_NUFFT_VERIFY"] = "1"          # built-in self-check during the warm-up calls only
            for _ in range(2):
                engine.ls_power_shared(d_t, d_Y, d_f, "amplitude", algo="nufft", out=d_P)
            torch.cuda.synchronize()
            os.environ.pop("LKB_NUFFT_VERIFY", None)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(args.steps):
                engine.ls_power_shared(d_t, d_Y, d_f, "amplitude", algo="nufft", out=d_P)
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / args.steps
            got = d_P[:: max(1, B // 16)].cpu().numpy().astype(np.float64)
            excess = float(np.max(np.abs(got - ref) / (1e-5 * ref.max(axis=1, keepdims=True) + 1e-4 * ref)))
            out["modes"][name] = {"ms_per_step": ms, "value": float(F) * N * B / (ms * 1e-3), "unit": UNIT,
                                  "worst_tolerance_excess_vs_default_path": excess, "parity": bool(excess < 1.5)}
        except Exception as e:
            out["modes"][name] = {"error": repr(e)}
    print(json.dumps(out), flush=True)


def nufft_leg(args):
    """Parent side: run `nufft_leg_child` in a subprocess with a timeout; never raises."""
    import subprocess
    try:
        cp = subprocess.run([sys.executable, os.path.abspath(__file__), "--nufft-leg", "--steps", str(max(2, args.steps)),
                             "--workload", args.workload, "--seed", str(args.seed)], capture_output=True, text=True,
                            timeout=180, env={k: v for k, v in os.environ.items()
                                              if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")})
        lines = [ln for ln in cp.stdout.strip().splitlines() if ln.startswith("{")]
        if cp.returncode != 0 or not lines:
            return {"error": "child exit code %d: %s" % (cp.returncode, (cp.stderr or "")[-400:])}
        res = json.loads(lines[-1])
        res["note"] = ("opt-in path (algo='nufft'), not the reported metric: measured in a child process after the "
                       "headline timing; parity = against the default path on 16 light curves (two fp32 paths, "
                       "so up to 1.5x the single-path tolerance)")
        return res
    except Exception as e:                                        # timeout, JSON error, ...
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--algo", default="auto", choices=["auto", "simt", "tcgen05", "nufft"],
                    help="nufft: the opt-in spread+FFT path (ls_nufft.cu); its roofline is the HBM one")
    ap.add_argument("--seed", type=int, default=1002)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary legs (BLS, flatten, regression, ragged LS)")
    ap.add_argument("--legs", default="bls,flatten,regress,ls_ragged", help="comma list of secondary legs to run")
    ap.add_argument("--chunks", type=int, default=0,
                    help="N > 1: pieces per rank, one asynchronous all-gather each (0 = by rank count: c2 1 / 2 / 4 pieces at "
                         "<= 2 / <= 4 / more ranks, c5 4)")
    ap.add_argument("--nufft-leg", action="store_true", help=argparse.SUPPRESS)      # internal: child of secondary.ls_nufft
    ap.add_argument("--nufft-variants", action="store_true",
                    help="also time the NUFFT path's transform variants in a child process (secondary.ls_nufft)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the power rows of the last step (a fixed, seeded sample of at "
                         "most 48 MB) to DIR/power.npy, float32, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.nufft_leg:
        nufft_leg_child(args)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    from lightkurve_b200 import engine

    assert torch.cuda.is_available(), "bench.py (our arm) needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    engine.init(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    dev = torch.device("cuda", local_rank)
    if args.workload.startswith("c5"):
        run_c5(args, engine, torch, dist, rank, world, local_rank, dev)
        if world > 1:
            dist.destroy_process_group()
        return
    w = WORKLOADS[args.workload]
    B, N, F = w["B"], w["N"], w["F"]
    t, Y, freq = make_workload(args.workload, args.seed + rank)      # every rank: its own 1024 targets
    d_t = torch.tensor(t, device=dev)
    d_f = torch.tensor(freq, device=dev)
    d_Y = torch.tensor(Y, device=dev)
    d_P = torch.empty((B, F), dtype=torch.float32, device=dev)
    d_all = torch.empty((world * B, F), dtype=torch.float32, device=dev) if world > 1 else None
    h_Y = torch.from_numpy(Y).pin_memory()
    h_P = torch.empty((B, F), dtype=torch.float32).pin_memory()

    # N > 1: the rank's batch goes through the library in `pieces` calls on the same grid (the y-independent tables are
    # built once and found cached by the later calls) and every piece's power rows are handed to an ASYNCHRONOUS
    # all-gather while the next piece is computed; the gathered array is piece-major: [piece][rank][B / pieces, F]
    auto_pieces = 1 if world <= 2 else (2 if world <= 4 else 4)   # the all-gather volume per rank grows with world - 1
    pieces = max(1, min(args.chunks if args.chunks > 0 else auto_pieces, B // 64)) if world > 1 else 1
    pb_rows = B // pieces
    assert pb_rows * pieces == B
    s_h2d, s_d2h = torch.cuda.Stream(), torch.cuda.Stream()

    def step_resident():
        if world == 1:
            engine.ls_power_shared(d_t, d_Y, d_f, "amplitude", algo=args.algo, out=d_P)
            return
        works = []
        for c in range(pieces):
            rows = slice(c * pb_rows, (c + 1) * pb_rows)
            engine.ls_power_shared(d_t, d_Y[rows], d_f, "amplitude", algo=args.algo, out=d_P[rows])
            works.append(dist.all_gather_into_tensor(d_all[c * world * pb_rows:(c + 1) * world * pb_rows], d_P[rows],
                                                     async_op=True))
        for wk in works:
            wk.wait()

    h_Y_np, h_P_np = h_Y.numpy(), h_P.numpy()                 # numpy views of the page-locked buffers

    def step_e2e():
        if world == 1:
            # the reference-facing call with HOST buffers: the C ABI stages the flux rows up and the power rows
            # down itself (chunk-pipelined over light-curve tiles, two copy streams) and returns synchronised
            engine.ls_power_shared(t, h_Y_np, freq, "amplitude", algo=args.algo, out=h_P_np)
            return
        cur = torch.cuda.current_stream()
        ev_in = []
        s_h2d.wait_stream(cur)
        with torch.cuda.stream(s_h2d):                        # H2D of this step's inputs (pinned), piece by piece
            for c in range(pieces):
                rows = slice(c * pb_rows, (c + 1) * pb_rows)
                d_Y[rows].copy_(h_Y[rows], non_blocking=True)
                e = torch.cuda.Event()
                e.record(s_h2d)
                ev_in.append(e)
        works = []
        for c in range(pieces):
            rows = slice(c * pb_rows, (c + 1) * pb_rows)
            cur.wait_event(ev_in[c])
            engine.ls_power_shared(d_t, d_Y[rows], d_f, "amplitude", algo=args.algo, out=d_P[rows])
            works.append(dist.all_gather_into_tensor(d_all[c * world * pb_rows:(c + 1) * world * pb_rows], d_P[rows],
                                                     async_op=True))
            s_d2h.wait_stream(cur)
            with torch.cuda.stream(s_d2h):                    # D2H of this rank's result rows (pinned)
                h_P[rows].copy_(d_P[rows], non_blocking=True)
        for wk in works:
            wk.wait()
        cur.wait_stream(s_d2h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        step_resident()
    barrier()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    engine.profile_enable(True)
    l0 = engine.launch_count()
    ms_res = timed(step_resident, args.steps)
    launches = engine.launch_count() - l0
    kms = engine.profile_read()
    engine.profile_enable(False)
    clocks = sampler.stop() if sampler else None
    family = engine.ls_last_algo()             # what `auto` resolved to: "nufft", "tcgen05" or "simt"
    escalated = engine.ls_last_escalated()     # light curves of the last step that took the double-precision pass
    # the last resident step's power rows (the path of the reported value), copied before the end-to-end steps run
    dumped = power_sample(d_P) if args.dump_outputs and rank == 0 else None

    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)

    secondary = None
    if not args.no_secondary and args.workload == "c2":
        secondary = {}
        del d_Y, d_P, d_all, h_Y, h_P, h_Y_np, h_P_np               # the legs bring their own buffers
        torch.cuda.empty_cache()
        legs = {"bls": secondary_bls, "flatten": secondary_flatten, "regress": secondary_regress,
                "ls_ragged": secondary_ls_ragged}
        for name in [x for x in args.legs.split(",") if x]:
            try:
                secondary[name] = legs[name](engine, torch, dist, rank, world, dev, cpu_baseline=not args.no_cpu_baseline)
            except Exception as e:                                # the headline line must survive every leg
                secondary[name] = {"error": repr(e)}
        if world == 1 and rank == 0 and args.nufft_variants:
            secondary["ls_nufft"] = nufft_leg(args)

    units_per_step = float(F) * N * B * world
    value = units_per_step * args.steps / (ms_res * 1e-3)
    e2e = units_per_step * args.steps / (ms_e2e * 1e-3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained"
        k_ms = float(np.mean(kms)) if len(kms) else float("nan")
        flops = 4.0 * F * N * B                                # algorithmic: 2 (cos,sin) x 2 flop per MAC
        achieved = flops / (k_ms * 1e-3) / 1e12
        traffic = None
        try:      # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "bench_kernel_traffic.json")))
            if args.workload == "c2" and family == "tcgen05":
                traffic = tj["ls_tcg_kernel"]["traffic_bytes_per_launch"]
        except Exception:
            pass
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved / peak_tf, "traffic": traffic,
                    "traffic_source": "static: one ncu --set full capture of this kernel on this workload, committed as "
                                      "profiles/bench_kernel_traffic.json (not re-measured in this run)" if traffic else None,
                    "kernel": "ls_tcg_kernel" if family == "tcgen05" else "ls_shared_simt_kernel", "kernel_ms": k_ms,
                    "peak_source": peak_src,
                    "note": "algorithmic flops 4*F*N*B; the split-fp16 scheme issues 3x that on the tensor pipe"}
        if family == "nufft" and not os.environ.get("LKB_NUFFT_FFT"):
            # v2 transform (nufft_v2.cuh): per light curve the centred flux is read by the spreading, the pruned fine
            # grid G (n1max rows of 512 complex cells) and the column transforms T (M / 2 complex points) are written
            # once and read once, the power row is written once (DESIGN.md K2n byte model; tables are L2-resident)
            pfine = _nufft_fine_log2(1 + F)
            Mh = 2 ** (pfine - 1)
            reach = freq[0] * (t[-1] - t[0]) * 2 ** pfine + 16
            n1max = int(np.ceil(np.ceil(reach / 2) / 512))
            nbytes = B * (4.0 * N + 2 * 8.0 * n1max * 512 + 2 * 8.0 * Mh + 4.0 * F)
            hbm = float(peaks.get("hbm_gbs", 6589.3))
            roofline = {"bound": "hbm", "achieved": nbytes / (k_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                        "frac": nbytes / (k_ms * 1e-3) / 1e9 / hbm,
                        # DRAM bytes of the four batch kernels of one step at this exact shape, from the committed ncu
                        # capture (spread 0.66 + cols 2.52 + rows 2.55 + low rows 0.28 GB): 1.03x the algorithmic bytes
                        "traffic": 6.003e9 if (B, N, F) == (1024, 65000, 100000) else None,
                        "traffic_source": "static: ncu --set full dram__bytes_read+write per launch, "
                                          "profiles/r02_nufft_v2_realmode_b.json (not re-measured in this run)",
                        "kernel": "nufft2_spread + nufft2_cols + nufft2_rows(finish) + nufft2_lowrows", "kernel_ms": k_ms,
                        "bytes_per_launch": nbytes,
                        "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
                        "note": "algorithmic bytes per light curve = 4 N (flux) + 2 x 8 x %d (pruned grid, written + read) + "
                                "2 x 8 x %d (column transforms, written + read) + 4 F (power)" % (n1max * 512, Mh)}
        elif family == "nufft":
            # HBM sweep: fine grids [B/2, M] complex64 written once by the spreading, read + written by every Stockham
            # pass, two modes per output read by the finish kernel; flux read once, power written once
            # (DESIGN.md K2n).  k0 = 1 on the bench grid (f0 = df).
            pfine = _nufft_fine_log2(1 + F)
            npass = (pfine + 3) // 4
            npairs = (B + 1) // 2
            nbytes = npairs * (2 ** pfine) * 8.0 * (1 + 2 * npass) + npairs * 16.0 * F + 4.0 * B * N + 4.0 * B * F
            hbm = float(peaks.get("hbm_gbs", 6589.3))
            roofline = {"bound": "hbm", "achieved": nbytes / (k_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                        "frac": nbytes / (k_ms * 1e-3) / 1e9 / hbm, "traffic": None,
                        "kernel": "nufft_spread + %d nufft_fft_pass + nufft_finish" % npass, "kernel_ms": k_ms,
                        "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
                        "note": "algorithmic bytes = fine grids (1 + 2 passes) + unpack reads + flux + power"}
        cpu = None
        if not args.no_cpu_baseline:
            n_cpu = min(B, 96)                                  # ~13 s of one core at config 2
            ts, Ys, fs = t, Y[:n_cpu], freq
            rate, secs = cpu_reference_rate(ts, Ys, fs, n_cpu, 1)
            cpu = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": "%d of %d light curves (%.1f s), astropy method='fast' (lightkurve default) restated "
                             "in oracle/ls.py, 1 process; equivalent bin*cadence/s = F*N*n/time" % (n_cpu, B, secs)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 spreading + FFT, f64 phase (nufft)" if family == "nufft" else
                     "f16x2-split in / f32 accumulate (tcgen05), f64 phase",
            "data": "synthetic",
            "config": {"workload": "%s: %s" % (args.workload, w["desc"]), "batch_per_gpu": B, "cadences": N,
                       "frequencies": F, "normalization": "amplitude", "algo": args.algo, "kernel_family": family,
                       "escalated_per_step": escalated,
                       "sharding": "by target, %d rank(s), %s" % (world, "no collective" if world == 1 else
                                   "%d asynchronous NCCL all-gathers of [%d x %d] power blocks per step, overlapped with the "
                                   "next piece's kernels" % (pieces, world * pb_rows, F)),
                       "l2": "inputs+outputs per step (%.0f MB) exceed the 126 MB L2" % ((Y.nbytes + B * F * 4) / 1e6)},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(Y.nbytes) * world,
                    "d2h_bytes_per_step": int(B * F * 4) * world, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "secondary": secondary,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"power": dumped})
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
