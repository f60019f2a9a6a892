#!/usr/bin/env python
"""bench.py -- retrospective forecasts/sec (network + GPR) on the north retrospective sweep (BASELINE.json
configs[1]: 1985-2020 x June/July/August/September inits x Pan-Arctic/Beaufort/Chukchi = 432 forecasts from
144 SIC (57x57) + 36 SST (26x90) network builds, synthetic NSIDC-shaped monthly fields 1979-2020).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]        # reference algorithm on the host cores

One step = one pass of the whole hot path (detrend -> correlation/tau -> domain growth/merge -> node series/links
-> batched GP) over one batch of MEMBERS perturbed-SIC ensemble members of that sweep (BASELINE.json configs[4] /
SURVEY.md 8(d): member m = base fields + 0.05 N(0,1), seed base + m; MEMBERS x 432 forecasts per step per GPU).  The
members share one device batch, so the latency-bound domain-growth chains of different networks overlap.  N>1: one
process per GPU (torchrun), rank r runs members r*MEMBERS .. (r+1)*MEMBERS-1 (no data-path collective; weak scaling),
value = all forecasts / max-over-ranks device time.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FMIN, FMAX, FIRST = 1985, 2020, 1979
TFULL = FMAX - FIRST + 1
MEMBERS = 8      # ensemble members per GPU per step (--members)
METRIC = "retrospective forecasts/sec (network+GPR)"
WORKLOAD = ("north retrospective sweep 1985-2020 x June/July/August/September inits x 3 regions: 432 forecasts, "
            "144 SIC 57x57 + 36 SST 26x90 network builds, T=7..42")


def make_workload(member=0):
    """Synthetic inputs of BASELINE.json configs[1].  Member 0 is the base realisation; member m > 0 is the perturbed-SIC
    ensemble member of SURVEY.md 8(d) / BASELINE.json configs[4]: base field + 0.05 * N(0,1) with seed base_seed + m
    (concentrations stay in [0, 1], saturated samples and land stay as they are; the SIE targets are shared)."""
    from seaiceextentforecasting_b200 import synthetic as syn
    from seaiceextentforecasting_b200.config import CONFIGS, NORTH_INITS
    sic = {}
    for i, name in enumerate(NORTH_INITS):
        sic[name], _ = syn.make_field(57, 57, TFULL, 1000 + i)
    sie = dict(zip(CONFIGS["north_june"].regions, syn.make_sie(sic["north_september"], TFULL, 1000)))
    sst, _ = syn.make_field(26, 90, TFULL, 2000, latlon=True, saturate=False, n_modes=60, noise=0.6,
                            blob=(2.0, 5.0))
    if member > 0:
        rng = np.random.default_rng(5000 + member)
        for name in NORTH_INITS:
            f = sic[name]
            inside = (f > 0.0) & (f < 1.0)              # NaN (land) compares False
            sic[name] = np.where(inside, np.clip(f + 0.05 * rng.standard_normal(f.shape), 0.0, 1.0), f)
        sst = sst + 0.05 * rng.standard_normal(sst.shape)      # NaN land stays NaN
    return dict(sic=sic, sie=sie, sst=sst, psar=syn.make_psar(57, 57), lat=syn.make_lat_grid(26, 90))


def make_workload_south(member=0):
    """Synthetic inputs of BASELINE.json configs[2]: south February retrospective sweep 1985-2020 on the 81x81 grid
    (`make_npstere_grid(-55,180,1e5)`, south/February1st.py:79), Pan-Antarctic / Ross / Weddell (108 forecasts from 36
    network builds).  Member m > 0: perturbed like make_workload."""
    from seaiceextentforecasting_b200 import synthetic as syn
    from seaiceextentforecasting_b200.config import CONFIGS
    f, _ = syn.make_field(81, 81, TFULL, 3000)
    sie = dict(zip(CONFIGS["south_february"].regions, syn.make_sie(f, TFULL, 3000)))
    if member > 0:
        rng = np.random.default_rng(7000 + member)
        inside = (f > 0.0) & (f < 1.0)
        f = np.where(inside, np.clip(f + 0.05 * rng.standard_normal(f.shape), 0.0, 1.0), f)
    return dict(sic={"south_february": f}, sie=sie, sst=None, psar=syn.make_psar(81, 81), lat=None)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, enabled=True):
        # gpu_index: an index or a comma-separated list.  One poller (rank 0, all local GPUs) per job: every nvidia-smi
        # query takes driver locks, so one poller per rank perturbs the launches of all ranks
        self.idx, self.proc, self.lines, self.enabled = gpu_index, None, [], enabled

    def start(self):
        if not self.enabled:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.enabled:
            return None
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                clk, cmax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            if t0 - 0.05 <= t <= t1 + 0.05:
                sm.append(clk)
                mx.append(cmax)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                     parts[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:   # region shorter than the sampling period: fall back to all samples
            for t, line in self.lines:
                parts = [p.strip() for p in line.split(",")]
                try:
                    sm.append(float(parts[1]))
                    mx.append(float(parts[2]))
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ shared
def bench_config(members, world):
    """The `config` object of the JSON line: identical for both arms (it names the workload, nothing run-dependent)."""
    return {"workload": WORKLOAD, "grid": "57x57 SIC + 26x90 SST", "years": [FMIN, FMAX],
            "members_per_gpu": members, "forecasts_per_step_per_gpu": 432 * members,
            "members": "member 0 = base realisation, member m = base + 0.05*N(0,1), seed base+m (perturbed-SIC ensemble, "
                       "SURVEY.md 8(d)); rank r of N runs members r*M..(r+1)*M-1",
            "parallelism": "task-parallel: independent members / (init, year) tasks, no data-path collective",
            "l2": "working set per step = members x 7.2 GB of correlation matrices >> 126 MB L2: no flush needed"}


# ------------------------------------------------------------------------------------------------ reference arm
def _ref_task(args):
    """One (config, year) task of the sweep with the oracle port (reference algorithm, numpy/scipy).
    Returns (forecasts produced, forecasts on which the reference raises, seconds)."""
    import warnings
    warnings.simplefilter("ignore")
    from oracle import sweep as osweep
    from seaiceextentforecasting_b200.config import CONFIGS
    name, year, member = args
    w = _ref_task.cache.get(member)
    if w is None:
        w = make_workload(member)
        cfgs = [CONFIGS[n] for n in w["sic"]]
        w["tables"] = {reg: osweep.sie_tables(w["sie"][reg], FMIN, FMAX) for reg in cfgs[0].regions}
        _ref_task.cache[member] = w
    cfg = CONFIGS[name]
    sie_dt = {r: w["tables"][r][0] for r in cfg.regions}
    sie_tr = {r: w["tables"][r][1] for r in cfg.regions}
    t0 = time.perf_counter()
    res, _ = osweep.run_job(cfg, year, w["sic"][name], w["psar"], sie_dt, sie_tr, FMIN, w["sst"], w["lat"],
                            record_failures=True)
    failed = sum(1 for r in res if r["failed"] is not None)
    return len(res) - failed, failed, time.perf_counter() - t0


_ref_task.cache = {}


def sample_tasks(count, members=1):
    """A bounded, T-representative sample of the members x 144 (init, year) tasks: years spread evenly over 1985-2020,
    inits and members cycled."""
    from seaiceextentforecasting_b200.config import NORTH_INITS
    years = np.linspace(FMIN, FMAX, count).round().astype(int)
    return [(NORTH_INITS[i % 4], int(y), (i // 4) % max(1, members)) for i, y in enumerate(years)]


def cpu_baseline_single(n_tasks=4):
    tasks = sample_tasks(n_tasks)
    t0 = time.perf_counter()
    res = [_ref_task(t) for t in tasks]
    dt = time.perf_counter() - t0
    n = sum(r[0] + r[1] for r in res)       # a forecast on which the reference raises still cost its network build
    return {"value": n / dt, "unit": "forecasts/s", "cores": 1, "kind": "port",
            "sample": f"{len(tasks)} of 144 (init,year) tasks of member 0 = {n} of 432 forecasts "
                      f"({sum(r[1] for r in res)} of them raise in the reference), years {[t[1] for t in tasks]}, "
                      f"{dt:.1f} s, oracle port (numpy/scipy, bitmap lookups instead of the reference's list scans: "
                      "~9x faster than the literal reference on area_level)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 48))
    n_tasks = max(procs, 8)
    tasks = sample_tasks(n_tasks, args.members)
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        for _ in range(args.warmup):
            pool.map(_ref_task, tasks[:procs])
        t0 = time.perf_counter()
        n = nfail = 0
        for _ in range(args.steps):
            res = pool.map(_ref_task, tasks)
            n += sum(r[0] + r[1] for r in res)
            nfail += sum(r[1] for r in res)
        dt = time.perf_counter() - t0
    value = n / dt
    line = {"metric": METRIC, "value": value, "unit": "forecasts/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": bench_config(args.members, args.gpus),
            "cpu_baseline": {"value": value, "unit": "forecasts/s", "cores": procs, "kind": "port",
                             "sample": f"each step = {n_tasks} (init,year) tasks (years spread evenly over 1985-2020, inits and "
                                       f"members cycled) of the {144 * args.members} tasks of one {args.members}-member step = "
                                       f"{3 * n_tasks} of {432 * args.members} forecasts, over a {procs}-process pool "
                                       f"({cores} host cores); throughput per task is what is compared (tasks are "
                                       f"independent); {nfail} sampled forecasts raise in the reference and are counted (their "
                                       "network builds were done); oracle port of the reference algorithm (the reference is "
                                       "Python and cannot travel to the GPU box; the port's area_level is ~9x faster)"},
            "e2e": {"value": value, "unit": "forecasts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------ our arm
def fp64_gemm_peak(torch):
    """cuBLAS DGEMM burst peak (TFLOP/s): the denominator for the DMMA correlation kernel and the GP stage, measured here
    because MEASURED_PEAKS.json only carries HBM and bf16 figures."""
    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    best = 0.0
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del a, b
    return best


def corr_25km(torch, dist, fp64_peak, world, rank):
    """BASELINE.json's second figure: all-pairs correlation + tau on the 25 km 448x304 grid (configs[3]), R not stored,
    tile rows sharded over the ranks (`sie_corr_tau(shard_rank, shard_count)`), the NCCL all-reduce of (sum, count)
    INSIDE the timed region; aggregate TFLOP/s of the upper-triangle algorithmic work N(N+1)T against the FP64 tensor
    peak measured above (x world).  Device-timed, MAX over ranks."""
    from seaiceextentforecasting_b200 import synthetic as syn
    from seaiceextentforecasting_b200.engine import NetworkBatch, h2d, r_crit_ttest
    from seaiceextentforecasting_b200.parallel import tau_from_shards
    X, Y, T = 448, 304, 42
    data, _ = syn.make_field(X, Y, T, 7, n_modes=200)
    n_upper = int((~np.isnan(data).any(axis=2)).sum())
    eng = NetworkBatch(X, Y, T, 1, latlon=False, n_upper=n_upper, keep_R=False, max_areas=8)
    fields = h2d(data.reshape(1, X * Y, T))
    jf = torch.zeros(1, dtype=torch.int32, device="cuda")
    jT = torch.full((1,), T, dtype=torch.int32, device="cuda")
    rc = h2d(np.array([r_crit_ttest(T, 0.01)]))
    eng.detrend_zscore(fields, jf, jT, True)

    def step():
        eng.corr_tau(rc, store_R=False, shard_rank=rank, shard_count=world)
        return tau_from_shards(eng.tau_sum, eng.tau_cnt)

    for _ in range(3):
        tau = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        tau = step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    N = int(eng.n_nodes.item())
    tf = N * (N + 1.0) * T / (ms * 1e-3) / 1e12
    out = {"workload": f"448x304 grid, {N} nodes, T={T}, R not stored, 128-row tile rows round-robin over {world} rank(s)",
           "ms": ms, "tflops_fp64_aggregate": tf, "peak_tflops_fp64_per_gpu": fp64_peak,
           "frac": tf / (fp64_peak * world) if fp64_peak else None, "tau": float(tau.item()),
           "collective": "NCCL all-reduce of (sum, count) inside the timed region" if world > 1 else "none (1 GPU)",
           "flop_model": "N(N+1)T per network (upper triangle)"}
    del eng
    torch.cuda.empty_cache()
    return out


def gp_flops(raw, n_rows):
    """Algorithmic FP64 flop of the GP stage from the per-problem records (SURVEY.md 8(d)): expm = the GEMMs of the
    Pade order scipy's algorithm picks (3 for A^2/A^4/A^6 + 1 / 2 / 5 more for m <= 5 / m <= 9 / m = 13) + s squarings
    at 2 Np^3 each + the LU solve 8 Np^3 / 3; X E and (X E) X^T; two Cholesky factorisations of n x n."""
    ok = raw["info"] == 0
    Np = raw["n_pred"][ok].astype(np.float64)
    m = raw["expm_m"][ok]
    s = raw["expm_s"][ok].astype(np.float64)
    n = n_rows[ok].astype(np.float64)
    gemms = np.where(m <= 5, 4.0, np.where(m <= 9, 5.0, 8.0)) + s
    return float((2.0 * Np ** 3 * gemms + 8.0 * Np ** 3 / 3.0 + 2.0 * n * Np ** 2 + 2.0 * n * n * Np
                  + 2.0 * (2.0 * n ** 3 / 3.0)).sum())


def stage_times(marks_all, steps):
    stage_ms = {}
    for marks in marks_all:
        last = {}
        for name, ev in marks:          # consecutive marks of one chain (sic.* / sst.* / gp.*) bracket a stage
            tag = name.split(".")[0]
            if tag in last and not name.endswith(".start"):
                stage_ms[name] = stage_ms.get(name, 0.0) + last[tag].elapsed_time(ev)
            last[tag] = ev
    return {k: v / steps for k, v in stage_ms.items()}


def roofline_table(sw, stage_ms, hbm_peak, hbm_src, fp64_peak):
    """One entry per stage of the step (timed in a separate pass with one batch per grid so that events bracket every
    stage): algorithmic bytes / flop per launch (DESIGN.md section 4) over the measured stage time."""
    roof = {}
    fp64_src = ("cuBLAS DGEMM 6144^3 burst measured in this run (MEASURED_PEAKS.json has no FP64 figure; DMMA and DFMA "
                "peaks are nominally equal on B200)")

    def hbm(name, nbytes, note, **extra):
        ms = stage_ms.get(name)
        if ms:
            ach = nbytes / (ms * 1e-3) / 1e9
            roof[name] = dict({"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                               "traffic": None, "ms": ms, "peak_source": hbm_src, "model": note}, **extra)

    for tag, eng, T in (("sic", sw.sic, sw.plan.job_T), ("sst", sw.sst, sw.plan.sst_T)):
        if eng is None:
            continue
        N = eng.n_nodes.cpu().numpy().astype(np.float64)
        T = T.astype(np.float64)
        nA = eng.n_areas.cpu().numpy().astype(np.int64)
        starts = eng.area_start.cpu().numpy()
        members = np.array([starts[b, nA[b]] for b in range(len(nA))], dtype=np.float64)
        hbm(tag + ".detrend_zscore", float((16.0 * eng.C * T).sum() + (8.0 * N * eng.Tp).sum()),
            "16 C T bytes per window (read raw, write residuals) + 8 N Tp (z rows)")
        ms = stage_ms.get(tag + ".corr_tau")
        if ms and fp64_peak:        # upper triangle only: N(N+1)T flop against 4 N^2 stored bytes -> 10.5 flop/B at T = 42,
            fl = float((N * (N + 1.0) * T).sum())             # above the FP64 ridge (~5.5 flop/B): tensor-bound
            ach = fl / (ms * 1e-3) / 1e12
            roof[tag + ".corr_tau"] = {"bound": "tensor", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
                                       "frac": ach / fp64_peak, "traffic": None, "ms": ms, "peak_source": fp64_src,
                                       "store_GBps": float((4.0 * N * N).sum()) / (ms * 1e-3) / 1e9,
                                       # the launch mixes windows on both sides of the ridge (T ~ 22): per network the
                                       # binding roof is max(flop / tensor peak, stored bytes / HBM peak)
                                       "two_roof_ideal_ms": float(np.maximum(N * (N + 1.0) * T / (fp64_peak * 1e12),
                                                                             4.0 * N * N / (hbm_peak * 1e9)).sum() * 1e3),
                                       "frac_two_roofs": float(np.maximum(N * (N + 1.0) * T / (fp64_peak * 1e12),
                                                                          4.0 * N * N / (hbm_peak * 1e9)).sum() * 1e3) / ms,
                                       "model": "N(N+1)T flop per network (upper triangle) on the FP64 tensor pipe (DMMA); "
                                                "4 N^2 bytes stored (upper triangle of R) + 8 N Tp read"}
        hbm(tag + ".area_level", 8.0 * float(eng.area_work.cpu().numpy()[:, 0].sum()),
            "8 B x correlations the reference's growth/merge consumes (counted on the device); the kernel is a chain "
            "of dependent decisions, latency-bound by design: the fraction is reported, not claimed as a target")
        hbm(tag + ".intra_links", float((8.0 * members * T + 4.0 * members + 8.0 * eng.C).sum()),
            "8 (member cells) T + 4 (member cells) + 8 C bytes per network")
    ms = stage_ms.get("gp")
    if ms and fp64_peak:
        n_rows = sw.plan.prob["n"]
        fl = gp_flops(sw.raw, n_rows)
        ach = fl / (ms * 1e-3) / 1e12
        roof["gp"] = {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                      "traffic": None, "ms": ms, "peak_source": fp64_src, "problems_per_s": sw.P / (ms * 1e-3),
                      "model": "expm GEMMs of the Pade order + squarings (2 Np^3 each) + LU solve 8 Np^3/3 + X E + "
                               "(X E) X^T + 2 Cholesky (2 n^3/3 each), summed over the problems' records"}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        for name in roof:
            if name in traffic:
                roof[name]["traffic"] = traffic[name]
    except (OSError, ValueError):
        pass
    return roof


def extra_sweeps(torch, members_done):
    """Rank 0, N=1 only: the other single-GPU configurations of BASELINE.json as extra fields of the line --
    configs[2] south February 81x81 sweep (device-timed steps) and a configs[4] slice: every GP problem of one member
    of the north sweep on the reference's 20 x 20 (l, sigma) grid (`sie_gp_hyper_grid`: problems/s)."""
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    out = {}
    SM = 4                                   # ensemble members batched per step, like the north sweep (one member alone
    ws = [make_workload_south(m) for m in range(SM)]   # = 36 growth jobs + 108 GP problems: a fraction of one wave of CTAs)
    w = ws[0]
    sw = RetrospectiveSweep(["south_february"], [x["sic"] for x in ws], w["sie"], FMIN, FMAX, w["psar"], max_pred=512)
    sw.upload()
    for _ in range(2):
        sw.compute()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        sw.compute()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    raw = sw.download()
    out["south_february"] = {"workload": f"BASELINE configs[2]: south February 1985-2020, 36 SIC 81x81 network builds + 108 forecasts "
                                         f"per member, {SM} perturbed members per step",
                             "members": SM, "ms_per_step": ms, "forecasts_per_s": sw.P / (ms * 1e-3),
                             "failures_like_reference": int((raw["info"] == -1).sum()),
                             "max_predictors": int(raw["n_pred"].max())}
    del sw
    torch.cuda.empty_cache()
    return out


def hyper_grid_slice(torch, sw, fp64_peak):
    """configs[4] slice on the north sweep that was just run: all GP problems x 20 l x 20 sigma."""
    torch.cuda.synchronize()
    sw.hyper_grid()                       # warm-up (allocates)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rec = sw.hyper_grid()
    dt = time.perf_counter() - t0
    ok = rec["info"] == 0
    return {"workload": f"BASELINE configs[4] slice: {sw.P} GP problems x 20 l x 20 sigma (north/June1st.py:210-211 grids)",
            "evaluations": int(rec.size), "seconds": dt, "evaluations_per_s": rec.size / dt,
            "finite": int(ok.sum()), "timing": "wall clock around RetrospectiveSweep.hyper_grid incl. the D2H of "
                                               f"{rec.nbytes} result bytes"}


RECORD_FIELDS = ("fmean", "fvar", "sigma_f", "nlml", "n_pred", "info")
OUT_KEYS = ("_fmean", "_fvar", "_fmean_rt", "_raw_fmean", "_raw_fvar", "_raw_fmean_rt")


def dump_outputs(dirname, sw, out, prefix=""):
    """What one step returns to a caller of RetrospectiveSweep.run / run_many, as float64 .npy files in `dirname`:
    `<config>.<region><key>.npy` [members, years] (the assembled forecast dict of every member) and
    `records.<field>.npy` [problems] (the GP records `sw.raw`, in the plan's problem order).
    A problem with no forecast (record info != 0: info = -1 where the reference's forecast() raises) comes back as NaN;
    its entries are written as 0 and marked by `<config>.<region>_no_forecast.npy` (1.0) and `records.info.npy`, so
    that two runs compare element by element.  Any other non-finite value is written as it is."""
    os.makedirs(dirname, exist_ok=True)
    failed = sw.raw["info"] != 0
    flag = np.zeros(len(sw.raw), dtype=sw.raw.dtype)
    flag["fmean"] = failed
    flags = sw.plan.assemble(flag)           # same layout as `out`: 1.0 in <region>_raw_fmean where a problem failed
    members, mflags = (out, flags) if isinstance(out, list) else ([out], [flags])
    arrays = {}
    for cfg in sw.cfgs:
        for reg in cfg.regions:
            no = np.stack([f[cfg.name][reg + "_raw_fmean"] for f in mflags]) != 0.0
            arrays[f"{cfg.name}.{reg}_no_forecast"] = no.astype(np.float64)
            for key in OUT_KEYS:
                a = np.stack([np.asarray(m[cfg.name][reg + key], dtype=np.float64) for m in members])
                arrays[f"{cfg.name}.{reg}{key}"] = np.where(no, 0.0, a)
    for f in RECORD_FIELDS:
        a = sw.raw[f].astype(np.float64)
        arrays["records." + f] = a if f in ("n_pred", "info") else np.where(failed, 0.0, a)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, prefix + name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as entry
    from seaiceextentforecasting_b200 import build as b
    if rank == 0 and b.needs_build():
        entry.build()
    if world > 1:
        dist.barrier()
    from seaiceextentforecasting_b200 import parallel
    from seaiceextentforecasting_b200.config import NORTH_INITS
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep

    M = args.members
    ws = [make_workload(member=rank * M + m) for m in range(M)]
    sw = RetrospectiveSweep(NORTH_INITS, [w["sic"] for w in ws], ws[0]["sie"], FMIN, FMAX, ws[0]["psar"],
                            [w["sst"] for w in ws], ws[0]["lat"])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident steps (inputs already in HBM)
    sw.upload()
    for _ in range(args.warmup):
        sw.compute()
    sync_all()
    sampler = ClockSampler(",".join(str(i) for i in range(world)) if world > 1 else local, enabled=(rank == 0))
    sampler.start()
    time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        sw.compute()
    e1.record()
    sync_all()
    t_wall1 = time.perf_counter()
    dev_ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t_wall0, t_wall1)
    # per-stage device times (for the roofline block): same work, every stage alone on one stream so that events
    # bracket exactly one stage with nothing else on the GPU; not part of the headline timing
    # (minimum over the passes, each pass synchronised: a host-side stall between two launches of a pass - e.g. the
    # clock poller's last nvidia-smi call holding the driver - would otherwise be booked to whatever stage it hit)
    stage_ms = {}
    for _ in range(min(args.steps, 5)):
        marks = []
        sw.compute(marks, waves=0)
        sync_all()
        for k, v in stage_times([marks], 1).items():
            stage_ms[k] = min(stage_ms.get(k, v), v)
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    nf = torch.tensor([float(sw.n_forecasts)], dtype=torch.float64, device="cuda")
    per_rank_ms = [dev_ms / args.steps]
    if world > 1:
        allms = [torch.zeros_like(tmax) for _ in range(world)]
        dist.all_gather(allms, tmax)
        per_rank_ms = [float(t.item()) / args.steps for t in allms]     # ranks run different members (different fields)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(nf, op=dist.ReduceOp.SUM)
    ms_per_step = float(tmax.item()) / args.steps
    total_forecasts = float(nf.item())
    value = total_forecasts / (ms_per_step * 1e-3)

    # ---------------- end to end through the public API: pinned host -> device, compute, device -> host
    for out in sw.run_many(max(2, min(args.warmup, 3))):     # warm-up through the same loop: its second input buffer set,
        pass                                                 # copy stream and pinned result buffers are created once
    sync_all()
    t0 = time.perf_counter()
    for out in sw.run_many(args.steps):      # every step: H2D of its inputs, the hot path, D2H of its results; the host
        pass                                 # assembles step i while step i+1 is on the device (forecast.run_many)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = total_forecasts / (float(e2e_t.item()) / args.steps)
    like_ref = int((sw.raw["info"] == -1).sum())
    other_bad = int(((sw.raw["info"] != 0) & (sw.raw["info"] != -1)).sum())
    sw.check_status(sw.raw)
    if args.dump_outputs:                    # `out` / sw.raw: the last timed step's results
        dump_outputs(args.dump_outputs, sw, out, prefix=f"rank{rank}." if world > 1 else "")

    # ---------------- strong scaling of the same step: this rank's members split over ALL ranks by (member, init, year)
    #                  task, records all-gathered as tensors, the assembled result compared with the unsharded one
    strong = None
    if world > 1 and not args.no_strong:
        ws0 = [make_workload(member=m) for m in range(M)]            # every rank shards the SAME members 0..M-1
        shard = RetrospectiveSweep(NORTH_INITS, [w["sic"] for w in ws0], ws0[0]["sie"], FMIN, FMAX, ws0[0]["psar"],
                                   [w["sst"] for w in ws0], ws0[0]["lat"], rank=rank, world=world)
        shard.upload()
        for _ in range(3):
            shard.compute()
        sync_all()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(3, args.steps // 2)
        s0.record()
        for _ in range(reps):
            shard.compute()
            recs = parallel.gather_records(shard.plan, None, device="cuda", raw_dev=shard.gp.out)   # NCCL all-gather
        s1.record()
        sync_all()
        sm = torch.tensor([s0.elapsed_time(s1) / reps], dtype=torch.float64, device="cuda")
        dist.all_reduce(sm, op=dist.ReduceOp.MAX)
        full = shard.plan.assemble(*recs)
        equal = None
        if rank == 0:                                               # rank 0 ran exactly these members unsharded above
            ref = sw.plan.assemble(sw.raw)
            equal = all(np.array_equal(np.asarray(a[c][k]), np.asarray(r[c][k]), equal_nan=True)
                        for a, r in zip(full, ref) for c in r for k in r[c]) if M > 1 else \
                all(np.array_equal(np.asarray(full[c][k]), np.asarray(ref[c][k]), equal_nan=True) for c in ref for k in ref[c])
        strong = {"workload": f"the same {M}-member step ({432 * M} forecasts) split over {world} GPUs by (member, init, year) "
                              "task (SweepPlan(rank, world)); GP records all-gathered as tensors over NCCL inside the timed "
                              "region", "ms_per_step": float(sm.item()),
                  "value": 432.0 * M / (float(sm.item()) * 1e-3), "unit": "forecasts/s", "scaling": "strong",
                  "assembled_equals_unsharded_bit_for_bit": equal}
        del shard

    fp64_peak = fp64_gemm_peak(torch)
    roof = roofline_table(sw, stage_ms, hbm_peak, hbm_src, fp64_peak)
    top = max(roof, key=lambda k: roof[k]["ms"]) if roof else None
    main_roof = dict(roof[top], kernel=top) if top else None
    corr25 = corr_25km(torch, dist, fp64_peak, world, rank) if args.corr25 else None
    extras = {}
    if world == 1 and not args.no_extras:
        extras["hyper_grid"] = hyper_grid_slice(torch, sw, fp64_peak)
    areas_mean = float(sw.sic.n_areas.cpu().numpy().mean())
    n_launch = sw.kernel_launches()
    h2d_b, d2h_b = sw.h2d_bytes(), sw.d2h_bytes()
    waves_desc = (f"{len(sw.waves)} waves on separate streams, window-length edges T={list(sw.wave_T)}: "
                  + "; ".join(f"{jr[1]-jr[0]} SIC networks + {pr[1]-pr[0]} GP problems" for (jr, sr, pr) in sw.waves)
                  + ("; each wave's GP = a launch for the SIC-only problems + one for the SST-reading ones" if sw.gp_sst else "")
                  ) if sw.multi_wave else "single wave"
    if world == 1 and not args.no_extras:
        del sw
        torch.cuda.empty_cache()
        extras.update(extra_sweeps(torch, M))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "forecasts/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(M, world),
            "e2e": {"value": e2e_value, "unit": "forecasts/s", "h2d_bytes_per_step": h2d_b,
                    "d2h_bytes_per_step": d2h_b, "ms_per_step": 1e3 * float(e2e_t.item()) / args.steps},
            "gpu_launches": args.steps * n_launch,
            "clocks": clocks, "per_rank_ms_per_step": per_rank_ms,
            "roofline": main_roof,
            "roofline_all": roof,
            "schedule": waves_desc + "; domain growth = persistent grid popping jobs longest-window-first; stage_ms / "
                        "roofline timed in a separate pass with every stage alone on the GPU; e2e loop = RetrospectiveSweep.run_many (step i+1's H2D on a copy stream into a second input buffer while step i computes; step i's "
                        "D2H + host assemble overlap step i+1)",
            "corr_25km": corr25,
            "strong_scaling": strong,
            "stage_ms": stage_ms,
            "gp_failures": {"like_reference": like_ref, "other": other_bad,
                            "note": "info = -1: fewer than two predictors pass the script's selection rule; the reference's "
                                    "forecast() raises there (tests/golden/bench_north_m0.npz records the same 6 of 432)"},
            "checks": {"forecasts_per_rank": 432 * M, "areas_mean": areas_mean},
        }
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_single()
        else:
            line["cpu_baseline"] = None
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--members", type=int, default=MEMBERS, help="ensemble members per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the south-sweep / hyper-grid extra fields (N=1)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (N>1)")
    ap.add_argument("--no-corr25", dest="corr25", action="store_false",
                    help="skip the 25 km all-pairs correlation probe (second half of BASELINE.json's metric)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the forecasts and GP records of the last timed step to DIR/<name>.npy (float64; "
                         "with N > 1 every rank writes its own members as rank<r>.<name>.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this repo's CUDA path computed: not with --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # stdout carries ONE JSON line: libraries that write to file descriptor 1 (NCCL prints its version banner there when
    # NCCL_DEBUG is set) are pointed at stderr, and the line goes to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
