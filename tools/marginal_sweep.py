"""Marginalised retrospective sweep on the bench's 8-member north step (bench.make_workload): every forecast the average
of its problem's forecasts over the reference's 20 x 20 (l, sigma_n~) grid, weighted by marginal likelihood
(RetrospectiveSweep(hyper_grid=(LS, SS), hyper_mode="marginal")), next to the plain and the tuned (grid argmin) step.

    python tools/marginal_sweep.py [--steps K] [--reps R] [--kernel-reps N] [--out FILE]

In one process: the plain, tuned and marginal steps device-resident (inputs in HBM, CUDA events after warm-up, the
three alternated R times, K steps each); sie_gp_grid_marginal alone over the step's full P x 400 grid records (N
launches back to back, and N launches each after a 256 MB write that evicts L2), against the bytes it must read; the
grid posterior's concentration (ESS, largest weight); skill (SweepPlan.skill) of the three modes and the coverage of
their 5-95 % intervals (Gaussian for plain / tuned, the mixture's quantiles for marginal; synthetic data, a report
only); the card's name and power limit (read-only query).  Prints one JSON line and writes it to --out."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from seaiceextentforecasting_b200.config import LS, NORTH_INITS, SS  # noqa: E402
from seaiceextentforecasting_b200.forecast import (FIRST_YEAR, GP_MARGINAL_DTYPE, GP_RESULT_DTYPE,  # noqa: E402
                                                   RetrospectiveSweep, grid_marginal)

M = 8                                  # members per step (bench.MEMBERS)
LEVELS = (0.05, 0.5, 0.95)
Z95 = 1.6448536269514722               # norm.ppf(0.95)
HBM_GBS = 6541.8                       # measured B200 HBM read bandwidth the kernel's byte count is compared with
SECTOR = 32


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def sweep(ws, mode):
    kw = {} if mode == "plain" else dict(hyper_grid=(LS, SS), hyper_mode="argmin" if mode == "tuned" else "marginal")
    if mode == "marginal":
        kw["quantiles"] = LEVELS
    return RetrospectiveSweep(NORTH_INITS, [w["sic"] for w in ws], ws[0]["sie"], bench.FMIN, bench.FMAX, ws[0]["psar"],
                              [w["sst"] for w in ws], ws[0]["lat"], **kw)


def device_ms(sw, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sw.compute()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def sectors_read(n_records):
    """32-B sectors sie_gp_grid_marginal must read from n_records contiguous records (base 256-B aligned): every sector
    holding a byte of fmean, fvar, nlml or info of some record (computed from the record layout)."""
    isz = GP_RESULT_DTYPE.itemsize
    spans = [(GP_RESULT_DTYPE.fields[f][1], GP_RESULT_DTYPE.fields[f][0].itemsize) for f in ("fmean", "fvar", "nlml",
                                                                                             "info")]
    period = isz * SECTOR // math.gcd(isz, SECTOR)          # the sector pattern repeats every lcm(80, 32) bytes
    per = period // isz
    sec = set()
    for r in range(per):
        for off, size in spans:
            b0 = r * isz + off
            sec.update(range(b0 // SECTOR, (b0 + size - 1) // SECTOR + 1))
    full, rest = divmod(n_records, per)
    tail = set()
    for r in range(rest):
        for off, size in spans:
            b0 = r * isz + off
            tail.update(range(b0 // SECTOR, (b0 + size - 1) // SECTOR + 1))
    return full * len(sec) + len(tail), len(sec) / per


def kernel_alone(sw, reps):
    """sie_gp_grid_marginal over the sweep's device grid records (the last step's), into scratch outputs."""
    g, P = sw.tune, sw.P
    n_grid = len(g.ells) * len(g.sigs)
    out = torch.empty(P * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    stats = torch.empty(P * GP_MARGINAL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    quant = torch.empty(P * len(LEVELS), dtype=torch.float64, device="cuda")
    q = torch.tensor(LEVELS, dtype=torch.float64, device="cuda")
    for _ in range(3):
        grid_marginal(g.out, P, n_grid, q, out, stats, quant)
    torch.cuda.synchronize()
    # back to back: the 110 MB of records may stay in the 126 MB L2 between launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        grid_marginal(g.out, P, n_grid, q, out, stats, quant)
    e1.record()
    torch.cuda.synchronize()
    warm = e0.elapsed_time(e1) / reps
    # each launch after a 256 MB write: the records come from HBM
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        flush.fill_(1)
        a.record()
        grid_marginal(g.out, P, n_grid, q, out, stats, quant)
        b.record()
    torch.cuda.synchronize()
    cold = sorted(a.elapsed_time(b) for a, b in evs)
    same = torch.equal(out, sw.gp.out[:out.numel()]) and torch.equal(stats, sw._mstats) and \
        torch.equal(quant, sw._quant[:quant.numel()])
    n_sec, per_rec = sectors_read(P * n_grid)
    need = n_sec * SECTOR
    cold_med = statistics.median(cold)
    return {"problems": P, "grid_points": n_grid, "records_bytes": P * n_grid * GP_RESULT_DTYPE.itemsize,
            "sectors_per_record": per_rec, "bytes_to_read": need,
            "floor_ms_at_hbm": need / (HBM_GBS * 1e9) * 1e3, "hbm_gbs_assumed": HBM_GBS,
            "ms_back_to_back": warm, "ms_after_l2_flush_median": cold_med, "ms_after_l2_flush_min": cold[0],
            "achieved_gbs_after_l2_flush": need / (cold_med * 1e-3) / 1e9,
            "timing": f"CUDA events; back to back: {reps} launches in one window (records possibly L2-resident); "
                      f"after flush: {reps} launches each timed alone after a 256 MB device write",
            "outputs_equal_the_step": bool(same)}


def skill_summary(plans, outs):
    """Mean over members of SweepPlan.skill (rt, dt) per config and region."""
    res = {}
    for plan, o in zip(plans, outs):
        for m, gpr in enumerate(o):
            for cfg, (rt, dt) in plan.skill(gpr).items():
                r = res.setdefault(cfg, {"rt": [], "dt": []})
                r["rt"].append(rt)
                r["dt"].append(dt)
    return {c: {k: np.nanmean(np.asarray(v, dtype=float), axis=0).round(3).tolist() for k, v in d.items()}
            for c, d in res.items()}


def coverage(sw, outs, mode):
    """Share of (member, config, region, year) forecasts whose detrended observation lies in the 5-95 % interval."""
    plan = sw.plan
    inside = total = 0
    for gpr in outs:
        for cfg in plan.cfgs:
            g = gpr[cfg.name]
            for reg in cfg.regions:
                obs = np.array([plan.sie_dt[reg][t - (plan.fmin - 1), t - FIRST_YEAR] for t in plan.years])
                if mode == "marginal":
                    lo, hi = g[reg + "_quantiles"][:, 0], g[reg + "_quantiles"][:, 2]
                else:
                    sd = np.sqrt(g[reg + "_raw_fvar"])
                    lo, hi = g[reg + "_raw_fmean"] - Z95 * sd, g[reg + "_raw_fmean"] + Z95 * sd
                ok = np.isfinite(lo) & np.isfinite(hi)
                inside += int(((obs >= lo) & (obs <= hi) & ok).sum())
                total += int(ok.sum())
    return {"inside": inside, "forecasts": total, "share": inside / max(total, 1)}


def clean(x):
    if isinstance(x, float) and not math.isfinite(x):
        return None
    if isinstance(x, dict):
        return {k: clean(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [clean(v) for v in x]
    return x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-reps", type=int, default=200)
    ap.add_argument("--out")
    args = ap.parse_args()
    import __graft_entry__ as entry
    entry.build()
    ws = [bench.make_workload(m) for m in range(M)]
    result = {"tool": "tools/marginal_sweep.py", "card": card(),
              "workload": f"bench.make_workload members 0..{M - 1}: {M} x 432 north forecasts per step, grid "
                          f"{len(LS)} l x {len(SS)} sigma_n~ (north/June1st.py:210-211), quantile levels {LEVELS}"}
    sws = {mode: sweep(ws, mode) for mode in ("plain", "tuned", "marginal")}
    for sw in sws.values():
        sw.upload()
        for _ in range(args.warmup):
            sw.compute()
    torch.cuda.synchronize()
    ms = {k: [] for k in sws}
    names = list(sws)
    for r in range(args.reps):
        for name in (names if r % 2 == 0 else names[::-1]):
            ms[name].append(device_ms(sws[name], args.steps))
    med = {k: statistics.median(v) for k, v in ms.items()}
    P = sws["plain"].P
    result["device_resident"] = {
        "timing": f"CUDA events around {args.steps} back-to-back compute() calls, {args.reps} repetitions alternating "
                  "plain / tuned / marginal (order reversed every other repetition), after warm-up; median reported",
        "ms_per_step": ms, "median_ms_per_step": med,
        "forecasts_per_s": {k: P / (v * 1e-3) for k, v in med.items()},
        "marginal_minus_tuned_ms": med["marginal"] - med["tuned"],
        "kernel_launches": {k: sw.kernel_launches() for k, sw in sws.items()},
        "d2h_bytes": {k: sw.d2h_bytes() for k, sw in sws.items()}}
    outs = {}
    for name, sw in sws.items():
        sw.upload()
        sw.compute()
        outs[name] = sw.plan.assemble(sw.download(), selection=sw.selection, marginal=sw.marginal)
    result["grid_marginal_kernel"] = kernel_alone(sws["marginal"], args.kernel_reps)
    mg = sws["marginal"].marginal
    ok = mg["n_admissible"] > 0
    ess = mg["ess"][ok]
    result["posterior"] = {"problems": int(P), "with_admissible_points": int(ok.sum()),
                           "n_admissible_median": float(np.median(mg["n_admissible"][ok])),
                           "ess_quartiles": np.percentile(ess, [0, 25, 50, 75, 100]).tolist(),
                           "w_max_quartiles": np.percentile(mg["w_max"][ok], [0, 25, 50, 75, 100]).tolist(),
                           "share_ess_below_2": float((ess < 2).mean()),
                           "argmax_equals_tuned_best": float((mg["argmax"] == sws["tuned"].best_index()).mean())}
    result["skill_mean_over_members"] = {k: skill_summary([sws[k].plan], [outs[k]]) for k in sws}
    result["coverage_5_95"] = {k: coverage(sws[k], outs[k], k) for k in sws}
    result["note"] = "synthetic inputs: skill and coverage are a report, not evidence about real forecasts"
    line = json.dumps(clean(result))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
