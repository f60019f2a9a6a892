"""Ensemble forecasts of the bench's north marginalised sweep (forecast.EnsembleForecast): every member's predictive
distribution of a (config, region, year) pooled into one on the device (sie_gp_ensemble).

    python tools/ensemble_sweep.py [--batches K] [--kernel-reps N] [--out FILE]

In one process:
  * sie_gp_ensemble alone at E = 432 problems for (M, n_grid) in (8, 1), (1024, 1), (8, 400), (64, 400), (1024, 400):
    the records are a real 8-member marginal step's (bench.make_workload members 0..7; its forecast records for
    n_grid = 1, its 20 x 20 grid records for n_grid = 400) tiled across the M slots (slot s = member s % 8), so the
    weights are as concentrated as in the product.  CUDA events over up to N launches after warm-up.  Reported next to
    the time: the component-CDF evaluations the bisection did (counted on the host by replaying each level's halvings
    from the device's result) per second, and the bytes the kernel moves (the records once, the staged components
    written once and read once per CDF pass) against HBM bandwidth.
  * streaming: K batches of 8 members (bench.make_workload(8 b + i)) through one marginal sweep: load_inputs ->
    upload -> compute, timed with and without EnsembleForecast.add (alternated, CUDA events around the enqueue and a
    synchronise), then result(); the ensemble forecast's skill (SweepPlan.skill) next to the mean member skill, and
    the coverage of the 5-95 % intervals of both (synthetic data: a report only).
  * the card's name and power limit (read-only query).
Prints one JSON line and writes it to --out."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from seaiceextentforecasting_b200.config import LS, NORTH_INITS, SS  # noqa: E402
from seaiceextentforecasting_b200.engine import h2d  # noqa: E402
from seaiceextentforecasting_b200.forecast import (FIRST_YEAR, GP_ENSEMBLE_DTYPE, GP_RESULT_DTYPE,  # noqa: E402
                                                   EnsembleForecast, RetrospectiveSweep, ensemble_slots, gp_ensemble,
                                                   gp_ensemble_scratch_bytes)

B = 8                                  # members per batch (bench.MEMBERS)
LEVELS = (0.05, 0.5, 0.95)
HBM_GBS = 6541.8                       # measured B200 HBM read bandwidth (tools/marginal_sweep.py's reference)
SIZES = ((8, 1), (1024, 1), (8, 400), (64, 400), (1024, 400))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def marginal_sweep(ws):
    return RetrospectiveSweep(NORTH_INITS, [w["sic"] for w in ws], ws[0]["sie"], bench.FMIN, bench.FMAX,
                              ws[0]["psar"], [w["sst"] for w in ws], ws[0]["lat"], hyper_grid=(LS, SS),
                              hyper_mode="marginal", quantiles=LEVELS)


def components(rec):
    """Host replay of the kernel's staging on records [E][M][n]: (e > 0 component count [E], lo [E], hi [E])."""
    nl = np.where((rec["info"] == 0) & np.isfinite(rec["nlml"]), rec["nlml"], np.inf)
    m = nl.min(axis=2, keepdims=True)
    with np.errstate(invalid="ignore", over="ignore"):
        e = np.where(np.isfinite(m), np.exp(m - nl), 0.0)
    pos = e > 0
    sd = np.sqrt(np.maximum(np.where(pos, rec["fvar"], 0.0), 0.0))
    mu = np.where(pos, rec["fmean"], 0.0)
    lo = np.where(pos, mu - 40 * sd, np.inf).reshape(len(rec), -1).min(axis=1)
    hi = np.where(pos, mu + 40 * sd, -np.inf).reshape(len(rec), -1).max(axis=1)
    return pos.reshape(len(rec), -1).sum(axis=1), lo, hi


def halvings(lo, hi, result):
    """CDF passes of one level's bisection, replayed from its result: a visited midpoint c has F(c) >= q exactly when
    c >= the result, so the path is fixed by it."""
    if not (np.isfinite(result) and result != lo and result != hi):
        return 0 if result == lo else None         # lower end: no pass; upper end: unknown (<= 128), not counted
    a, b, n = lo, hi, 0
    for _ in range(128):
        c = 0.5 * a + 0.5 * b
        if c == a or c == b:
            break
        n += 1
        if c >= result:
            b = c
        else:
            a = c
    return n


def kernel_alone(base1, base400, E, reps):
    """base1 / base400: device records [E][8][n] of a real step; tiled to M slots."""
    q = torch.tensor(LEVELS, dtype=torch.float64, device="cuda")
    res = []
    for M, n in SIZES:
        base = base1 if n == 1 else base400
        rb = n * GP_RESULT_DTYPE.itemsize
        slot = torch.arange(M, device="cuda") % 8
        rec = base.view(E, 8, rb).index_select(1, slot).contiguous()
        out = torch.empty(E * GP_ENSEMBLE_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        quant = torch.empty(E * len(LEVELS), dtype=torch.float64, device="cuda")
        scratch = torch.empty(gp_ensemble_scratch_bytes(E, M, n), dtype=torch.uint8, device="cuda")
        gp_ensemble(rec, E, M, n, q, out, quant, scratch)            # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gp_ensemble(rec, E, M, n, q, out, quant, scratch)
        torch.cuda.synchronize()
        first = time.perf_counter() - t0
        k = int(max(3, min(reps, math.ceil(2.0 / max(first, 1e-6)))))
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        for a, b in evs:
            a.record()
            gp_ensemble(rec, E, M, n, q, out, quant, scratch)
            b.record()
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in evs)
        # host count of the work, from the 8 base members (slot s holds member s % 8)
        host = base.view(E, 8, rb).cpu().numpy().view(GP_RESULT_DTYPE).reshape(E, 8, n)
        reps8 = np.bincount(np.arange(M) % 8, minlength=8)
        cnt8 = np.array([components(host[:, i:i + 1])[0] for i in range(8)]).T          # [E][8]
        n_c = (cnt8 * reps8).sum(axis=1)
        _, lo, hi = components(host)
        qr = quant.cpu().numpy().reshape(E, len(LEVELS))
        passes, evals, unknown = np.zeros(E), 0.0, 0
        for e in range(E):
            if n_c[e] == 0:
                continue
            hv = [halvings(lo[e], hi[e], x) for x in qr[e]]
            unknown += sum(h is None for h in hv)
            hv = [h or 0 for h in hv]
            # one pass at (lo, hi), then per group of ENS_QB = 4 levels as many passes as its longest bisection
            passes[e] = 1 + sum(max(hv[i:i + 4]) for i in range(0, len(hv), 4))
            evals += float(n_c[e]) * (2 + sum(hv))
        rec_bytes = E * M * rb
        moved = rec_bytes + float(np.sum(n_c)) * 24 + float(np.sum(n_c * passes)) * 24
        med = statistics.median(ms)
        res.append({"M": M, "n_grid": n, "E": E, "launches_timed": k, "ms_median": med, "ms_min": ms[0],
                    "components_staged": int(np.sum(n_c)), "cdf_passes_per_problem_mean": float(np.mean(passes)),
                    "component_cdf_evaluations": evals, "component_cdf_evaluations_per_s": evals / (med * 1e-3),
                    "levels_at_the_upper_end_not_counted": int(unknown),
                    "record_bytes": rec_bytes, "bytes_moved_model": moved,
                    "gbs_model": moved / (med * 1e-3) / 1e9, "hbm_gbs_reference": HBM_GBS,
                    "store_gb": rec_bytes / 1e9, "scratch_gb": scratch.numel() / 1e9})
        del rec, scratch
        torch.cuda.empty_cache()
    return res


def obs_dt(plan, reg):
    return np.array([plan.sie_dt[reg][t - (plan.fmin - 1), t - FIRST_YEAR] for t in plan.years])


def coverage(plan, dicts, lo_hi):
    inside = total = 0
    for gpr in dicts:
        for cfg in plan.cfgs:
            g = gpr[cfg.name]
            for reg in cfg.regions:
                lo, hi = lo_hi(g, reg)
                obs = obs_dt(plan, reg)
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
    if isinstance(x, (np.floating, np.integer)):
        return clean(x.item())
    return x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    import __graft_entry__ as entry
    entry.build()
    result = {"tool": "tools/ensemble_sweep.py", "card": card(),
              "workload": f"bench.make_workload members, {B} per batch, north 4-init marginal sweep (432 problems per "
                          f"member, {len(LS)} x {len(SS)} grid), quantile levels {LEVELS}"}
    K = args.batches
    sw = marginal_sweep([bench.make_workload(m) for m in range(B)])
    sw.upload()
    sw.compute()
    ens = EnsembleForecast(sw, B * K, LEVELS)
    one = EnsembleForecast(sw, B, LEVELS)                             # the first batch: the kernel's base records
    one.add(sw)
    base400 = one.store.clone()
    E = one.E
    base1 = torch.empty(E * B * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    base1.view(E * B, -1).index_copy_(0, h2d(ensemble_slots(sw.plan, B)[1]),
                                      sw.gp.out[:sw.P * GP_RESULT_DTYPE.itemsize].view(sw.P, -1))
    del one
    torch.cuda.synchronize()
    result["kernel_alone"] = kernel_alone(base1, base400, E, args.kernel_reps)
    del base1, base400
    torch.cuda.empty_cache()

    ms = {"without_add": [], "with_add": []}
    members = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for b in range(K):
        ws = [bench.make_workload(B * b + i) for i in range(B)]
        sw.load_inputs([w["sic"] for w in ws], [w["sst"] for w in ws])
        for kind in (("without_add", "with_add") if b % 2 == 0 else ("with_add", "without_add")):
            torch.cuda.synchronize()
            e0.record()
            sw.upload()
            sw.compute()
            if kind == "with_add":
                ens.add(sw, B * b)
            e1.record()
            torch.cuda.synchronize()
            ms[kind].append(e0.elapsed_time(e1))
        members += sw.plan.assemble(sw.download(), marginal=sw.marginal)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d = ens.result()
    result_s = time.perf_counter() - t0
    plan = sw.plan
    med = {k: statistics.median(v) for k, v in ms.items()}
    result["streaming"] = {
        "batches": K, "members": B * K, "ms_per_step": ms, "median_ms_per_step": med,
        "add_overhead_ms_per_step": med["with_add"] - med["without_add"],
        "timing": "CUDA events around upload + compute (+ add) of one batch after a synchronise, the two kinds "
                  "alternated per batch (order reversed every other batch)",
        "result_s": result_s, "store_gb": ens.store.numel() / 1e9, "scratch_gb": ens._scratch.numel() / 1e9}
    member_skill = {}
    for gpr in members:
        for cfg, (rt, dt) in plan.skill(gpr).items():
            r = member_skill.setdefault(cfg, {"rt": [], "dt": []})
            r["rt"].append(rt)
            r["dt"].append(dt)
    ens_skill = {cfg: {"rt": rt, "dt": dt} for cfg, (rt, dt) in plan.skill(d).items()}
    result["skill"] = {"ensemble": ens_skill,
                       "mean_member": {c: {k: np.nanmean(np.asarray(v, dtype=float), axis=0).round(3).tolist()
                                           for k, v in r.items()} for c, r in member_skill.items()}}
    def interval(g, reg):
        return g[reg + "_quantiles"][:, 0], g[reg + "_quantiles"][:, -1]
    result["coverage_5_95"] = {"ensemble": coverage(plan, [d], interval),
                               "members_marginal": coverage(plan, members, interval)}
    r = ens.records
    ok = r["n_members"] > 0
    result["pool"] = {"problems": int(len(r)), "with_members": int(ok.sum()),
                      "n_members_quartiles": np.percentile(r["n_members"], [0, 25, 50, 75, 100]).tolist(),
                      "var_between_share_quartiles": np.percentile(r["var_between"][ok] / r["fvar"][ok],
                                                                   [0, 25, 50, 75, 100]).tolist()}
    result["note"] = "synthetic inputs: skill and coverage are a report, not evidence about real forecasts"
    line = json.dumps(clean(result))
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
