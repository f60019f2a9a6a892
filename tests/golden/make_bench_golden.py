"""Full-size golden fixtures of the BENCHMARKED workloads, made by the UNMODIFIED reference (authoring container only).

    python tests/golden/make_bench_golden.py north0 [north1] [south] [--procs 6]

  * bench_north_m0.npz : BASELINE.json configs[1] = `bench.make_workload(0)`: 1985-2020 x June/July/August/September
                         inits x 3 regions (432 forecasts, 144 SIC 57x57 + 36 SST 26x90 network builds)
  * bench_north_m1.npz : the perturbed-SIC ensemble member `bench.make_workload(1)` (configs[4])
  * bench_south_feb.npz: BASELINE.json configs[2] = `bench.make_workload_south(0)`: south February 1985-2020 x 3
                         regions (108 forecasts, 36 SIC 81x81 network builds)

Every network is built by the reference's own `detrend` + `networks` functions (AST-lifted from the retrospective
script, calling /root/reference/ComplexNetworks.py as is; a recording wrapper around `Network.intra_links` only reads
`tau` off the object).  Every forecast is produced by the script's own `forecast()`, AST-lifted with two mechanical
edits: `.round(3)` stripped (un-rounded outputs; a second, un-stripped run gives the rounded ones and `skill`) and the
body of its `for year` loop wrapped in try/except so that a (year, region) on which the reference raises (no / one
predictor selected: IndexError / ValueError) is recorded as NaN instead of aborting the other 431 forecasts.
The oracle (`oracle/`) is run beside it on every GP problem and on a sample of the networks and must agree
(asserted here), which pins the oracle at full size too; its per-problem `sigma_f / nlml / n_pred` (values the
reference computes but does not return) are stored as well.

Node series (`anom`, float64 and nearly incompressible) are stored in full only for the networks of ANOM_YEARS
(`anom_jobs`), so that each fixture stays under 1 MB; every network keeps its per-area sum of squares (`anom_sumsq`,
aligned with `V_keys`) and its largest |value| (`anom_absmax`).
Inputs are NOT stored: they are regenerated from seeds by bench.make_workload*; `input_sha256` guards the generators.
Nothing is copied from the reference: functions are parsed out of the files where they lie and exec'd.
"""
import argparse
import ast
import hashlib
import inspect
import multiprocessing as mp
import os
import sys
import time
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
warnings.simplefilter("ignore")

import make_golden as mg  # noqa: E402  (imports the reference ComplexNetworks + the lifting helpers)

import bench  # noqa: E402
from oracle import gp as ogp  # noqa: E402
from oracle import sweep as osweep  # noqa: E402
from seaiceextentforecasting_b200.config import CONFIGS, RULE_ALL, RULE_POS, RULE_POS_SIG  # noqa: E402

REF = mg.REF
FMIN, FMAX = bench.FMIN, bench.FMAX
SCRIPTS = {name: rel for name, (rel, _, _) in mg.SWEEPS.items()}
# windows T = 7, 9, 21, 32, 42 (short to full length), incl. the networks tests/test_bench_golden_gpu.py rebuilds on the CPU
ANOM_YEARS = (1985, 1987, 1999, 2010, 2020)
_TAU_LOG = []
_orig_intra = mg.REFCN.Network.intra_links


def _recording_intra_links(self, *a, **k):       # reads tau off the object the reference's networks() keeps local
    _TAU_LOG.append(float(self.tau))
    return _orig_intra(self, *a, **k)


mg.REFCN.Network.intra_links = _recording_intra_links


class _TryYearBody(ast.NodeTransformer):
    """for year in ...: <body>   ->   for year in ...: try: <body> except (...): outputs[year-fmin] = nan"""

    def visit_For(self, node):
        self.generic_visit(node)
        if isinstance(node.target, ast.Name) and node.target.id == "year":
            handler = ast.parse(
                "try:\n    pass\nexcept (IndexError, ValueError, np.linalg.LinAlgError):\n"
                "    fmean[year-fmin] = np.nan\n    fvar[year-fmin] = np.nan\n    fmean_rt[year-fmin] = np.nan\n").body[0]
            handler.body = node.body
            node.body = [handler]
        return node


def lift_forecast(path, strip_round):
    tree = ast.parse(open(path, encoding="utf-8").read())
    ns = {"np": np, "linregress": mg.linregress, "pearsonr": mg.pearsonr, "expm": mg.expm, "CN": mg.REFCN}
    body = []
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in ("forecast", "skill"):
            if node.name == "forecast":
                if strip_round:
                    node = mg._StripRound3().visit(node)
                node = _TryYearBody().visit(node)
            body.append(node)
    mod = ast.Module(body=body, type_ignores=[])
    ast.fix_missing_locations(mod)
    exec(compile(mod, path, "exec"), ns)
    return ns


_W = {}


def _workload(kind):
    if kind not in _W:
        _W[kind] = bench.make_workload_south(0) if kind == "south" else bench.make_workload(int(kind[-1]))
    return _W[kind]


def _network_task(args):
    """One network build by the reference's detrend + networks (one year window)."""
    kind, name, year, check_oracle = args
    w = _workload(kind)
    t0 = time.perf_counter()
    if name == "sst":
        ns = mg.lift(os.path.join(REF, SCRIPTS["north_june"]), ("detrend", "networks"))
        ds = {"data": w["sst"], "lat": w["lat"]}
        latlon = True
    else:
        ns = mg.lift(os.path.join(REF, SCRIPTS[name]), ("detrend", "networks"))
        ds = {"data": w["sic"][name], "psar": w["psar"]}
        latlon = False
    ns["detrend"](ds, year, year)
    del _TAU_LOG[:]
    if "latlon" in inspect.signature(ns["networks"]).parameters:
        ns["networks"](ds, year, year, latlon=latlon)
    else:
        assert not latlon
        ns["networks"](ds, year, year)
    V, anoms = ds["nodes_" + str(year)], ds["anoms_" + str(year)]
    tau = _TAU_LOG[-1]
    if check_oracle:
        oV, oan, otau = osweep.build_network(ds["data"], year, latlon, w["lat"] if latlon else w["psar"])
        assert list(oV) == list(V) and all(oV[k] == V[k] for k in V), (kind, name, year, "oracle V differs")
        assert otau == tau, (kind, name, year, otau, tau)
        assert all(np.array_equal(oan[k], anoms[k]) for k in V), (kind, name, year, "oracle anomaly differs")
    keys, lens, cells = mg.pack_V(V)
    an = np.array([anoms[k] for k in V], dtype=np.float64)
    return dict(name=name, year=year, keys=keys, lens=lens, cells=cells.astype(np.int16), tau=tau, anom=an,
                seconds=time.perf_counter() - t0, oracle_checked=bool(check_oracle))


def input_digest(w):
    h = hashlib.sha256()
    for name in sorted(w["sic"]):
        h.update(np.ascontiguousarray(w["sic"][name]).tobytes())
    for reg in sorted(w["sie"]):
        h.update(np.ascontiguousarray(w["sie"][reg], dtype=np.float64).tobytes())
    if w.get("sst") is not None:
        h.update(np.ascontiguousarray(w["sst"]).tobytes())
    h.update(np.ascontiguousarray(w["psar"]).tobytes())
    return h.hexdigest()


def make(kind, procs):
    w = _workload(kind)
    names = list(w["sic"])
    use_sst = any(CONFIGS[n].use_sst for n in names)
    years = list(range(FMIN, FMAX + 1))
    tasks = [(kind, n, y, (i % 8) == 0) for i, (y, n) in enumerate((y, n) for y in reversed(years) for n in names)]
    if use_sst:
        tasks += [(kind, "sst", y, (y % 8) == 0) for y in reversed(years)]
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_network_task, tasks, chunksize=1)
    print(f"{kind}: {len(tasks)} reference network builds in {time.perf_counter() - t0:.0f} s wall, "
          f"{sum(r['seconds'] for r in res):.0f} s CPU", flush=True)
    nets = {(r["name"], r["year"]): r for r in res}

    # ---- GP: the scripts' own forecast()/skill() on the reference's node series
    regions = CONFIGS[names[0]].regions
    SIEs, SIEs_dt, SIEs_trend = mg.ref_read_sie_tables([w["sie"][r] for r in regions], regions, FMIN, FMAX)
    out = dict(kind=kind, fmin=FMIN, fmax=FMAX, input_sha256=input_digest(w), config_names=np.array(names),
               impl="reference (/root/reference, numpy %s)" % np.__version__)
    gp_rows = []
    for name in names:
        cfg = CONFIGS[name]
        SIC = {}
        for y in years:
            r = nets[(name, y)]
            V = {int(k): None for k in r["keys"]}
            SIC["anoms_" + str(y)] = {k: r["anom"][a] for a, k in enumerate(V)}
        SST = None
        if cfg.use_sst:
            SST = {}
            for y in years:
                r = nets[("sst", y)]
                SST["anoms_" + str(y)] = {int(k): r["anom"][a] for a, k in enumerate(r["keys"])}
        gpr = {}
        for tag, strip in (("raw", True), ("rnd", False)):
            ns = lift_forecast(os.path.join(REF, SCRIPTS[name]), strip)
            ns.update(SIEs=SIEs, SIEs_dt=SIEs_dt, SIEs_trend=SIEs_trend, SIC=SIC, SST=SST)
            GPR = ns["forecast"](FMIN, FMAX)
            gpr[tag] = GPR
            if tag == "rnd":
                ns["GPR"] = GPR
                sk_rt, sk_dt, _ = ns["skill"](FMIN, FMAX)
                out[f"skill_rt_{name}"] = np.array(sk_rt, dtype=np.float64)
                out[f"skill_dt_{name}"] = np.array(sk_dt, dtype=np.float64)
            for reg in regions:
                for suf in ("_fmean", "_fvar", "_fmean_rt"):
                    out[f"{tag}_{name}_{reg}{suf}"] = np.asarray(GPR[reg + suf], dtype=np.float64)
        # the oracle on every problem: must agree with the reference; supplies sigma_f / nlml / n_pred
        rule_name = {RULE_POS: "pos", RULE_ALL: "all", RULE_POS_SIG: "pos_sig"}
        for k, reg in enumerate(regions):
            for y in years:
                row = y - (FMIN - 1) - 1
                yv = SIEs_dt[reg][row, 0:y - 1979]
                slope, icpt = SIEs_trend[reg][row]
                ref_fm = gpr["raw"][reg + "_fmean"][y - FMIN]
                ref_fv = gpr["raw"][reg + "_fvar"][y - FMIN]
                try:
                    o = ogp.forecast_one(yv, SIC["anoms_" + str(y)], SST["anoms_" + str(y)] if SST else None,
                                         rule_name[cfg.rule[k]], cfg.alpha, cfg.zscore, cfg.ell[k], cfg.sig[k], slope,
                                         icpt, y - 1979)
                    failed = 0
                except (IndexError, ValueError, np.linalg.LinAlgError):
                    o = dict(fmean=np.nan, fvar=np.nan, sigma_f=np.nan, nlml=np.nan, n_pred=-1, cond=np.nan)
                    failed = 1
                assert failed == int(np.isnan(ref_fm)), (name, reg, y, "oracle and reference disagree on failure")
                if not failed:
                    assert abs(o["fmean"] - ref_fm) <= 1e-10 * max(1.0, abs(ref_fm)), (name, reg, y, o["fmean"], ref_fm)
                    assert abs(o["fvar"] - ref_fv) <= 1e-10 * max(1.0, abs(ref_fv)), (name, reg, y, o["fvar"], ref_fv)
                gp_rows.append((names.index(name), k, y, o["fmean"], o["fvar"], o["sigma_f"], o["nlml"], o["n_pred"],
                                failed, o["cond"]))
    g = np.array(gp_rows, dtype=np.float64)
    out.update(gp_cfg=g[:, 0].astype(np.int32), gp_region=g[:, 1].astype(np.int32), gp_year=g[:, 2].astype(np.int32),
               gp_fmean=g[:, 3], gp_fvar=g[:, 4], gp_sigma_f=g[:, 5], gp_nlml=g[:, 6], gp_n_pred=g[:, 7].astype(np.int32),
               gp_failed=g[:, 8].astype(np.int8), gp_cond=g[:, 9])
    # ---- networks, job order = task order
    out["job_cfg"] = np.array([names.index(t[1]) if t[1] != "sst" else -1 for t in tasks], dtype=np.int32)
    out["job_year"] = np.array([t[2] for t in tasks], dtype=np.int32)
    out["job_tau"] = np.array([nets[(t[1], t[2])]["tau"] for t in tasks])
    out["job_oracle_checked"] = np.array([nets[(t[1], t[2])]["oracle_checked"] for t in tasks])
    out["V_nkeys"] = np.array([len(nets[(t[1], t[2])]["keys"]) for t in tasks], dtype=np.int32)
    out["V_keys"] = np.concatenate([nets[(t[1], t[2])]["keys"] for t in tasks]).astype(np.int32)
    out["V_lens"] = np.concatenate([nets[(t[1], t[2])]["lens"] for t in tasks]).astype(np.int32)
    out["V_cells"] = np.concatenate([nets[(t[1], t[2])]["cells"] for t in tasks]).astype(np.int16)
    anoms = [nets[(t[1], t[2])]["anom"] for t in tasks]
    out["anom_sumsq"] = np.concatenate([(a * a).sum(axis=1) for a in anoms])
    out["anom_absmax"] = np.array([np.abs(a).max() for a in anoms])
    out["anom_jobs"] = np.array([j for j, t in enumerate(tasks) if t[2] in ANOM_YEARS], dtype=np.int32)
    out["anom"] = np.concatenate([anoms[j].reshape(-1) for j in out["anom_jobs"]])
    fname = {"north0": "bench_north_m0.npz", "north1": "bench_north_m1.npz", "south": "bench_south_feb.npz"}[kind]
    np.savez_compressed(os.path.join(HERE, fname), **out)
    nfail = int(out["gp_failed"].sum())
    print(f"{kind}: wrote {fname}: {len(tasks)} networks, {len(gp_rows)} forecasts, {nfail} on which the reference raises; "
          f"max n_pred {int(out['gp_n_pred'].max())}, areas {int(out['V_nkeys'].min())}..{int(out['V_nkeys'].max())}",
          flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("kinds", nargs="+", choices=["north0", "north1", "south"])
    ap.add_argument("--procs", type=int, default=6)
    a = ap.parse_args()
    for kind in a.kinds:
        make(kind, a.procs)
