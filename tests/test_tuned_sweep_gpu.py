"""Tuned retrospective sweeps (RetrospectiveSweep(hyper_grid=(ells, sigs))): every forecast at the on-device minimum of
MLII's nlML over the reference's (l, sigma_n~) grid (north/June1st.py:210-211), against numpy's argmin over the grid
records, the plain forecast at the selected point, the oracle's MLII on the whole grid, across schedules, and through
ensemble streaming (load_inputs)."""
import warnings

import numpy as np
import pytest

from seaiceextentforecasting_b200 import synthetic as syn
from seaiceextentforecasting_b200.config import CONFIGS, LS, NORTH_INITS, SS

pytestmark = pytest.mark.gpu
FMIN, FMAX = 1993, 1996
FIELDS = ("fmean", "fvar", "sigma_f", "nlml", "g_ell", "g_sig", "n_pred", "expm_m", "expm_s", "info")   # not the cycles


def gp_tol(rec, cond):
    """The conditioning-aware bound of tests/test_sweep_gpu.py."""
    return max(1e-9, 64.0 * 2.0 ** int(rec["expm_s"]) * 2.0 ** -53, 8.0 * float(cond) * 2.0 ** -53)


def small_inputs(member=0):
    """The 4-init + SST north sweep of test_multi_init_north_sweep_matches_oracle (15x15, 1993-1996); member > 0 is
    perturbed like bench.make_workload's ensemble members (same land / NaN mask, so the same capacities)."""
    Tfull = FMAX - 1979 + 1
    sic, sie0 = {}, None
    for i, name in enumerate(NORTH_INITS):
        f, _ = syn.make_field(15, 15, Tfull, 300 + i, n_modes=50, noise=0.5, blob=(1.0, 2.5))
        sic[name] = f
        if sie0 is None:
            sie0 = syn.make_sie(f, Tfull, 300)
    sie = dict(zip(CONFIGS["north_june"].regions, sie0))
    sst, _ = syn.make_field(8, 18, Tfull, 399, latlon=True, saturate=False, n_modes=20, noise=0.5, blob=(1.0, 2.5))
    if member > 0:
        rng = np.random.default_rng(5000 + member)
        for name in NORTH_INITS:
            f = sic[name]
            inside = (f > 0.0) & (f < 1.0)
            sic[name] = np.where(inside, np.clip(f + 0.05 * rng.standard_normal(f.shape), 0.0, 1.0), f)
        sst = sst + 0.05 * rng.standard_normal(sst.shape)
    return dict(sic=sic, sie=sie, sst=sst, psar=syn.make_psar(15, 15), lat=syn.make_lat_grid(8, 18))


def small_sweep(w, hyper_grid=(LS, SS)):
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    return RetrospectiveSweep(NORTH_INITS, w["sic"], w["sie"], FMIN, FMAX, w["psar"], w["sst"], w["lat"], wave_T=(16,),
                              hyper_grid=hyper_grid)


def numpy_argmin(rec):
    nl = np.where((rec["info"] == 0) & np.isfinite(rec["nlml"]), rec["nlml"], np.inf).ravel()
    return -1 if np.isinf(nl).all() else int(np.argmin(nl))


def assert_same_records(a, b):
    for f in FIELDS:
        assert np.array_equal(a[f], b[f], equal_nan=True), f


@pytest.fixture(scope="module")
def tuned_small(lib_built):
    w = small_inputs()
    sw = small_sweep(w)
    assert sw.multi_wave and sw.gp_sst          # waves on separate streams + the SST split: every GP launch kind
    out = sw.run()
    return w, sw, out, sw.raw.copy(), sw.grid_records(), sw.best_index(), sw.tuned_problems()


def test_selection_is_numpy_argmin(tuned_small):
    _, sw, out, raw, grid, best, tuned = tuned_small
    assert grid.shape == (sw.P, len(LS), len(SS)) and best.shape == (sw.P,)
    for p in range(sw.P):
        assert best[p] == numpy_argmin(grid[p]), p
    assert (best >= 0).sum() >= 30 and (best == -1).sum() >= 1
    # the tuned dict carries what each forecast used
    for p, (ci, k, year) in enumerate(sw.plan.prob_meta):
        g = out[sw.cfgs[ci].name]
        reg, i = sw.cfgs[ci].regions[k], year - FMIN
        assert g[reg + "_grid_index"][i] == best[p]
        assert g[reg + "_ell"][i] == tuned["ell"][p] and g[reg + "_sig"][i] == tuned["sig"][p]


def test_tuned_forecast_is_the_plain_forecast_at_the_selected_point(tuned_small):
    from seaiceextentforecasting_b200.engine import h2d
    from seaiceextentforecasting_b200.forecast import GpBatch
    _, sw, _, raw, grid, best, tuned = tuned_small
    host = sw.plan.prob.copy()
    nsig = len(SS)
    for p in range(sw.P):
        if best[p] >= 0:
            host["ell"][p], host["sig"][p] = LS[best[p] // nsig], SS[best[p] % nsig]
    assert tuned.tobytes() == host.tobytes()
    gp = GpBatch(sw.P, max_pred=sw.gp.max_pred)
    gp.run(h2d(host.view(np.uint8)), sw.dev["y"], sw.sic, sw.sst)
    assert_same_records(gp.results()[:sw.P], raw)
    for p in np.nonzero((best >= 0) & (raw["info"] == 0))[0]:
        g = grid[p].reshape(-1)[best[p]]
        assert abs(raw["nlml"][p] - g["nlml"]) <= 1e-9 * max(1.0, abs(g["nlml"])), (p, raw[p], g)


def test_tuned_sweep_matches_oracle_mlii_on_the_grid(tuned_small):
    """The oracle's MLII (north/June1st.py:235-257) on all 400 grid points of every problem: the GPU's choice is the
    oracle's minimum up to the conditioning-aware bound (the same index wherever the runner-up is farther away than
    that), and the forecast there is the oracle's."""
    from oracle import gp as ogp
    from oracle import sweep as osw
    w, sw, out, raw, grid, best, _ = tuned_small
    years = sw.years
    tables = {reg: osw.sie_tables(w["sie"][reg], FMIN, FMAX) for reg in CONFIGS["north_june"].regions}
    sst_nets = {}
    n_ok = n_fail = n_strict = 0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for ci, cfg in enumerate(sw.cfgs):
            for year in years:
                _, anoms, _ = osw.build_network(w["sic"][cfg.name], year, False, w["psar"])
                sst_anoms = None
                if cfg.use_sst:
                    if year not in sst_nets:
                        sst_nets[year] = osw.build_network(w["sst"], year, True, w["lat"])[1]
                    sst_anoms = sst_nets[year]
                for k, reg in enumerate(cfg.regions):
                    p = sw.plan.prob_meta.index((ci, k, year))
                    row = year - (FMIN - 1) - 1
                    y = tables[reg][0][row, 0:year - 1979]
                    slope, icpt = tables[reg][1][row]
                    try:
                        Xfull = ogp.select_predictors(y, anoms, sst_anoms, osw._RULES[cfg.rule[k]], cfg.alpha)
                        X, Xs, M = ogp.design(Xfull, cfg.zscore)
                    except osw.FAILS:                   # the reference's forecast() raises: same as the plain sweep
                        assert best[p] == -1 and raw["info"][p] == -1, (cfg.name, reg, year, raw[p])
                        assert np.isnan(out[cfg.name][reg + "_raw_fmean"][year - FMIN])
                        n_fail += 1
                        continue
                    yc = y[:, None]
                    nl = np.array([[ogp.mlii((np.log(l), np.log(s)), X, yc, M)[0] for s in SS] for l in LS]).ravel()
                    nl = np.where(np.isfinite(nl), nl, np.inf)
                    assert np.isfinite(nl).any() and best[p] >= 0, (cfg.name, reg, year)
                    b, ob = int(best[p]), int(np.argmin(nl))
                    assert np.isfinite(nl[b]), (cfg.name, reg, year, b, ob)
                    at_b = ogp.gp_fit_predict(X, Xs, yc, M, LS[b // len(SS)], SS[b % len(SS)])
                    at_ob = ogp.gp_fit_predict(X, Xs, yc, M, LS[ob // len(SS)], SS[ob % len(SS)])
                    t = max(gp_tol(raw[p], at_b["cond"]), gp_tol(grid[p].reshape(-1)[ob], at_ob["cond"]))
                    lo = nl[ob]
                    assert nl[b] - lo <= t * max(1.0, abs(lo)), (cfg.name, reg, year, b, ob, nl[b], lo, t)
                    second = np.partition(nl, 1)[1]
                    if second - lo > t * max(1.0, abs(lo)):
                        assert b == ob, (cfg.name, reg, year, b, ob, lo, second)
                        n_strict += 1
                    # the forecast at the selected point
                    tb = gp_tol(raw[p], at_b["cond"])
                    rf, rv = at_b["fmean"], at_b["fvar"]
                    rrt = rf + (slope * (year - 1979) + icpt)
                    scale = max(abs(rf), np.sqrt(abs(rv)))
                    g, i = out[cfg.name], year - FMIN
                    assert raw["info"][p] == 0
                    assert abs(g[reg + "_raw_fmean"][i] - rf) <= tb * scale, (cfg.name, reg, year, raw[p], rf)
                    assert abs(g[reg + "_raw_fvar"][i] - rv) <= tb * max(abs(rv), scale ** 2), (cfg.name, reg, year)
                    assert abs(g[reg + "_raw_fmean_rt"][i] - rrt) <= tb * max(scale, abs(rrt)), (cfg.name, reg, year)
                    n_ok += 1
    assert n_ok >= 30 and n_fail >= 1 and n_ok + n_fail == 48 and n_strict >= 1, (n_ok, n_fail, n_strict)
    print(f"oracle grid parity: {n_ok} tuned forecasts, {n_strict} with a unique minimum, {n_fail} reference failures")


def test_tuned_records_do_not_depend_on_the_schedule(tuned_small):
    """waves = 0 (one stream), waves = 1, the multi-wave default, run_many and CUDA-graph replay: the same records."""
    _, _, _, raw, grid, best, tuned = tuned_small
    sw = small_sweep(small_inputs())
    sw.upload()
    results = []
    for waves in (0, 1, None):
        sw.compute(waves=waves)
        results.append((sw.download().copy(), sw.selection.copy(), sw.grid_records()))
    outs = list(sw.run_many(2))
    results.append((sw.raw.copy(), sw.selection.copy(), sw.grid_records()))
    sw.use_graph = True
    outs += list(sw.run_many(2))
    results.append((sw.raw.copy(), sw.selection.copy(), sw.grid_records()))
    for r, sel, gr in results:
        assert_same_records(r, raw)
        assert np.array_equal(sel["best"], best)
        assert np.array_equal(sel["ell"], tuned["ell"]) and np.array_equal(sel["sig"], tuned["sig"])
        assert_same_records(gr, grid)
    for o in outs[1:]:
        for c in outs[0]:
            for k, v in outs[0][c].items():
                assert np.array_equal(o[c][k], v, equal_nan=True), (c, k)


def test_load_inputs_streams_a_new_member(lib_built):
    """A sweep built for member 0 and fed member 1 through load_inputs == a sweep constructed on member 1."""
    w0, w1 = small_inputs(0), small_inputs(1)
    a = small_sweep(w0)
    a.run()
    raw0 = a.raw.copy()
    a.load_inputs(w1["sic"], w1["sst"])
    out_a = a.run()
    b = small_sweep(w1)
    out_b = b.run()
    assert not np.array_equal(raw0["fmean"], b.raw["fmean"], equal_nan=True)     # the members really differ
    assert_same_records(a.raw, b.raw)
    assert np.array_equal(a.selection, b.selection)
    for c in out_b:
        for k, v in out_b[c].items():
            assert np.array_equal(out_a[c][k], v, equal_nan=True), (c, k)
    list(a.run_many(2))                                                 # the double-buffered loop reads the new inputs too
    assert_same_records(a.raw, b.raw)
    with pytest.raises(ValueError):
        a.load_inputs([w1["sic"], w1["sic"]])


def test_full_size_tuned_step_invariants(lib_built):
    """The bench's 8-member north step (bench.make_workload): every problem the plain sweep solves finds an admissible
    grid point, and wherever the script's (l, sigma_n~) is itself a grid point the tuned nlML is not above it."""
    import torch

    import bench
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    ws = [bench.make_workload(m) for m in range(8)]
    args = (NORTH_INITS, [x["sic"] for x in ws], ws[0]["sie"], bench.FMIN, bench.FMAX, ws[0]["psar"],
            [x["sst"] for x in ws], ws[0]["lat"])
    plain = RetrospectiveSweep(*args)
    plain.run()
    raw_plain = plain.raw.copy()
    del plain
    torch.cuda.empty_cache()
    sw = RetrospectiveSweep(*args, hyper_grid=(LS, SS))
    out = sw.run()
    assert len(out) == 8 and len(sw.raw) == 8 * 432
    best, grid = sw.best_index(), sw.grid_records()
    assert (best[raw_plain["info"] == 0] >= 0).all()
    assert (sw.raw["info"][best >= 0] == 0).all()
    hits = 0
    for p, (ci, k, year) in enumerate(sw.plan.prob_meta):
        cfg = sw.cfgs[ci]
        i = int(np.argmin(np.abs(np.log(LS) - np.log(cfg.ell[k]))))
        j = int(np.argmin(np.abs(np.log(SS) - np.log(cfg.sig[k]))))
        if not (np.isclose(LS[i], cfg.ell[k], rtol=1e-12) and np.isclose(SS[j], cfg.sig[k], rtol=1e-12)):
            continue
        g = grid[p, i, j]
        if g["info"] != 0 or not np.isfinite(g["nlml"]):
            continue
        assert sw.raw["nlml"][p] <= g["nlml"] + 1e-9 * max(1.0, abs(g["nlml"])), (p, sw.raw[p], g)
        hits += 1
    assert hits >= sw.P // 2
