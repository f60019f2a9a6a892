"""GPU parity of the batched retrospective sweep (the bench workload) against the golden outputs of the unmodified
reference scripts (tests/golden/sweep_*.npz) and against the oracle on a multi-init north sweep."""
import glob
import os

import numpy as np
import pytest

from seaiceextentforecasting_b200 import synthetic as syn
from seaiceextentforecasting_b200.config import CONFIGS, NORTH_INITS

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SWEEPS = sorted(glob.glob(os.path.join(GOLD, "sweep_*.npz")))


def unpack_V(g, suffix=""):
    keys, lens, cells = g["V_keys" + suffix], g["V_lens" + suffix], g["V_cells" + suffix]
    V, off = {}, 0
    for k, ln in zip(keys, lens):
        V[int(k)] = [[int(a), int(b)] for a, b in cells[off:off + ln]]
        off += ln
    return V


def gp_tol(rec, cond):
    """1e-9 relative (north_star), widened only by the conditioning of the reference's own arithmetic: expm's s
    squarings amplify rounding by ~2^s (SURVEY.md H3; scipy itself moves that much under a 1-ulp input perturbation,
    tests/test_expm_spec.py) and two backward-stable Cholesky solves differ by ~cond(K) eps (SURVEY.md H4; `cond` is
    the oracle's 2-norm condition number of the kernel matrix)."""
    return max(1e-9, 64.0 * 2.0 ** int(rec["expm_s"]) * 2.0 ** -53, 8.0 * float(cond) * 2.0 ** -53)


def oracle_sweep(cfgs, sic, sie, fmin, fmax, psar, sst=None, lat=None):
    import warnings

    from oracle import sweep as osweep
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return osweep.retro_sweep(cfgs, sic, sie, fmin, fmax, psar, sst, lat, record_failures=True)


@pytest.mark.parametrize("path", SWEEPS, ids=[os.path.basename(p) for p in SWEEPS])
def test_sweep_matches_reference_golden(lib_built, path):
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    g = np.load(path)
    name = os.path.basename(path)[len("sweep_"):-len(".npz")]
    cfg = CONFIGS[name]
    fmin, fmax = int(g["fmin"]), int(g["fmax"])
    sie = {r: g["sie"][i] for i, r in enumerate(cfg.regions)}
    sw = RetrospectiveSweep([name], {name: g["sic"]}, sie, fmin, fmax, g["psar"],
                            g["sst"] if cfg.use_sst else None, g["sst_lat"] if cfg.use_sst else None)
    out = sw.run()
    raw = sw.raw
    assert (raw["info"] == 0).all()
    # condition numbers for the tolerance come from the oracle run on the same inputs (seconds at this size); its
    # forecasts must equal the golden ones (the oracle is pinned: tests/test_oracle_golden.py)
    ora = oracle_sweep([cfg], {name: g["sic"]}, sie, fmin, fmax, g["psar"], g["sst"] if cfg.use_sst else None,
                       g["sst_lat"] if cfg.use_sst else None)[name]
    # every network of the sweep: bit-exact area membership and order
    for (st, V), (ci, ny) in zip(sw.sic.areas_to_host(), sw.plan.jobs):
        assert st == 0
        assert V == unpack_V(g, f"_{ny}"), ny
    for k, reg in enumerate(cfg.regions):
        for i, year in enumerate(sw.years):
            rec = raw[sw.plan.prob_meta.index((0, k, year))]
            t = gp_tol(rec, ora[reg + "_cond"][i])
            rf, rv, rrt = (g["raw_" + reg + suf][i] for suf in ("_fmean", "_fvar", "_fmean_rt"))
            # natural scale of the predictive mean: itself or the predictive standard deviation (the mean is a sum of
            # O(sqrt(fvar))-sized terms that may cancel); of the variance: itself
            scale = max(abs(rf), np.sqrt(abs(rv)))
            assert abs(out[name][reg + "_raw_fmean"][i] - rf) <= t * scale, (reg, year, rec, rf)
            assert abs(out[name][reg + "_raw_fvar"][i] - rv) <= t * max(abs(rv), scale ** 2), (reg, year, rec, rv)
            assert abs(out[name][reg + "_raw_fmean_rt"][i] - rrt) <= t * max(scale, abs(rrt)), (reg, year, rec, rrt)
            # the reference's own output format: rounded to 3 d.p. -- checked wherever the conditioning-aware bound
            # is itself below the rounding step (July/Chukchi's l = 3.1e10 needs s ~ 56 squarings: scipy's own
            # result moves in the 3rd decimal under a 1-ulp input perturbation, tests/test_expm_spec.py)
            if t * max(scale, abs(rrt)) < 5e-4:
                for suf in ("_fmean", "_fvar", "_fmean_rt"):
                    assert abs(out[name][reg + suf][i] - g["rnd_" + reg + suf][i]) <= 1.0e-3 + 1e-12, (reg, suf, year)
    # skill() is a 3-d.p. output computed from the 3-d.p. forecasts: one unit in the last place (a forecast within the
    # bound above of a rounding boundary can move one digit) wherever every forecast of the region is well conditioned
    sk = sw.plan.skill(out)[name]
    for k, reg in enumerate(cfg.regions):
        recs = [raw[sw.plan.prob_meta.index((0, k, year))] for year in sw.years]
        if max(gp_tol(r, c) for r, c in zip(recs, ora[reg + "_cond"])) * 10.0 < 5e-4:
            assert abs(sk[0][k] - g["skill_rt"][k]) <= 1e-3 + 1e-12, (reg, sk[0][k], g["skill_rt"][k])
            assert abs(sk[1][k] - g["skill_dt"][k]) <= 1e-3 + 1e-12, (reg, sk[1][k], g["skill_dt"][k])


def test_multi_init_north_sweep_matches_oracle(lib_built):
    """All four north inits + SST in one batch (the bench's structure -- cross-config job indices, waves on separate
    streams, the SST-partitioned problem order -- at a size the oracle finishes in seconds).  Where the reference's
    forecast() raises (fewer than two predictors pass the selection rule) the kernel must report info = -1 for exactly
    that (config, region, year) and everything else must still match."""
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    fmin, fmax = 1993, 1996
    Tfull = fmax - 1979 + 1
    sic, sie0 = {}, None
    for i, name in enumerate(NORTH_INITS):
        f, _ = syn.make_field(15, 15, Tfull, 300 + i, n_modes=50, noise=0.5, blob=(1.0, 2.5))
        sic[name] = f
        if sie0 is None:
            sie0 = syn.make_sie(f, Tfull, 300)
    sie = dict(zip(CONFIGS["north_june"].regions, sie0))
    sst, _ = syn.make_field(8, 18, Tfull, 399, latlon=True, saturate=False, n_modes=20, noise=0.5, blob=(1.0, 2.5))
    psar, lat = syn.make_psar(15, 15), syn.make_lat_grid(8, 18)
    sw = RetrospectiveSweep(NORTH_INITS, sic, sie, fmin, fmax, psar, sst, lat, wave_T=(16,))
    assert sw.multi_wave                       # the multi-stream schedule is what is being tested
    out = sw.run()
    cfgs = [CONFIGS[n] for n in NORTH_INITS]
    ora = oracle_sweep(cfgs, sic, sie, fmin, fmax, psar, sst, lat)
    for (st, V), (ci, ny) in zip(sw.sic.areas_to_host(), sw.plan.jobs):
        assert V == ora[cfgs[ci].name]["V"][ny]
    n_ok = n_fail = 0
    for ci, cfg in enumerate(cfgs):
        for k, reg in enumerate(cfg.regions):
            for i, year in enumerate(sw.years):
                rec = sw.raw[sw.plan.prob_meta.index((ci, k, year))]
                if ora[cfg.name][reg + "_failed"][i] is not None:
                    assert rec["info"] == -1, (cfg.name, reg, year, rec)
                    assert np.isnan(out[cfg.name][reg + "_raw_fmean"][i])
                    n_fail += 1
                    continue
                assert rec["info"] == 0, (cfg.name, reg, year, rec)
                n_ok += 1
                t = gp_tol(rec, ora[cfg.name][reg + "_cond"][i])
                rf, rv = ora[cfg.name][reg + "_fmean"][i], ora[cfg.name][reg + "_fvar"][i]
                scale = max(abs(rf), np.sqrt(abs(rv)))      # the predictive standard deviation is the mean's scale
                assert abs(out[cfg.name][reg + "_raw_fmean"][i] - rf) <= t * scale, (cfg.name, reg, year, rec, rf)
                assert abs(out[cfg.name][reg + "_raw_fvar"][i] - rv) <= t * max(abs(rv), scale ** 2), (cfg.name, reg, year)
    assert n_ok >= 30 and n_fail >= 1 and n_ok + n_fail == 48


def test_time_varying_nan_mask_matches_oracle_and_capacity_failures_raise(lib_built):
    """A cell whose only NaN lies in a late year (data gap, mask change) is a node in the short windows and not in the
    long ones (`detrend` works on the prefix, north/retrospective_forecasts/September1st_retro.py:178-195): the node
    capacity must cover the largest window-specific node count, and the domains / forecasts must match the oracle for
    every window.  A build that exceeds a capacity must raise instead of returning NaN forecasts that look like a
    reference failure."""
    from seaiceextentforecasting_b200 import _lib
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    fmin, fmax = 1992, 1996
    Tfull = fmax - 1979 + 1
    f, _ = syn.make_field(15, 15, Tfull, 411, n_modes=50, noise=0.5, blob=(1.0, 2.5))
    f = f.copy()
    ocean = np.argwhere(~np.isnan(f).any(axis=2))
    rng = np.random.default_rng(5)
    pick = ocean[rng.choice(len(ocean), 12, replace=False)]
    for q, (i, j) in enumerate(pick):
        f[i, j, Tfull - 1 - (q % 3)] = np.nan          # NaN in one of the last three years only
    name = "north_september"
    cfg = CONFIGS[name]
    sie = dict(zip(cfg.regions, syn.make_sie(np.nan_to_num(f), Tfull, 411)))
    psar = syn.make_psar(15, 15)
    sw = RetrospectiveSweep([name], {name: f}, sie, fmin, fmax, psar)
    out = sw.run()
    n_nodes = sw.sic.n_nodes.cpu().numpy()
    assert len(set(n_nodes.tolist())) > 1                      # the windows really have different node sets
    ora = oracle_sweep([cfg], {name: f}, sie, fmin, fmax, psar)[name]
    for (st, V), (ci, ny) in zip(sw.sic.areas_to_host(), sw.plan.jobs):
        assert st == 0 and V == ora["V"][ny], ny
    for k, reg in enumerate(cfg.regions):
        for i, year in enumerate(sw.years):
            rec = sw.raw[sw.plan.prob_meta.index((0, k, year))]
            if ora[reg + "_failed"][i] is not None:
                assert rec["info"] == -1
                continue
            assert rec["info"] == 0
            t = gp_tol(rec, ora[reg + "_cond"][i])
            rf, rv = ora[reg + "_fmean"][i], ora[reg + "_fvar"][i]
            scale = max(abs(rf), np.sqrt(abs(rv)))
            assert abs(out[name][reg + "_raw_fmean"][i] - rf) <= t * scale, (reg, year, rec, rf)
            assert abs(out[name][reg + "_raw_fvar"][i] - rv) <= t * max(abs(rv), scale ** 2), (reg, year)
    # area capacity exceeded -> loud failure, not NaN records
    small = RetrospectiveSweep([name], {name: f}, sie, fmin, fmax, psar, max_areas=2)
    with pytest.raises(_lib.SieError):
        small.run()


def test_sweep_hyper_grid_contains_the_script_settings(lib_built):
    """configs[4]: the whole sweep on the 20 x 20 hyper-parameter grid.  The scripts' own (l, sigma) settings are grid
    points (`ls[16], ss[1]` ... north/June1st.py:210-213), so those grid entries must reproduce the forecasts."""
    import bench
    from seaiceextentforecasting_b200.config import CONFIGS
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    w = bench.make_workload(3)
    names = ["north_june", "north_september"]
    sw = RetrospectiveSweep(names, {n: w["sic"][n] for n in names}, w["sie"], 2012, 2020, w["psar"], w["sst"], w["lat"])
    sw.run()
    raw = sw.raw.copy()
    ells, sigs = np.logspace(-7, 2, 20), np.logspace(-3, 9, 20)
    grid = sw.hyper_grid(ells, sigs)
    assert grid.shape == (sw.P, 20, 20)
    hits = 0
    for p, (ci, k, year) in enumerate(sw.plan.prob_meta):
        cfg = sw.cfgs[ci]
        i = int(np.argmin(np.abs(np.log(ells) - np.log(cfg.ell[k]))))
        j = int(np.argmin(np.abs(np.log(sigs) - np.log(cfg.sig[k]))))
        if not (np.isclose(ells[i], cfg.ell[k], rtol=1e-12) and np.isclose(sigs[j], cfg.sig[k], rtol=1e-12)):
            continue
        g, r = grid[p, i, j], raw[p]
        assert g["info"] == r["info"] and g["n_pred"] == r["n_pred"]
        if r["info"] == 0:
            for key in ("fmean", "fvar", "sigma_f", "nlml"):
                assert abs(g[key] - r[key]) <= 1e-9 * max(1.0, abs(r[key])), (p, key, g[key], r[key])
        hits += 1
    assert hits >= sw.P // 2


def test_run_many_equals_run(lib_built):
    """`run_many(n)` (bench.py's end-to-end loop: step i's results are read back and assembled while step i+1 is on the
    device) yields, step by step, exactly what `run()` returns."""
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    fmin, fmax = 1993, 1996
    Tfull = fmax - 1979 + 1
    names = NORTH_INITS[1:3]
    sic = {}
    for i, name in enumerate(names):
        sic[name], _ = syn.make_field(15, 15, Tfull, 310 + i, n_modes=50, noise=0.5, blob=(1.0, 2.5))
    sie = dict(zip(CONFIGS[names[0]].regions, syn.make_sie(sic[names[0]], Tfull, 310)))
    sw = RetrospectiveSweep(names, sic, sie, fmin, fmax, syn.make_psar(15, 15))
    ref = sw.run()
    raw_ref = sw.raw.copy()
    outs = list(sw.run_many(3))
    assert len(outs) == 3
    sw.use_graph = True                      # the CUDA-graph replay of the step must give the same records
    outs += list(sw.run_many(2))
    for f in ("fmean", "fvar", "sigma_f", "nlml", "g_ell", "g_sig", "n_pred", "expm_m", "expm_s", "info"):   # not the cycle counters
        assert np.array_equal(sw.raw[f], raw_ref[f], equal_nan=True), f
    for out in outs:
        assert out.keys() == ref.keys()
        for cfg in ref:
            for k, v in ref[cfg].items():
                assert np.array_equal(np.asarray(out[cfg][k]), np.asarray(v), equal_nan=True), (cfg, k)
    assert sw.d2h_bytes() == sw.P * 80


def test_full_size_north_sweep_invariants(lib_built):
    """BASELINE.json configs[1] at its full size (the bench workload: 144 SIC 57x57 + 36 SST 26x90 networks, 432
    forecasts; the oracle needs ~10 minutes for it) through size-independent properties: every network builds, areas
    partition the labelled cells, the stored upper triangle of R is finite in [-1, 1] with a NaN diagonal, node series are the scaled sums of their
    member cells, every forecast but the known ill-conditioned July/Chukchi configuration is finite with positive variance,
    and a second run reproduces the first bit for bit."""
    import bench
    from seaiceextentforecasting_b200 import _lib
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    w = bench.make_workload(0)
    sw = RetrospectiveSweep(NORTH_INITS, w["sic"], w["sie"], bench.FMIN, bench.FMAX, w["psar"], w["sst"], w["lat"])
    out = sw.run()
    raw = sw.raw.copy()
    assert len(raw) == 432
    for eng in (sw.sic, sw.sst):
        st = eng.status.cpu().numpy()
        assert (st == _lib.SIE_JOB_OK).all()
        na = eng.n_areas.cpu().numpy()
        assert (na >= 2).all()
        lab = eng.label.cpu().numpy()
        starts = eng.area_start.cpu().numpy()
        cells = eng.area_cells.cpu().numpy()
        for b in (0, len(na) // 2, len(na) - 1):
            assert starts[b, na[b]] == (lab[b] >= 0).sum()                  # areas partition the labelled cells
            for a in (0, na[b] - 1):
                mem = cells[b, starts[b, a]:starts[b, a + 1]]
                assert (lab[b, mem] == a).all() and len(set(mem.tolist())) == len(mem)
        N = int(eng.n_nodes[0].item())
        R = eng.R[0, :N, :N].cpu().numpy()
        up = R[np.triu_indices(N, 1)]                                       # only the upper triangle is stored
        assert np.isnan(np.diag(R)).all() and np.isfinite(up).all() and np.abs(up).max() <= 1.0
        # node series of job 0, area 0: sequential row-major sum of dt * scale over the member cells (ComplexNetworks.py:303-306)
        T0 = int(eng.job_T[0].item())
        mem = np.sort(cells[0, starts[0, 0]:starts[0, 1]])
        dt0 = eng.dt[0].cpu().numpy()
        scale = (sw.dev["psar"] if eng is sw.sic else sw.dev["lat"]).cpu().numpy().reshape(-1)
        acc = np.zeros(T0)
        for c in mem:
            acc = acc + dt0[c, :T0] * scale[c]
        assert np.array_equal(eng.anomaly[0, 0, :T0].cpu().numpy(), acc)
    bad = raw["info"] != 0
    # the only non-zero info is -1 = "the reference's forecast() raises" (fewer than two predictors selected): the 6
    # (north_august, Chukchi) problems tests/golden/bench_north_m0.npz records for this workload
    assert (raw["info"][bad] == -1).all() and bad.sum() == 6
    ok = ~bad
    assert np.isfinite(raw["fmean"][ok]).all() and (raw["fvar"][ok] > 0).all()
    sw.run()
    for f in ("fmean", "fvar", "nlml", "n_pred", "info"):
        assert np.array_equal(sw.raw[f], raw[f], equal_nan=True), f
