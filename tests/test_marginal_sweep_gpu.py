"""Marginalised retrospective sweeps (RetrospectiveSweep(hyper_grid=(ells, sigs), hyper_mode="marginal")): every
forecast the marginal-likelihood-weighted average of its problem's forecasts over the reference's (l, sigma_n~) grid
(north/June1st.py:210-211), with predictive quantiles of the mixture.  Checked against oracle/marginal.py on the
device's own grid records, on hand-made records, against the oracle's GP fits at every grid point, across schedules,
through ensemble streaming (load_inputs) and at full size."""
import warnings

import numpy as np
import pytest

from seaiceextentforecasting_b200.config import CONFIGS, LS, NORTH_INITS, SS
from test_tuned_sweep_gpu import FIELDS, FMAX, FMIN, gp_tol, small_inputs

pytestmark = pytest.mark.gpu
LEVELS = (0.05, 0.25, 0.5, 0.75, 0.95)
MOMENTS = ("fmean", "fvar", "nlml")


def marginal_sweep(w, levels=LEVELS):
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    return RetrospectiveSweep(NORTH_INITS, w["sic"], w["sie"], FMIN, FMAX, w["psar"], w["sst"], w["lat"], wave_T=(16,),
                              hyper_grid=(LS, SS), hyper_mode="marginal", quantiles=levels)


def device_best(sw):
    """sie_gp_grid_select's choice on the sweep's device grid records."""
    import torch

    from seaiceextentforecasting_b200.forecast import GP_PROBLEM_DTYPE, grid_select
    g = sw.tune
    tuned = torch.empty(sw.P * GP_PROBLEM_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    best = torch.empty(sw.P, dtype=torch.int32, device="cuda")
    grid_select(g.out, sw.dev["prob"], sw.P, g.ell_dev, g.sig_dev, tuned, best)
    return best.cpu().numpy()


def run_marginal(rec, levels=LEVELS):
    """sie_gp_grid_marginal on host records rec [P][n_grid] -> (records [P], stats [P], quantiles [P][n_q])."""
    import torch

    from seaiceextentforecasting_b200.engine import h2d
    from seaiceextentforecasting_b200.forecast import GP_MARGINAL_DTYPE, GP_RESULT_DTYPE, grid_marginal
    P, n = rec.shape
    nq = len(levels)
    out = torch.empty(P * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    stats = torch.empty(P * GP_MARGINAL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    quant = torch.empty(max(1, P * nq), dtype=torch.float64, device="cuda")
    grid_marginal(h2d(np.ascontiguousarray(rec).view(np.uint8).reshape(-1)), P, n,
                  h2d(np.asarray(levels, dtype=np.float64)) if nq else None, out, stats, quant)
    return (out.cpu().numpy().view(GP_RESULT_DTYPE), stats.cpu().numpy().view(GP_MARGINAL_DTYPE),
            quant.cpu().numpy()[:P * nq].reshape(P, nq))


def check_against_numpy(grid, raw, stats, quant, levels=LEVELS, jumps=False):
    """The device's marginal of every problem == oracle/marginal.py on the same records (1e-13 relative; the quantiles
    through the oracle CDF, within 1e-12 of their level -- `jumps` (point masses): F(x) >= q > F(the next lower double)
    within 1e-12).  Returns the number of problems with |A| >= 1."""
    from oracle import marginal as om
    n_ok = 0
    for p in range(len(raw)):
        g = grid[p].reshape(-1)
        r = om.marginal(g["fmean"], g["fvar"], g["nlml"], g["info"], levels)
        assert stats["n_admissible"][p] == r["n_admissible"] and stats["argmax"][p] == r["argmax"], p
        if r["n_admissible"] == 0:
            assert all(np.isnan(raw[f][p]) for f in MOMENTS) and np.isnan(quant[p]).all(), p
            assert np.isnan(stats["ess"][p]) and np.isnan(stats["w_max"][p])
            for f in FIELDS:
                if f not in MOMENTS:
                    assert np.array_equal(raw[f][p], g[f][0], equal_nan=True), (p, f)
            continue
        scale = max(abs(r["fmean"]), np.sqrt(r["fvar"]))
        assert abs(raw["fmean"][p] - r["fmean"]) <= 1e-13 * scale, (p, raw["fmean"][p], r["fmean"])
        assert abs(raw["fvar"][p] - r["fvar"]) <= 1e-13 * r["fvar"], (p, raw["fvar"][p], r["fvar"])
        assert abs(raw["nlml"][p] - r["nlml"]) <= 1e-13 * max(1.0, abs(r["nlml"])), (p, raw["nlml"][p], r["nlml"])
        assert abs(stats["ess"][p] - r["ess"]) <= 1e-13 * r["ess"], p
        assert abs(stats["w_max"][p] - r["w_max"]) <= 1e-13 * r["w_max"], p
        for f in FIELDS:                                   # every other field is the largest-weight record's
            if f not in MOMENTS:
                assert np.array_equal(raw[f][p], g[f][r["argmax"]], equal_nan=True), (p, f)
        adm = r["w"] > 0
        mu, var = np.where(adm, g["fmean"], 0.0), np.where(adm, g["fvar"], 0.0)
        for t, x in zip(levels, quant[p]):
            if jumps:
                assert om.mixture_cdf(x, r["w"], mu, var) >= t - 1e-12, (p, t, x)
                assert om.mixture_cdf(np.nextafter(x, -np.inf), r["w"], mu, var) < t + 1e-12, (p, t, x)
            else:
                assert abs(om.mixture_cdf(x, r["w"], mu, var) - t) <= 1e-12, (p, t, x)
        assert np.all(np.diff(quant[p]) >= 0), p
        n_ok += 1
    return n_ok


@pytest.fixture(scope="module")
def marg_small(lib_built):
    w = small_inputs()
    sw = marginal_sweep(w)
    assert sw.multi_wave and sw.gp_sst          # waves on separate streams + the SST split: every GP launch kind
    out = sw.run()
    return w, sw, out, sw.raw.copy(), sw.marginal.copy(), sw.grid_records()


def test_marginal_matches_numpy_on_the_device_records(marg_small):
    _, sw, out, raw, marg, grid = marg_small
    assert grid.shape == (sw.P, len(LS), len(SS)) and marg["quantiles"].shape == (sw.P, len(LEVELS))
    n_ok = check_against_numpy(grid, raw, marg, marg["quantiles"])
    assert n_ok >= 30 and (marg["n_admissible"] == 0).sum() >= 1, n_ok
    assert (raw["info"][marg["n_admissible"] == 0] == -1).all()      # a reference failure keeps info = -1
    assert np.array_equal(marg["argmax"], device_best(sw))           # argmax == sie_gp_grid_select's best
    for p, (ci, k, year) in enumerate(sw.plan.prob_meta):            # the assembled dict carries the posterior
        g, reg, i = out[sw.cfgs[ci].name], sw.cfgs[ci].regions[k], year - FMIN
        assert g[reg + "_grid_index"][i] == marg["argmax"][p]
        assert np.array_equal(g[reg + "_ess"][i], marg["ess"][p], equal_nan=True)
        assert np.array_equal(g[reg + "_quantiles"][i], marg["quantiles"][p], equal_nan=True)
        assert g[reg + "_raw_fmean"][i] == raw["fmean"][p] or np.isnan(raw["fmean"][p])
    print(f"marginal == numpy on device records: {n_ok} problems, median ESS {np.nanmedian(marg['ess']):.1f}")


def test_one_admissible_point_is_that_record_bit_for_bit(marg_small):
    _, sw, _, _, marg, grid = marg_small
    p = int(np.nonzero(marg["n_admissible"] >= 2)[0][0])
    rec = grid[p].reshape(1, -1).copy()
    keep = int(np.nonzero((rec["info"][0] == 0) & np.isfinite(rec["nlml"][0]))[0][-1])
    rec["info"][0, np.arange(rec.shape[1]) != keep] = 1
    raw, stats, quant = run_marginal(rec)
    assert raw["fmean"][0] == rec["fmean"][0, keep] and raw["fvar"][0] == rec["fvar"][0, keep]
    assert raw["nlml"][0] == rec["nlml"][0, keep]
    assert stats["ess"][0] == 1.0 and stats["w_max"][0] == 1.0 and stats["argmax"][0] == keep
    check_against_numpy(rec.reshape(1, 1, -1), raw, stats, quant)


def test_hand_made_records(lib_built):
    """A empty, one point, nlML ties, v <= 0 (point masses), an nlML spread of 1e4 (weights underflow to 0), and a grid
    past the shared-memory stage (same bits as the staged path when the extra points carry no weight)."""
    from seaiceextentforecasting_b200.forecast import GP_RESULT_DTYPE
    rng = np.random.default_rng(11)
    n, P = 400, 6
    rec = np.zeros((P, n), dtype=GP_RESULT_DTYPE)
    rec["fmean"] = rng.normal(0.0, 0.4, (P, n))
    rec["fvar"] = rng.uniform(0.01, 0.3, (P, n))
    rec["nlml"] = rng.uniform(-3.0, 3.0, (P, n))
    rec["sigma_f"] = np.arange(P * n).reshape(P, n)               # names the record the other fields come from
    rec["info"][0] = 2                                            # 0: A empty (failed points)
    rec["info"][0, 5] = -1
    rec["nlml"][0, :7] = np.inf
    rec["info"][1] = 1                                            # 1: one point
    rec["info"][1, 123] = 0
    rec["nlml"][2] = 4.25                                         # 2: all tied -> uniform weights, argmax 0
    rec["fvar"][3, ::3] = 0.0                                     # 3: point masses and negative variances
    rec["fvar"][3, 1::7] = -1e-9
    rec["nlml"][3, 0::3] -= 2.0
    rec["nlml"][4] = rng.uniform(0.0, 1e4, n)                     # 4: spread 1e4
    rec["nlml"][5, 1::2] = np.nan                                 # 5: half the points have a NaN nlML
    raw, stats, quant = run_marginal(rec)
    check_against_numpy(rec.reshape(P, 1, n), raw, stats, quant, jumps=True)
    assert np.isnan(raw["fmean"][0]) and raw["info"][0] == 2 and raw["sigma_f"][0] == rec["sigma_f"][0, 0]
    assert stats["n_admissible"][0] == 0 and stats["argmax"][0] == -1
    assert raw["fmean"][1] == rec["fmean"][1, 123] and raw["fvar"][1] == rec["fvar"][1, 123]
    assert np.allclose(stats["ess"][2], n, rtol=1e-13) and stats["argmax"][2] == 0
    assert np.isfinite(raw["fmean"][4]) and np.isfinite(raw["fvar"][4]) and np.isfinite(quant[4]).all()
    assert np.isfinite(stats["ess"][4]) and stats["ess"][4] >= 1.0
    assert stats["n_admissible"][5] == n // 2
    # 520 points > the 500 staged in shared memory: the extra inadmissible points change no bit
    big = np.zeros((P, 520), dtype=GP_RESULT_DTYPE)
    big[:, :n] = rec
    big["info"][:, n:] = 1
    big["nlml"][:, n:] = -1e6
    raw2, stats2, quant2 = run_marginal(big)
    for f in FIELDS:
        assert np.array_equal(raw2[f], raw[f], equal_nan=True), f
    assert stats2.tobytes() == stats.tobytes() and np.array_equal(quant2, quant, equal_nan=True)
    _, _, none = run_marginal(rec, levels=())                     # no quantiles: NULL q / quant
    assert none.shape == (P, 0)


@pytest.fixture(scope="module")
def oracle_fits(marg_small):
    """oracle.gp.gp_fit_predict at all 400 grid points of every problem of the small sweep:
    {p: (fits [n_ell * n_sig] of dicts or None where the oracle raises)}, and the problems where the reference fails.
    Each fit also carries `prior_var` = k(x*, x*) + sigma_n = sigma_f (x* expm(l M) x*^T + sigma_n~), the prior
    variance fvar is computed from (fvar = prior_var - v^T v)."""
    from scipy.linalg import expm

    from oracle import gp as ogp
    from oracle import sweep as osw
    w, sw, _, _, _, _ = marg_small
    tables = {reg: osw.sie_tables(w["sie"][reg], FMIN, FMAX) for reg in CONFIGS["north_june"].regions}
    fits, fails, sst_nets = {}, [], {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for ci, cfg in enumerate(sw.cfgs):
            for year in sw.years:
                _, anoms, _ = osw.build_network(w["sic"][cfg.name], year, False, w["psar"])
                sst_anoms = None
                if cfg.use_sst:
                    if year not in sst_nets:
                        sst_nets[year] = osw.build_network(w["sst"], year, True, w["lat"])[1]
                    sst_anoms = sst_nets[year]
                for k, reg in enumerate(cfg.regions):
                    p = sw.plan.prob_meta.index((ci, k, year))
                    y = tables[reg][0][year - (FMIN - 1) - 1, 0:year - 1979]
                    try:
                        Xfull = ogp.select_predictors(y, anoms, sst_anoms, osw._RULES[cfg.rule[k]], cfg.alpha)
                        X, Xs, M = ogp.design(Xfull, cfg.zscore)
                    except osw.FAILS:
                        fails.append(p)
                        continue
                    row = []
                    for ell in LS:
                        xs_e_xs = float((Xs @ expm(ell * M) @ Xs.T)[0, 0])
                        for sig in SS:
                            try:
                                f = ogp.gp_fit_predict(X, Xs, y[:, None], M, ell, sig)
                                f["prior_var"] = f["sigma_f"] * (xs_e_xs + sig)
                                row.append(f if np.isfinite(f["nlml"]) else None)
                            except (np.linalg.LinAlgError, ValueError, OverflowError):
                                row.append(None)
                    fits[p] = row
    return fits, fails


def test_grid_fmean_fvar_match_oracle(marg_small, oracle_fits):
    """The grid records' fmean / fvar (what the marginal consumes) against the oracle's fit at every grid point of one
    problem per script configuration, within the conditioning-aware bound of the plain sweep's parity test (gp_tol with
    cond(K)).  The scale includes the prior standard deviation: fvar = prior_var - v^T v cancels at the ill-conditioned
    grid corners, so its rounding is relative to prior_var, not to the (small) result; fmean = k*^T K^-1 y likewise."""
    _, sw, _, _, _, grid = marg_small
    fits, _ = oracle_fits
    for ci, cfg in enumerate(sw.cfgs):
        p = next(p for p in sorted(fits) if sw.plan.prob_meta[p][0] == ci)
        g = grid[p].reshape(-1)
        n_cmp = 0
        for kk, f in enumerate(fits[p]):
            if f is None or g["info"][kk] != 0 or not np.isfinite(g["nlml"][kk]):
                continue
            t = gp_tol(g[kk], f["cond"])
            rf, rv = f["fmean"], f["fvar"]
            scale = max(abs(rf), np.sqrt(abs(rv)), np.sqrt(abs(f["prior_var"])))
            assert abs(g["fmean"][kk] - rf) <= t * scale, (cfg.name, p, kk, g["fmean"][kk], rf, t)
            assert abs(g["fvar"][kk] - rv) <= t * max(abs(rv), scale ** 2), (cfg.name, p, kk, g["fvar"][kk], rv, t)
            n_cmp += 1
        assert n_cmp >= 100, (cfg.name, p, n_cmp)
        print(f"{cfg.name}: problem {p}, {n_cmp} grid points checked against the oracle")


def test_marginal_matches_oracle_fits(marg_small, oracle_fits):
    """The device's marginal against the oracle's marginal built from oracle fits at all 400 points.

    Bound (first order).  Per grid point the device is within d_mu_k = t_k s_k of the oracle's mean, d_v_k =
    t_k max(|v_k|, s_k^2) of its variance and d_k = t_k max(1, |nlml_k|) of its nlML (gp_tol t_k with cond(K), s_k =
    max(|mu_k|, sqrt|v_k|, prior sd_k) as in test_grid_fmean_fvar_match_oracle).  With D = max_k d_k, log w_k = -nlml_k - logsumexp(-nlml) moves by at most 2D, so
    |dw_k| <= 2D w_k, and since sum dw = 0:
        |d fmean| <= sum w |d_mu| + 2D sum w |mu - fmean|
        |d fvar|  <= sum w |d_v| + 2 sum w |mu - fmean| (|d_mu| + |d fmean|) + 2D sum w |v + (mu - fmean)^2 - fvar|
        |d nlml|  <= D (a weighted mean of the d_k).
    Points admissible on one side only carry weight W_x (device weights for device-only points, oracle weights for
    oracle-only ones); they add W_x max|mu - fmean| (mean) and W_x max|v + (mu - fmean)^2 - fvar| (variance), doubled
    for the renormalisation.  The bounds are applied with a factor 4 for the dropped second-order terms."""
    from oracle import marginal as om
    _, sw, _, raw, marg, grid = marg_small
    fits, fails = oracle_fits
    for p in fails:
        assert marg["n_admissible"][p] == 0 and raw["info"][p] == -1 and np.isnan(raw["fmean"][p]), p
    worst = 0.0
    for p, row in fits.items():
        g = grid[p].reshape(-1)
        dev_adm = (g["info"] == 0) & np.isfinite(g["nlml"])
        orc_adm = np.array([f is not None for f in row])
        both = dev_adm & orc_adm
        assert both.any(), p
        mu = np.array([f["fmean"] if f is not None else 0.0 for f in row])
        v = np.array([f["fvar"] if f is not None else 0.0 for f in row])
        nl = np.array([f["nlml"] if f is not None else np.inf for f in row])
        o = om.marginal(mu, v, nl, np.where(orc_adm, 0, 1), ())
        ob = om.marginal(mu, v, nl, np.where(both, 0, 1), ())
        t = np.array([gp_tol(g[k], row[k]["cond"]) if both[k] else 0.0 for k in range(len(row))])
        pv = np.array([f["prior_var"] if f is not None else 0.0 for f in row])
        s = np.maximum(np.maximum(np.abs(mu), np.sqrt(np.abs(v))), np.sqrt(np.abs(pv)))
        d_mu, d_v = t * s, t * np.maximum(np.abs(v), s ** 2)
        D = float(np.max(t * np.maximum(1.0, np.abs(nl)), where=both, initial=0.0))
        w = ob["w"]
        dev_w = om.weights(g["nlml"], g["info"])[0]
        W_x = float(dev_w[dev_adm & ~orc_adm].sum() + o["w"][orc_adm & ~dev_adm].sum())
        cen = np.where(both | orc_adm, mu - o["fmean"], 0.0)
        spread = np.abs(np.where(both | orc_adm, v + cen ** 2 - o["fvar"], 0.0))
        b_mean = np.sum(w * d_mu) + 2 * D * np.sum(w * np.abs(cen)) + 2 * W_x * np.max(np.abs(cen))
        b_var = np.sum(w * d_v) + 2 * np.sum(w * np.abs(cen) * (d_mu + b_mean)) + 2 * D * np.sum(w * spread) + \
            2 * W_x * np.max(spread)
        b_nl = D + 2 * W_x + 1e-13 * max(1.0, abs(o["nlml"]))
        err = (abs(raw["fmean"][p] - o["fmean"]), abs(raw["fvar"][p] - o["fvar"]), abs(raw["nlml"][p] - o["nlml"]))
        assert err[0] <= 4 * b_mean + 1e-15, (p, err, b_mean, D, W_x)
        assert err[1] <= 4 * b_var + 1e-15, (p, err, b_var, D, W_x)
        assert err[2] <= 4 * b_nl, (p, err, b_nl, D, W_x)
        worst = max(worst, err[0] / max(4 * b_mean, 1e-300))
    assert len(fits) >= 30
    print(f"marginal vs oracle fits: {len(fits)} problems, worst mean error / bound {worst:.3g}")


def test_marginal_outputs_do_not_depend_on_the_schedule(marg_small):
    """waves = 0 (one stream), waves = 1, the multi-wave default, run_many and CUDA-graph replay: the same bits."""
    _, _, _, raw, marg, grid = marg_small
    sw = marginal_sweep(small_inputs())
    sw.upload()
    results = []
    for waves in (0, 1, None):
        sw.compute(waves=waves)
        results.append((sw.download().copy(), sw.marginal.copy(), sw.grid_records()))
    outs = list(sw.run_many(2))
    results.append((sw.raw.copy(), sw.marginal.copy(), sw.grid_records()))
    sw.use_graph = True
    outs += list(sw.run_many(2))
    results.append((sw.raw.copy(), sw.marginal.copy(), sw.grid_records()))
    for r, m, gr in results:
        for f in FIELDS:
            assert np.array_equal(r[f], raw[f], equal_nan=True), f
        assert m.tobytes() == marg.tobytes()
        for f in FIELDS:
            assert np.array_equal(gr[f], grid[f], equal_nan=True), f
    for o in outs[1:]:
        for c in outs[0]:
            for k, v in outs[0][c].items():
                assert np.array_equal(o[c][k], v, equal_nan=True), (c, k)
    assert sw.kernel_launches() > 0 and sw.d2h_bytes() == sw.P * (80 + 24 + 8 * len(LEVELS))


def test_load_inputs_streams_a_new_member(lib_built):
    """A marginal sweep built for member 0 and fed member 1 through load_inputs == one constructed on member 1."""
    w0, w1 = small_inputs(0), small_inputs(1)
    a = marginal_sweep(w0)
    a.run()
    a.load_inputs(w1["sic"], w1["sst"])
    out_a = a.run()
    b = marginal_sweep(w1)
    out_b = b.run()
    for f in FIELDS:
        assert np.array_equal(a.raw[f], b.raw[f], equal_nan=True), f
    assert a.marginal.tobytes() == b.marginal.tobytes()
    for c in out_b:
        for k, v in out_b[c].items():
            assert np.array_equal(out_a[c][k], v, equal_nan=True), (c, k)


def test_constructor_rejects_inconsistent_modes(lib_built):
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    w = small_inputs()
    args = (NORTH_INITS, w["sic"], w["sie"], FMIN, FMAX, w["psar"], w["sst"], w["lat"])
    for kw in (dict(hyper_mode="marginal"), dict(hyper_grid=(LS, SS), quantiles=(0.5,)),
               dict(hyper_grid=(LS, SS), hyper_mode="marginal", quantiles=(0.0, 0.5)),
               dict(hyper_grid=(LS, SS), hyper_mode="mean")):
        with pytest.raises(ValueError):
            RetrospectiveSweep(*args, **kw)


def test_marginal_forecast_single_problem(lib_built):
    """forecast.marginal_forecast == the device marginal of forecast.hyper_grid's records."""
    from seaiceextentforecasting_b200 import synthetic as syn
    from seaiceextentforecasting_b200.forecast import detrend, hyper_grid, marginal_forecast, networks
    data, _ = syn.make_field(16, 16, 30, seed=5)
    dt, _ = detrend(data)
    _, anoms = networks(dt, area=syn.make_psar(16, 16), latlon=False)
    y = np.random.default_rng(3).standard_normal(29)
    rec, stats, q = marginal_forecast(y, anoms, rule=1, quantiles=(0.1, 0.9))
    grid, _ = hyper_grid(y, anoms, rule=1)
    raw, st, qq = run_marginal(grid.reshape(1, -1), levels=(0.1, 0.9))
    for f in FIELDS:                                               # (the cycle counters differ between launches)
        assert np.array_equal(rec[f], raw[f][0], equal_nan=True), f
    assert stats.tobytes() == st[0].tobytes() and np.array_equal(q, qq[0], equal_nan=True)
    if stats["n_admissible"] > 0:
        assert q[0] < rec["fmean"] < q[1]


def test_full_size_marginal_step_invariants(lib_built):
    """The bench's 8-member north step (bench.make_workload): every problem the plain sweep solves has an admissible
    grid point, m <= nlml <= m + log|A|, 1 <= ESS <= |A|, and the quantiles increase with the level."""
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
    sw = RetrospectiveSweep(*args, hyper_grid=(LS, SS), hyper_mode="marginal", quantiles=LEVELS)
    out = sw.run()
    assert len(out) == 8 and len(sw.raw) == 8 * 432
    marg, grid = sw.marginal, sw.grid_records()
    nA = marg["n_admissible"]
    assert (nA[raw_plain["info"] == 0] >= 1).all()
    ok = nA >= 1
    nl = np.where((grid["info"] == 0) & np.isfinite(grid["nlml"]), grid["nlml"], np.inf).reshape(sw.P, -1)
    m = nl.min(axis=1)[ok]
    tol = 1e-12 * np.maximum(1.0, np.abs(m))
    r = sw.raw["nlml"][ok]
    assert np.all(r >= m - tol) and np.all(r <= m + np.log(nA[ok]) + tol)
    ess = marg["ess"][ok]
    assert np.all(ess >= 1.0 - 1e-12) and np.all(ess <= nA[ok] * (1 + 1e-12))
    assert np.all(np.diff(marg["quantiles"][ok], axis=1) >= 0)
    assert np.isfinite(sw.raw["fmean"][ok]).all() and np.isfinite(sw.raw["fvar"][ok]).all()
    print(f"full size: {ok.sum()} of {sw.P} problems marginalised, ESS median {np.median(ess):.2f}, "
          f"max {ess.max():.1f}; w_max median {np.median(marg['w_max'][ok]):.3f}")
