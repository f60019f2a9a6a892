"""GPU parity: batched GP kernel (K7-K9) vs the oracle's numpy/scipy restatement of forecast()/MLII().
Tolerance: 1e-9 relative (north_star), widened only by the documented conditioning terms:
  * expm with s squarings amplifies rounding by ~2^s (SURVEY.md H3; scipy itself moves this much under a
    1-ulp input perturbation, see tests/test_expm_spec.py) -> 64*2^s*2^-53
  * two backward-stable Cholesky solves differ by ~cond(K)*2^-53 (SURVEY.md H4)."""
import zlib

import numpy as np
import pytest

from seaiceextentforecasting_b200.config import CONFIGS, RULE_ALL, RULE_POS, RULE_POS_SIG

pytestmark = pytest.mark.gpu


def make_problem(seed, n, nA, nS=0, scale=1.0):
    rng = np.random.default_rng(seed)
    common = rng.standard_normal((3, n + 1))
    sic = {}
    for a in range(nA):
        w = rng.standard_normal(3) * 0.8
        sic[a * 2 + 1] = scale * (w @ common + rng.standard_normal(n + 1))
    sst = None
    if nS:
        sst = {a: 0.1 * (rng.standard_normal(3) @ common + rng.standard_normal(n + 1)) for a in range(nS)}
    y = np.round(0.3 * (common[0, :n] - common[1, :n]) + 0.2 * rng.standard_normal(n), 3)
    return y, sic, sst


def oracle_forecast(y, sic, sst, rule, alpha, zscore, ell, sig):
    from oracle import gp as og
    Xfull = og.select_predictors(y, sic, sst, {RULE_POS: "pos", RULE_ALL: "all", RULE_POS_SIG: "pos_sig"}[rule], alpha)
    X, Xs, M = og.design(Xfull, zscore)
    out = og.gp_fit_predict(X, Xs, y[:, None], M, ell, sig)
    n = len(y)
    from scipy.linalg import expm
    K = out["sigma_f"] * (X @ expm(ell * M) @ X.T + sig * np.eye(n))
    out["cond"] = np.linalg.cond(K)
    out["n_pred"] = Xfull.shape[1]
    out["X"], out["M"] = X, M
    return out


def tol(res, cond):
    return max(1e-9, 64.0 * 2.0 ** int(res["expm_s"]) * 2.0 ** -53, 8.0 * cond * 2.0 ** -53)


CASES = []
for name, cfg in CONFIGS.items():
    for k in range(3):
        CASES.append((name, k))


@pytest.mark.parametrize("name,k", CASES)
@pytest.mark.parametrize("n", [6, 20, 41])
def test_forecast_matches_oracle(lib_built, name, k, n):
    from seaiceextentforecasting_b200.forecast import forecast
    cfg = CONFIGS[name]
    # raw (un-z-scored) node series are sums over ~30 cells x sqrt(1e4): O(1e2..1e3); crc32, not hash(): str hashes
    # change from process to process, and a failing case must be reproducible
    seed = zlib.crc32(f"{name},{k},{n}".encode()) % 10000
    y, sic, sst = make_problem(seed, n, nA=12 + 2 * k, nS=6 if cfg.use_sst else 0,
                               scale=1.0 if cfg.zscore else 30.0)
    r = forecast(y, sic, sst, rule=cfg.rule[k], alpha=cfg.alpha, zscore=cfg.zscore, ell=cfg.ell[k], sig=cfg.sig[k])
    try:
        o = oracle_forecast(y, sic, sst, cfg.rule[k], cfg.alpha, cfg.zscore, cfg.ell[k], cfg.sig[k])
    except (np.linalg.LinAlgError, IndexError, ValueError):
        assert r["info"] != 0
        return
    assert r["info"] == 0
    assert r["n_pred"] == o["n_pred"]                      # identical predictor selection
    t = tol(r, o["cond"])
    scale = max(abs(o["fmean"]), np.sqrt(abs(o["fvar"])), 1e-3)
    assert abs(r["fmean"] - o["fmean"]) <= t * scale, (r["fmean"], o["fmean"], t)
    assert abs(r["fvar"] - o["fvar"]) <= t * max(abs(o["fvar"]), scale ** 2)
    assert abs(r["sigma_f"] - o["sigma_f"]) <= t * abs(o["sigma_f"])
    assert abs(r["nlml"] - o["nlml"]) <= t * max(1.0, abs(o["nlml"]))


@pytest.mark.parametrize("seed", range(6))
def test_mlii_matches_oracle(lib_built, seed):
    from oracle import gp as og
    from seaiceextentforecasting_b200.forecast import mlii
    n = [8, 15, 22, 30, 41, 12][seed]
    y, sic, _ = make_problem(100 + seed, n, nA=10)
    theta = np.log([np.logspace(-7, 2, 20)[8 + seed], np.logspace(-3, 9, 20)[2 + seed]])
    nl, g = mlii(theta, y, sic, rule=RULE_POS, zscore=True)
    Xfull = og.select_predictors(y, sic, None, "pos")
    X, Xs, M = og.design(Xfull, True)
    onl, og_ = og.mlii(theta, X, y[:, None], M)
    assert abs(nl - onl) <= 1e-9 * max(1.0, abs(onl))
    np.testing.assert_allclose(g, og_, rtol=1e-7, atol=1e-9 * max(1.0, np.abs(og_).max()))


import glob
import os

_GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_SWEEPS = sorted(glob.glob(os.path.join(_GOLD, "sweep_*.npz")))


@pytest.mark.parametrize("path", _SWEEPS, ids=[os.path.basename(p) for p in _SWEEPS])
def test_mlii_matches_reference_golden(lib_built, path):
    """The device `MLII` against the value and gradient the UNMODIFIED reference scripts' nested MLII() returned for the
    last target year of each golden sweep (tests/golden/make_golden.py lifts it out of the seven retrospective scripts):
    the problem is rebuilt exactly like tests/test_oracle_golden.py::test_mlii_oracle_equals_reference does."""
    from oracle import gp as ogp
    from oracle import sweep as osweep
    from seaiceextentforecasting_b200.forecast import forecast, mlii
    g = np.load(path)
    name = os.path.basename(path)[len("sweep_"):-len(".npz")]
    cfg = CONFIGS[name]
    fmin, fmax = int(g["fmin"]), int(g["fmax"])
    year = fmax
    ny = year - 1 if cfg.prev_year_network else year
    _, anoms, _ = osweep.build_network(g["sic"], ny, False, g["psar"])
    sst_anoms = None
    if cfg.use_sst:
        _, sst_anoms, _ = osweep.build_network(g["sst"], year, True, g["sst_lat"])
    row = year - (fmin - 1) - 1
    sdt = g["siedt_" + cfg.regions[0]]
    y = sdt[row, 1:year - 1979] if cfg.prev_year_network else sdt[row, 0:year - 1979]
    theta = np.asarray(g["mlii_theta"], dtype=np.float64)
    nl, grad = mlii(theta, y, anoms, sst_anoms, rule=cfg.rule[0], alpha=cfg.alpha, zscore=cfg.zscore)
    ref_nl, ref_grad = float(g["mlii_nl"]), np.asarray(g["mlii_grad"], dtype=np.float64)
    if not np.isfinite(ref_nl):
        assert nl == np.inf and np.isinf(grad).all()
        return
    # conditioning of this problem (same widening terms as the forecasts, module docstring)
    rec = forecast(y, anoms, sst_anoms, rule=cfg.rule[0], alpha=cfg.alpha, zscore=cfg.zscore, ell=float(np.exp(theta[0])),
                   sig=float(np.exp(theta[1])))
    rule = {RULE_POS: "pos", RULE_ALL: "all", RULE_POS_SIG: "pos_sig"}[cfg.rule[0]]
    X, Xs, M = ogp.design(ogp.select_predictors(y, anoms, sst_anoms, rule, cfg.alpha), cfg.zscore)
    from scipy.linalg import expm
    K = X @ expm(float(np.exp(theta[0])) * M) @ X.T + float(np.exp(theta[1])) * np.eye(len(y))
    t = tol(rec, np.linalg.cond(K))
    n = len(y)
    assert abs(nl - ref_nl) <= t * max(1.0, abs(ref_nl), 1.5 * n), (nl, ref_nl, t)
    # each gradient component is trace(K^-1 dK)/2 - a^T dK a/2 (north/June1st.py:248-252): a difference of two terms that
    # are larger than the result, and dK/dl = X (M Sigma) X^T + sn I is itself a product with heavy cancellation (M has
    # zero column sums, ||M||_1 ~ 1e6, |X| ~ 1e3 on these inputs).  The bound is the conditioning-aware one, relative to
    # the sum of the two terms' magnitudes, or -- where the reference's OWN result is less stable than that -- four
    # times the spread of the reference formula under 1-ulp relative perturbations of M (its own sensitivity, the
    # argument tests/test_expm_spec.py makes for expm).
    yv = np.asarray(y, dtype=np.float64)[:, None]
    ell_v, sig_v = float(np.exp(theta[0])), float(np.exp(theta[1]))
    St = expm(ell_v * M)
    Lt = np.linalg.cholesky(X @ St @ X.T + np.eye(n) * sig_v)
    sf = float((yv.T @ np.linalg.solve(Lt.T, np.linalg.solve(Lt, yv)))[0, 0] / n)
    S = sf * St
    Kf = X @ S @ X.T + np.eye(n) * sf * sig_v
    a = np.linalg.solve(Kf, yv)
    rng = np.random.default_rng(0)
    pert = np.array([ogp.mlii(theta, X, yv, M * (1.0 + 2.0 ** -52 * rng.standard_normal(M.shape)))[1] for _ in range(6)])
    spread = np.abs(pert - ref_grad[None, :]).max(axis=0)
    for gi, dK in enumerate((X @ (M @ S) @ X.T + np.eye(n) * sf * sig_v, X @ S @ X.T + np.eye(n) * sf)):
        mag = abs(np.trace(np.linalg.solve(Kf, dK))) / 2 + abs(float((a.T @ dK @ a)[0, 0])) / 2
        bound = max(1e-7 * abs(ref_grad[gi]), t * max(1.0, mag), 4.0 * spread[gi])
        assert abs(grad[gi] - ref_grad[gi]) <= bound, (gi, grad, ref_grad, t, mag, spread)


def test_not_spd_reports_like_reference(lib_built):
    """sigma_n~ = 0 with more rows than predictors: K is singular -> LinAlgError in forecast(), inf in MLII."""
    from seaiceextentforecasting_b200.forecast import forecast, mlii
    y, sic, _ = make_problem(5, 30, nA=3)
    r = forecast(y, sic, None, rule=RULE_ALL, ell=1e-3, sig=0.0)
    assert r["info"] > 0 or not np.isfinite(r["fmean"])
    # MLII's `except` branch (north/June1st.py:254-256): a non-SPD kernel matrix gives (inf, [inf, inf])
    nl, g = mlii(np.array([np.log(1e-3), -800.0]), y, sic, rule=RULE_ALL)
    from oracle import gp as og
    Xfull = og.select_predictors(y, sic, None, "all")
    X, Xs, M = og.design(Xfull, False)
    onl, ograd = og.mlii(np.array([np.log(1e-3), -800.0]), X, y[:, None], M)
    if np.isinf(onl):
        assert r["info"] > 0 and nl == np.inf and np.isinf(g).all()
    else:                                   # LAPACK got through the factorisation of the singular matrix: compare
        assert np.isfinite(nl) == np.isfinite(onl)


def test_constant_series_is_rejected_like_pearsonr_nan(lib_built):
    """A constant node series has Pearson r = NaN (scipy returns nan with a warning); `r > 0` is then False and the
    reference does not select it.  CUDA fmin/fmax would turn the NaN into +1 (ADVICE round 1)."""
    import warnings
    from seaiceextentforecasting_b200.forecast import forecast
    y, sic, _ = make_problem(11, 20, nA=8)
    sic[999] = np.full(21, 3.25)                       # constant series, appended last (dict order = column order)
    r = forecast(y, sic, None, rule=RULE_POS, zscore=False, ell=1e-2, sig=1.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = oracle_forecast(y, sic, None, RULE_POS, 0.05, False, 1e-2, 1.0)
    assert r["info"] == 0 and r["n_pred"] == o["n_pred"]
    assert abs(r["fmean"] - o["fmean"]) <= tol(r, o["cond"]) * max(abs(o["fmean"]), np.sqrt(abs(o["fvar"])))


@pytest.mark.parametrize("seed,zscore", [(0, True), (1, True), (2, False)])
def test_cg_refinement_matches_scipy_on_the_oracle(lib_built, seed, zscore):
    """SURVEY.md 8(f)-3: `minimize(MLII, x0=log(l_init, sigma_init), method='CG', jac=True)` (north/June1st.py:259-262,
    commented out in the reference) with MLII and its gradient on the device, against the same scipy call on the oracle's
    MLII.  The gradient "as written" in the reference is not the exact derivative of nlML, so scipy's CG stops with
    "precision loss" and its end point moves by ~5e-7 in nlML / ~4e-6 in theta under 1e-7-relative perturbations of the
    gradient (measured on the oracle): the comparison allows 2e-5 / 1e-4."""
    from oracle import gp as og
    from scipy.optimize import minimize
    from seaiceextentforecasting_b200.forecast import optimise_hyperparameters
    n = [20, 30, 41][seed]
    y, sic, _ = make_problem(300 + seed, n, nA=10, scale=1.0 if zscore else 5.0)
    ell0, sig0 = np.logspace(-7, 2, 20)[12], np.logspace(-3, 9, 20)[4]
    ell, sig, res = optimise_hyperparameters(y, sic, None, rule=RULE_POS, zscore=zscore, ell0=ell0, sig0=sig0)
    Xfull = og.select_predictors(y, sic, None, "pos")
    X, Xs, M = og.design(Xfull, zscore)
    ref = minimize(lambda th: og.mlii(th, X, y[:, None], M), x0=[np.log(ell0), np.log(sig0)], method="CG", jac=True,
                   options={"disp": False})
    assert np.isfinite(res.fun) and res.evaluations >= 2
    assert abs(res.fun - ref.fun) <= 2e-5 * max(1.0, abs(ref.fun)), (res.fun, ref.fun)
    assert np.abs(res.x - ref.x).max() <= 1e-4 * max(1.0, np.abs(ref.x).max()), (res.x, ref.x)
    v_ours_on_oracle, _ = og.mlii(res.x, X, y[:, None], M)          # our minimiser, judged by the oracle's objective
    assert abs(v_ours_on_oracle - ref.fun) <= 2e-5 * max(1.0, abs(ref.fun))
    assert abs(ell - np.exp(res.x[0])) <= 1e-12 * ell and abs(sig - np.exp(res.x[1])) <= 1e-12 * sig


@pytest.mark.parametrize("name,k", [("north_june", 0), ("north_august", 1), ("south_february", 2)])
def test_hyper_grid_matches_oracle(lib_built, name, k):
    """sie_gp_hyper_grid: the 20 x 20 (l, sigma_n~) grid of north/June1st.py:210-211, one expm per l, against MLII()
    of the oracle evaluated pair by pair (value and, for the June case, the gradient as written)."""
    from oracle import gp as og
    from seaiceextentforecasting_b200.forecast import hyper_grid
    cfg = CONFIGS[name]
    n = 20
    y, sic, sst = make_problem(77 + k, n, nA=10, nS=4 if cfg.use_sst else 0, scale=1.0 if cfg.zscore else 30.0)
    ells, sigs = np.logspace(-7, 2, 20), np.logspace(-3, 9, 20)
    want_grad = name == "north_june"
    rec, best = hyper_grid(y, sic, sst, rule=cfg.rule[k], alpha=cfg.alpha, zscore=cfg.zscore, ells=ells, sigs=sigs,
                           want_grad=want_grad)
    assert rec.shape == (20, 20)
    Xfull = og.select_predictors(y, sic, sst, {RULE_POS: "pos", RULE_ALL: "all", RULE_POS_SIG: "pos_sig"}[cfg.rule[k]],
                                 cfg.alpha)
    X, Xs, M = og.design(Xfull, cfg.zscore)
    from scipy.linalg import expm
    ref = np.full((20, 20), np.inf)
    checked = 0
    for i, ell in enumerate(ells):
        E = expm(ell * M)
        for j, sig in enumerate(sigs):
            val, grad = og.mlii(np.log([ell, sig]), X, y[:, None], M)
            r = rec[i, j]
            if not np.isfinite(val):
                assert r["info"] != 0
                continue
            ref[i, j] = val
            assert r["info"] == 0 and r["n_pred"] == Xfull.shape[1]
            sf = r["sigma_f"]
            cond = np.linalg.cond(sf * (X @ E @ X.T + sig * np.eye(n)))
            t = tol(r, cond)
            assert abs(r["nlml"] - val) <= t * max(1.0, abs(val)), (i, j, r["nlml"], val, t)
            if want_grad and cond < 1e8:
                assert abs(r["g_ell"] - grad[0]) <= 10 * t * max(1.0, abs(grad[0])), (i, j, r["g_ell"], grad[0])
                assert abs(r["g_sig"] - grad[1]) <= 10 * t * max(1.0, abs(grad[1])), (i, j, r["g_sig"], grad[1])
            checked += 1
    assert checked > 300
    # the grid minimum agrees wherever it is not a numerical tie
    ob = np.unravel_index(int(np.argmin(ref)), ref.shape)
    assert abs(ref[best] - ref[ob]) <= 1e-9 * max(1.0, abs(ref[ob]))
