"""Host side of ensemble forecasts (no GPU): the oracle's two-level pool against the grid marginal and the flattened
mixture, the (ensemble problem, member slot) mapping of streamed batches, the ensemble keys of the assembled GPR dict,
the SieGpEnsemble layout and the C ABI's argument checks."""
import ctypes

import numpy as np
import pytest

from oracle import ensemble as oe
from oracle import marginal as om
from seaiceextentforecasting_b200.config import CONFIGS, NORTH_INITS
from seaiceextentforecasting_b200.forecast import GP_ENSEMBLE_DTYPE, SweepPlan, ensemble_records, ensemble_slots

LEVELS = (0.05, 0.5, 0.95)


def _records(seed, M, n, bad=0.1):
    rng = np.random.default_rng(seed)
    fmean = rng.normal(0.0, 0.3, (M, n))
    fvar = rng.uniform(0.01, 0.2, (M, n))
    nlml = rng.uniform(-5.0, 5.0, (M, n))
    info = np.where(rng.uniform(size=(M, n)) < bad, 3, 0)
    return fmean, fvar, nlml, info


def test_one_member_is_its_grid_marginal():
    fmean, fvar, nlml, info = _records(1, 1, 400)
    r = oe.ensemble(fmean, fvar, nlml, info, LEVELS)
    m = om.marginal(fmean[0], fvar[0], nlml[0], info[0], LEVELS)
    assert r["n_members"] == 1 and r["fmean"] == m["fmean"] and r["var_within"] == m["fvar"]
    assert r["var_between"] == 0.0 and r["fvar"] == m["fvar"]
    assert np.array_equal(r["quantiles"], m["quantiles"])


def test_gaussian_members_pool_to_the_flattened_mixture():
    """n_grid = 1: the two-level moments are the moments of the equal-weight mixture of the members' Gaussians."""
    for seed in range(5):
        fmean, fvar, nlml, info = _records(10 + seed, 64, 1, bad=0.2)
        r = oe.ensemble(fmean, fvar, nlml, info, LEVELS)
        ok = info[:, 0] == 0
        mu, v = fmean[ok, 0], fvar[ok, 0]
        w = np.full(ok.sum(), 1.0 / ok.sum())
        mean = np.sum(w * mu)
        var = np.sum(w * (v + (mu - mean) ** 2))
        assert r["n_members"] == ok.sum()
        assert abs(r["fmean"] - mean) <= 1e-15 * max(1.0, abs(mean))
        assert abs(r["fvar"] - var) <= 1e-15 * max(1.0, var)
        assert np.array_equal(r["quantiles"], [om.mixture_quantile(t, w, mu, v) for t in LEVELS])


def test_members_without_a_forecast_do_not_count():
    fmean, fvar, nlml, info = _records(3, 6, 20)
    info[[1, 4]] = 1                                          # members 1 and 4: no admissible record
    r = oe.ensemble(fmean, fvar, nlml, info, LEVELS)
    keep = [0, 2, 3, 5]
    s = oe.ensemble(fmean[keep], fvar[keep], nlml[keep], info[keep], LEVELS)
    assert r["n_members"] == 4
    for k in ("fmean", "fvar", "var_within", "var_between"):
        assert r[k] == s[k], k
    assert np.array_equal(r["quantiles"], s["quantiles"])
    assert np.isnan(r["member_mean"][[1, 4]]).all() and (r["w"][[1, 4]] == 0).all()
    assert np.isclose(r["w"].sum(), 1.0, rtol=1e-14)
    info[:] = 2
    none = oe.ensemble(fmean, fvar, nlml, info, LEVELS)
    assert none["n_members"] == 0 and np.isnan(none["fmean"]) and np.isnan(none["quantiles"]).all()


def _sie():
    rng = np.random.default_rng(0)
    return {r: 10 + rng.standard_normal(42) for r in CONFIGS["north_june"].regions}


@pytest.mark.parametrize("members", [2, 4])
def test_streamed_batches_fill_every_slot_once(members):
    """Batches of `members` members at first_member = 0, members, 2 * members, ... of a 3-batch ensemble hit every
    (ensemble problem, slot) pair exactly once, and every problem's row names its own (config, region, year) and member;
    also after partition_sst permuted the problems."""
    for permute in (False, True):
        plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, members=members)
        if permute:
            before = list(plan.prob_meta)
            plan.partition_sst([(0, plan.P // 2), (plan.P // 2, plan.P)])
            assert plan.prob_meta != before
        n_members = 3 * members
        meta, rows = ensemble_slots(plan, n_members)
        ncell = sum(len(c.regions) for c in plan.cfgs) * len(plan.years)
        assert meta.shape == (ncell, 3) and rows.shape == (plan.P,)
        hits = np.zeros(len(meta) * n_members, dtype=int)
        for first in range(0, n_members, members):
            np.add.at(hits, rows + first, 1)
        assert (hits == 1).all()
        for p, (m, mb) in enumerate(zip(plan.prob_meta, plan.prob_member)):
            e, slot = divmod(int(rows[p]), n_members)
            assert tuple(meta[e]) == tuple(m) and slot == mb


def test_assemble_with_ensemble_adds_the_pool_keys():
    plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020)
    meta, _ = ensemble_slots(plan, 1)
    E = len(meta)
    pooled = np.zeros(E, dtype=GP_ENSEMBLE_DTYPE)
    pooled["fmean"] = np.arange(E) * 0.01
    pooled["var_within"] = 0.1 + np.arange(E) * 1e-3
    pooled["var_between"] = 0.02
    pooled["fvar"] = pooled["var_within"] + pooled["var_between"]
    pooled["n_members"] = np.arange(E) % 5
    quant = pooled["fmean"][:, None] + np.array([-0.3, 0.0, 0.3])
    rec = ensemble_records(pooled, quant)
    out = plan._assemble_one(rec, meta, ensemble=rec)
    plain = plan._assemble_one(pooled, meta)
    for ci, cfg in enumerate(plan.cfgs):
        g = out[cfg.name]
        for k, v in plain[cfg.name].items():
            assert np.array_equal(g[k], v, equal_nan=True), k
        assert set(g) - set(plain[cfg.name]) == {reg + s for reg in cfg.regions for s in (
            "_var_within", "_var_between", "_n_members", "_quantiles", "_quantiles_rt")}
        for k, reg in enumerate(cfg.regions):
            e = [int(np.nonzero((meta == (ci, k, y)).all(axis=1))[0][0]) for y in plan.years]
            assert np.array_equal(g[reg + "_raw_fmean"], pooled["fmean"][e])
            assert np.array_equal(g[reg + "_var_within"], pooled["var_within"][e])
            assert np.array_equal(g[reg + "_n_members"], pooled["n_members"][e])
            assert np.array_equal(g[reg + "_quantiles"], quant[e])
            line = g[reg + "_raw_fmean_rt"] - g[reg + "_raw_fmean"]
            assert np.allclose(g[reg + "_quantiles_rt"], quant[e] + line[:, None], rtol=1e-13, atol=0)
    assert plan.skill(out) == plan.skill(plain)                       # skill() reads an ensemble dict unchanged
    assert ensemble_records(pooled, np.zeros(0))["quantiles"].shape == (E, 0)


def test_gp_ensemble_layout_matches_the_header():
    from seaiceextentforecasting_b200 import _lib
    assert ctypes.sizeof(_lib.SieGpEnsemble) == 40 == GP_ENSEMBLE_DTYPE.itemsize
    for (name, _), f in zip(_lib.SieGpEnsemble._fields_, GP_ENSEMBLE_DTYPE.names):
        assert name == f and getattr(_lib.SieGpEnsemble, name).offset == GP_ENSEMBLE_DTYPE.fields[f][1]


def test_gp_ensemble_rejects_bad_arguments(lib_built):
    """Checked before anything is enqueued, so no device is needed."""
    from seaiceextentforecasting_b200 import _lib
    lib = _lib.load()
    buf = (ctypes.c_double * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    null = ctypes.c_void_p(0)
    need = lib.sie_gp_ensemble_scratch_bytes(4, 8, 400)
    assert need == 4 * 8 * 400 * 24 and lib.sie_gp_ensemble_scratch_bytes(0, 8, 400) == 0
    args = [p, 4, 8, 400, p, 3, p, p, p, need, null]
    for i in (0, 4, 6, 7, 8):                                        # each device pointer NULL in turn
        bad = list(args)
        bad[i] = null
        assert lib.sie_gp_ensemble(*bad) == -1, i
    for i, v in ((1, 0), (2, -1), (3, 0), (5, -1), (9, need - 1)):   # E, M, n_grid < 1, n_q < 0, scratch too small
        bad = list(args)
        bad[i] = v
        assert lib.sie_gp_ensemble(*bad) == -1, (i, v)
    assert b"sie_gp_ensemble" in lib.sie_last_error()
    for M, n in ((1025, 1), (1024, 1 << 21)):                        # above the member limit, M * n_grid >= 2^31
        bad = list(args)
        bad[2], bad[3] = M, n
        assert lib.sie_gp_ensemble(*bad) == -3, (M, n)
        assert b"sie_gp_ensemble" in lib.sie_last_error()
