"""Host side of marginalised retrospective sweeps (no GPU): the oracle's grid marginal and its invariances, the
marginal keys of the assembled GPR dict, the multi-rank gather of the marginal records (world_size 2 over gloo), the
SieGpMarginal layout and the C ABI's argument checks."""
import ctypes
import os
import socket

import numpy as np
import pytest
from scipy.stats import norm

from oracle import marginal as om
from seaiceextentforecasting_b200.config import CONFIGS, NORTH_INITS
from seaiceextentforecasting_b200.forecast import (GP_MARGINAL_DTYPE, GP_RESULT_DTYPE, SweepPlan, check_levels,
                                                   marginal_dtype, marginal_records)

LEVELS = (0.05, 0.5, 0.95)


def _grid(seed, n=400, bad=40):
    rng = np.random.default_rng(seed)
    fmean = rng.normal(0.0, 0.3, n)
    fvar = rng.uniform(0.01, 0.2, n)
    nlml = rng.uniform(-5.0, 5.0, n)
    info = np.zeros(n, dtype=np.int32)
    info[rng.choice(n, bad, replace=False)] = 3
    nlml[rng.choice(n, bad // 2, replace=False)] = np.inf
    return fmean, fvar, nlml, info


def test_oracle_one_admissible_point_is_that_gaussian():
    fmean, fvar, nlml, info = _grid(1)
    info[:] = 1
    info[17], nlml[17] = 0, 2.5
    r = om.marginal(fmean, fvar, nlml, info, LEVELS)
    assert r["fmean"] == fmean[17] and r["fvar"] == fvar[17]
    assert r["nlml"] == 2.5 and r["ess"] == 1.0 and r["w_max"] == 1.0
    assert r["n_admissible"] == 1 and r["argmax"] == 17
    ppf = norm.ppf(LEVELS, loc=fmean[17], scale=np.sqrt(fvar[17]))
    assert np.allclose(r["quantiles"], ppf, rtol=0, atol=1e-12 * np.sqrt(fvar[17]) * 40)


def test_oracle_equal_nlml_gives_equal_weights():
    fmean, fvar, _, info = _grid(2, bad=0)
    r = om.marginal(fmean, fvar, np.full(400, 7.0), info, LEVELS)
    assert np.allclose(r["w"], 1 / 400, rtol=1e-14, atol=0)
    assert np.isclose(r["ess"], 400, rtol=1e-12) and np.isclose(r["w_max"], 1 / 400, rtol=1e-12)
    assert np.isclose(r["fmean"], fmean.mean(), rtol=1e-12, atol=1e-15)
    assert np.isclose(r["fvar"], fvar.mean() + fmean.var(), rtol=1e-12)
    assert np.isclose(r["nlml"], 7.0, rtol=1e-14) and r["argmax"] == 0


def test_oracle_ignores_inadmissible_points():
    fmean, fvar, nlml, info = _grid(3)
    r = om.marginal(fmean, fvar, nlml, info, LEVELS)
    adm = (info == 0) & np.isfinite(nlml)
    wild = fmean.copy()
    wild[~adm] = 1e6
    nl2 = nlml.copy()
    nl2[(info != 0) & np.isfinite(nlml)] = -1e3           # a tiny nlML on a failed point must not count
    r2 = om.marginal(wild, np.where(adm, fvar, -1.0), nl2, info, LEVELS)
    for k in ("fmean", "fvar", "nlml", "ess", "w_max", "n_admissible", "argmax"):
        assert r[k] == r2[k], k
    assert np.array_equal(r["quantiles"], r2["quantiles"])
    assert r["n_admissible"] == adm.sum() and (r["w"][~adm] == 0).all()
    empty = om.marginal(fmean, fvar, nlml, np.ones(400), LEVELS)
    assert empty["n_admissible"] == 0 and empty["argmax"] == -1 and np.isnan(empty["fmean"])
    assert np.isnan(empty["quantiles"]).all()


def test_oracle_is_invariant_to_a_constant_nlml_shift():
    fmean, fvar, nlml, info = _grid(4)
    r = om.marginal(fmean, fvar, nlml, info, LEVELS)
    for c in (-300.0, 0.125, 1e3):
        s = om.marginal(fmean, fvar, nlml + c, info, LEVELS)
        for k in ("fmean", "fvar", "ess", "w_max"):
            assert np.isclose(s[k], r[k], rtol=1e-12, atol=1e-15), (c, k)
        assert np.allclose(s["quantiles"], r["quantiles"], rtol=0, atol=1e-12)
        assert np.isclose(s["nlml"], r["nlml"] + c, rtol=1e-14, atol=1e-12), c
        assert s["argmax"] == r["argmax"] and s["n_admissible"] == r["n_admissible"]


def test_oracle_quantiles_invert_the_mixture_cdf():
    fmean, fvar, nlml, info = _grid(5)
    fvar[::7] = 0.0                                       # point masses
    r = om.marginal(fmean, fvar, nlml, info, LEVELS)
    q = r["quantiles"]
    assert np.all(np.diff(q) >= 0)
    mu, var = np.where(r["w"] > 0, fmean, 0), np.where(r["w"] > 0, fvar, 0)
    for t, x in zip(LEVELS, q):
        assert om.mixture_cdf(x, r["w"], mu, var) >= t > om.mixture_cdf(np.nextafter(x, -np.inf), r["w"], mu, var)


def test_gp_marginal_layout_matches_the_header():
    from seaiceextentforecasting_b200 import _lib
    assert ctypes.sizeof(_lib.SieGpMarginal) == 24 == GP_MARGINAL_DTYPE.itemsize
    for (name, _), f in zip(_lib.SieGpMarginal._fields_, GP_MARGINAL_DTYPE.names):
        assert name == f and getattr(_lib.SieGpMarginal, name).offset == GP_MARGINAL_DTYPE.fields[f][1]
    assert marginal_dtype(3).itemsize == 48 and marginal_dtype(0).itemsize == 24


def test_levels_are_checked():
    assert check_levels(LEVELS).tolist() == list(LEVELS)
    assert check_levels(()).size == 0
    for bad in ((0.0,), (1.0,), (0.5, 1.2), (-0.1,), (np.nan,)):
        with pytest.raises(ValueError):
            check_levels(bad)


def _sie():
    rng = np.random.default_rng(0)
    return {r: 10 + rng.standard_normal(42) for r in CONFIGS["north_june"].regions}


def _pid(m, ci, k, year):
    return m * 10000 + ci * 1000 + k * 100 + (year - 2000)


def _fake(plan, n_q=3):
    """Records whose values name their problem: fmean = id, ess = id + 0.5, w_max = 1 / (id + 1), argmax = id % 7 - 1,
    quantiles = id + (0, 0.1, 0.2, ...)."""
    raw = np.zeros(plan.P, dtype=GP_RESULT_DTYPE)
    stats = np.zeros(plan.P, dtype=GP_MARGINAL_DTYPE)
    quant = np.zeros((plan.P, n_q))
    for i, ((ci, k, year), m) in enumerate(zip(plan.prob_meta, plan.prob_member)):
        pid = _pid(m, ci, k, year)
        raw["fmean"][i] = pid
        stats[i] = (pid + 0.5, 1.0 / (pid + 1), 400, pid % 7 - 1)
        quant[i] = pid + 0.1 * np.arange(n_q)
    return raw, marginal_records(stats, quant)


def test_assemble_with_marginal_adds_the_posterior_keys():
    for members in (1, 2):
        plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, members=members)
        raw, marg = _fake(plan)
        plain, mixed = plan.assemble(raw), plan.assemble(raw, marginal=marg)
        plains, mixeds = (plain, mixed) if members > 1 else ([plain], [mixed])
        for m, (p, t) in enumerate(zip(plains, mixeds)):
            for ci, cfg in enumerate(plan.cfgs):
                for k, reg in enumerate(cfg.regions):
                    for key, v in p[cfg.name].items():               # the plain keys are untouched
                        assert np.array_equal(t[cfg.name][key], v, equal_nan=True)
                    pid = np.array([_pid(m, ci, k, y) for y in plan.years], dtype=float)
                    assert np.array_equal(t[cfg.name][reg + "_grid_index"], pid % 7 - 1)
                    assert np.array_equal(t[cfg.name][reg + "_ess"], pid + 0.5)
                    assert np.array_equal(t[cfg.name][reg + "_w_max"], 1.0 / (pid + 1))
                    q = t[cfg.name][reg + "_quantiles"]
                    assert q.shape == (len(plan.years), 3)
                    assert np.array_equal(q, pid[:, None] + 0.1 * np.arange(3))
                    line = t[cfg.name][reg + "_raw_fmean_rt"] - t[cfg.name][reg + "_raw_fmean"]
                    assert np.allclose(t[cfg.name][reg + "_quantiles_rt"], q + line[:, None], rtol=1e-13, atol=0)
                assert set(t[cfg.name]) - set(p[cfg.name]) == {
                    reg + s for reg in cfg.regions
                    for s in ("_grid_index", "_ess", "_w_max", "_quantiles", "_quantiles_rt")}
            sk = plan.skill(t)                                       # skill() reads a marginal dict unchanged
            assert sk == plan.skill(p)
    plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020)
    raw, marg = _fake(plan, n_q=0)
    out = plan.assemble(raw, marginal=marg)
    assert out["north_june"][CONFIGS["north_june"].regions[0] + "_quantiles"].shape == (len(plan.years), 0)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    from seaiceextentforecasting_b200 import parallel
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ok = True
    for members in (1, 3):                                           # 3 members: ranks own unequal problem counts
        plan = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, rank=rank, world=world, members=members)
        full = SweepPlan(NORTH_INITS, _sie(), 2015, 2020, members=members)
        raw, marg = _fake(plan)
        out = parallel.gather_results(plan, raw, marginal=marg)
        full_raw, full_marg = _fake(full)
        ref = full.assemble(full_raw, marginal=full_marg)
        outs, refs = (out, ref) if members > 1 else ([out], [ref])
        for o, r in zip(outs, refs):
            for c in r:
                ok &= o[c].keys() == r[c].keys()
                ok &= all(np.array_equal(o[c][k], r[c][k], equal_nan=True) for k in r[c])
    if rank == 0:
        q.put(bool(ok))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_gather_assembles_the_marginal_sweep():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ok = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    assert ok


def test_grid_marginal_rejects_bad_arguments(lib_built):
    """Checked before anything is enqueued, so no device is needed."""
    from seaiceextentforecasting_b200 import _lib
    lib = _lib.load()
    buf = (ctypes.c_double * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    null = ctypes.c_void_p(0)
    args = [p, 4, 400, p, 3, p, p, p, null]
    for i in (0, 3, 5, 6, 7):                                        # each device pointer NULL in turn
        bad = list(args)
        bad[i] = null
        assert lib.sie_gp_grid_marginal(*bad) == -1, i
    for i, v in ((1, 0), (1, -2), (2, 0), (2, -1), (4, -1)):         # P, n_grid < 1, n_q < 0
        bad = list(args)
        bad[i] = v
        assert lib.sie_gp_grid_marginal(*bad) == -1, (i, v)
    assert b"sie_gp_grid_marginal" in lib.sie_last_error()
