"""Ensemble forecasts (forecast.EnsembleForecast, sie_gp_ensemble): every member's predictive distribution of a
(config, region, year) pooled into one on the device.  Checked against oracle/ensemble.py on hand-made records and on
the records of plain, tuned and marginalised 4-member sweeps, against the marginal sweep itself for one member, for
bitwise equality across batch orders and graph replay, and at full size."""
import numpy as np
import pytest

from seaiceextentforecasting_b200.config import LS, NORTH_INITS, SS
from test_tuned_sweep_gpu import FMAX, FMIN, small_inputs

pytestmark = pytest.mark.gpu
LEVELS = (0.05, 0.25, 0.5, 0.75, 0.95)
POOLED = ("fmean", "fvar", "var_within", "var_between", "n_members")


def run_ensemble(rec, levels=LEVELS):
    """sie_gp_ensemble on host records rec [E][M][n_grid] -> (GP_ENSEMBLE_DTYPE [E], quantiles [E][n_q])."""
    import torch

    from seaiceextentforecasting_b200.engine import h2d
    from seaiceextentforecasting_b200.forecast import GP_ENSEMBLE_DTYPE, gp_ensemble, gp_ensemble_scratch_bytes
    E, M, n = rec.shape
    nq = len(levels)
    out = torch.empty(E * GP_ENSEMBLE_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    quant = torch.empty(max(1, E * nq), dtype=torch.float64, device="cuda")
    scratch = torch.empty(gp_ensemble_scratch_bytes(E, M, n), dtype=torch.uint8, device="cuda")
    gp_ensemble(h2d(np.ascontiguousarray(rec).view(np.uint8).reshape(-1)), E, M, n,
                h2d(np.asarray(levels, dtype=np.float64)) if nq else None, out, quant, scratch)
    return out.cpu().numpy().view(GP_ENSEMBLE_DTYPE), quant.cpu().numpy()[:E * nq].reshape(E, nq)


def check_against_oracle(rec, pooled, quant, levels=LEVELS, jumps=False):
    """The device's pool of every problem == oracle/ensemble.py on the same records: moments within 1e-13 relative, the
    quantiles through the oracle CDF within 1e-12 of their level (`jumps`, point masses: F(x) >= q > F(the next lower
    double) within 1e-12).  Returns the number of problems with M' >= 1."""
    from oracle import ensemble as oe
    from oracle import marginal as om
    n_ok = 0
    for e in range(rec.shape[0]):
        g = rec[e]
        r = oe.ensemble(g["fmean"], g["fvar"], g["nlml"], g["info"], levels)
        assert pooled["n_members"][e] == r["n_members"], e
        if r["n_members"] == 0:
            assert all(np.isnan(pooled[f][e]) for f in POOLED[:4]) and np.isnan(quant[e]).all(), e
            continue
        scale = max(abs(r["fmean"]), np.sqrt(r["fvar"]))
        assert abs(pooled["fmean"][e] - r["fmean"]) <= 1e-13 * scale, (e, pooled["fmean"][e], r["fmean"])
        for f in ("fvar", "var_within", "var_between"):
            assert abs(pooled[f][e] - r[f]) <= 1e-13 * r["fvar"], (e, f, pooled[f][e], r[f])
        assert pooled["fvar"][e] == pooled["var_within"][e] + pooled["var_between"][e]
        for t, x in zip(levels, quant[e]):
            if jumps:
                assert om.mixture_cdf(x, r["w"], r["mu"], r["var"]) >= t - 1e-12, (e, t, x)
                assert om.mixture_cdf(np.nextafter(x, -np.inf), r["w"], r["mu"], r["var"]) < t + 1e-12, (e, t, x)
            else:
                assert abs(om.mixture_cdf(x, r["w"], r["mu"], r["var"]) - t) <= 1e-12, (e, t, x)
        assert np.all(np.diff(quant[e]) >= 0), e
        n_ok += 1
    return n_ok


def _random(rng, shape):
    from seaiceextentforecasting_b200.forecast import GP_RESULT_DTYPE
    rec = np.zeros(shape, dtype=GP_RESULT_DTYPE)
    rec["fmean"] = rng.normal(0.0, 0.4, shape)
    rec["fvar"] = rng.uniform(0.01, 0.3, shape)
    rec["nlml"] = rng.uniform(-3.0, 3.0, shape)
    return rec


def test_hand_made_records(lib_built):
    """M' = 0, one member, members without an admissible record mixed in, point masses, an nlML spread of 1e4 inside a
    member; then M = 1024 Gaussians and M = 16 members of 400 grid points."""
    rng = np.random.default_rng(21)
    E, M, n = 6, 5, 40
    rec = _random(rng, (E, M, n))
    rec["info"][0] = 2                                            # 0: no member has an admissible record
    rec["nlml"][0, 1] = np.inf
    rec["info"][1] = 1                                            # 1: one member (2), and one record of it
    rec["info"][1, 2, 17] = 0
    rec["info"][2, 0] = 3                                         # 2: members 0 and 3 without a forecast
    rec["nlml"][2, 3] = np.nan
    rec["fvar"][3, :, ::3] = 0.0                                  # 3: point masses and negative variances
    rec["fvar"][3, :, 1::7] = -1e-9
    rec["nlml"][4] = rng.uniform(0.0, 1e4, (M, n))                # 4: nlML spread 1e4 (weights underflow to 0)
    pooled, quant = run_ensemble(rec)
    assert check_against_oracle(rec, pooled, quant, jumps=True) == E - 1
    assert pooled["n_members"].tolist() == [0, 1, 3, 5, 5, 5]
    assert pooled["fmean"][1] == rec["fmean"][1, 2, 17] and pooled["var_within"][1] == rec["fvar"][1, 2, 17]
    assert pooled["var_between"][1] == 0.0
    assert np.isfinite(quant[4]).all()
    _, none = run_ensemble(rec, levels=())                        # no quantiles: NULL q / quant
    assert none.shape == (E, 0)

    big = _random(rng, (3, 1024, 1))                              # 1024 Gaussian members
    big["info"][1, ::3] = 1
    pooled, quant = run_ensemble(big)
    assert check_against_oracle(big, pooled, quant) == 3
    assert pooled["n_members"].tolist() == [1024, 1024 - 342, 1024]

    grid = _random(rng, (2, 16, 400))                             # 16 members of a 400-point grid
    grid["info"][0, 5] = 1
    grid["info"][:, :, ::11] = 4
    pooled, quant = run_ensemble(grid)
    assert check_against_oracle(grid, pooled, quant) == 2 and pooled["n_members"].tolist() == [15, 16]


def test_above_the_member_limit_is_refused(lib_built):
    from seaiceextentforecasting_b200._lib import SieError
    with pytest.raises(SieError, match="at most 1024"):
        run_ensemble(_random(np.random.default_rng(2), (1, 1025, 1)))


def sweep(ws, mode, **kw):
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    if mode != "plain":
        kw.update(hyper_grid=(LS, SS), hyper_mode="argmin" if mode == "tuned" else "marginal")
    return RetrospectiveSweep(NORTH_INITS, [w["sic"] for w in ws], ws[0]["sie"], FMIN, FMAX, ws[0]["psar"],
                              [w["sst"] for w in ws], ws[0]["lat"], wave_T=(16,), **kw)


def member_records(sw, ens):
    """The sweep's device records of its last step in the store's layout: host [E][members][n_grid]."""
    from seaiceextentforecasting_b200.forecast import ensemble_slots
    rec = sw.grid_records().reshape(sw.P, -1) if sw.hyper_mode == "marginal" else sw.raw.reshape(sw.P, 1)
    _, rows = ensemble_slots(sw.plan, sw.members)
    out = np.empty((ens.E * sw.members, rec.shape[1]), dtype=rec.dtype)
    out[rows] = rec
    return out.reshape(ens.E, sw.members, rec.shape[1])


def test_one_member_is_the_marginal_forecast(lib_built):
    """M = 1 on the small marginal sweep's grid records: fmean and var_within are the sweep's marginal fmean / fvar bit
    for bit, var_between is 0; the assembled dict keeps the member's keys."""
    from seaiceextentforecasting_b200.forecast import EnsembleForecast, ensemble_slots
    sw = sweep([small_inputs(0)], "marginal", quantiles=LEVELS)
    out = sw.run()
    ens = EnsembleForecast(sw, 1, LEVELS)
    ens.add(sw)
    d = ens.result()
    _, rows = ensemble_slots(sw.plan, 1)
    r = ens.records[rows]
    ok = sw.marginal["n_admissible"] > 0
    assert ok.sum() >= 30 and (~ok).sum() >= 1
    assert np.array_equal(r["fmean"], sw.raw["fmean"], equal_nan=True)
    assert np.array_equal(r["var_within"], sw.raw["fvar"], equal_nan=True)
    assert (r["var_between"][ok] == 0).all() and np.array_equal(r["n_members"], ok.astype(np.int32))
    assert np.isnan(r["quantiles"][~ok]).all()
    for c in out:
        for k, v in out[c].items():
            if not k.endswith(("_grid_index", "_ess", "_w_max", "_quantiles", "_quantiles_rt")):
                assert np.array_equal(d[c][k], v, equal_nan=True), (c, k)


@pytest.mark.parametrize("mode", ["plain", "tuned", "marginal"])
def test_four_member_sweeps_match_the_oracle(lib_built, mode):
    from seaiceextentforecasting_b200.forecast import EnsembleForecast
    sw = sweep([small_inputs(m) for m in range(4)], mode)
    sw.run()
    ens = EnsembleForecast(sw, 4, LEVELS)
    ens.add(sw)
    d = ens.result()
    rec = member_records(sw, ens)
    assert rec.shape == (ens.E, 4, 400 if mode == "marginal" else 1)
    n_ok = check_against_oracle(rec, ens.records, ens.records["quantiles"])
    adm = ((rec["info"] == 0) & np.isfinite(rec["nlml"])).any(axis=2).sum(axis=1)
    assert np.array_equal(ens.records["n_members"], adm) and (adm > 0).sum() == n_ok >= 30
    sk = sw.plan.skill(d)
    assert set(sk) == {c.name for c in sw.cfgs}
    print(f"{mode}: {n_ok} of {ens.E} problems pooled, n_members histogram {np.bincount(adm, minlength=5).tolist()}")


def test_outputs_do_not_depend_on_the_batches(lib_built):
    """One 4-member sweep added once == a 2-member sweep fed members {0, 1} then {2, 3} through load_inputs == the same
    batches in reverse order == those batches under CUDA-graph replay: the same bits."""
    from seaiceextentforecasting_b200.forecast import EnsembleForecast
    ws = [small_inputs(m) for m in range(4)]
    full = sweep(ws, "marginal")
    full.run()
    ens = EnsembleForecast(full, 4, LEVELS)
    ens.add(full)
    ref_dict = ens.result()
    ref = ens.records.copy()
    del full
    pair = sweep(ws[:2], "marginal")
    for graph, order in ((False, (0, 2)), (False, (2, 0)), (True, (2, 0))):
        pair.use_graph = graph
        ens = EnsembleForecast(pair, 4, LEVELS)
        for first in order:
            pair.load_inputs([w["sic"] for w in ws[first:first + 2]], [w["sst"] for w in ws[first:first + 2]])
            pair.upload()
            pair.compute()
            ens.add(pair, first)
        d = ens.result()
        assert ens.records.tobytes() == ref.tobytes(), (graph, order)
        for c in ref_dict:
            for k, v in ref_dict[c].items():
                assert np.array_equal(d[c][k], v, equal_nan=True), (graph, order, c, k)


def test_errors(lib_built):
    from seaiceextentforecasting_b200.forecast import EnsembleForecast
    w = small_inputs(0)
    sw = sweep([w], "plain")
    sw.run()
    ens = EnsembleForecast(sw, 2)
    ens.add(sw, 1)
    with pytest.raises(RuntimeError, match="never added"):                # member slot 0 is missing
        ens.result()
    with pytest.raises(ValueError):                                       # past the last slot
        ens.add(sw, 2)
    with pytest.raises(ValueError):
        ens.add(sw, -1)
    tuned = sweep([w], "tuned")
    with pytest.raises(ValueError, match="hyper mode"):                   # another hyper mode
        ens.add(tuned)
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    other = RetrospectiveSweep(NORTH_INITS, w["sic"], w["sie"], FMIN + 1, FMAX, w["psar"], w["sst"], w["lat"])
    with pytest.raises(ValueError):                                       # other years
        ens.add(other)
    ens.add(sw, 0)
    ens.result()
    ranked = RetrospectiveSweep(NORTH_INITS, w["sic"], w["sie"], FMIN, FMAX, w["psar"], w["sst"], w["lat"], rank=0,
                                world=2)
    with pytest.raises(NotImplementedError):
        EnsembleForecast(ranked, 2)


def test_full_size_ensemble_invariants(lib_built):
    """The bench's 8-member north marginal step pooled: fvar >= var_within >= 0, monotone quantiles, n_members <= 8 and
    NaN exactly where no member has a forecast."""
    import bench
    from seaiceextentforecasting_b200.forecast import EnsembleForecast, RetrospectiveSweep, ensemble_slots
    ws = [bench.make_workload(m) for m in range(8)]
    sw = RetrospectiveSweep(NORTH_INITS, [x["sic"] for x in ws], ws[0]["sie"], bench.FMIN, bench.FMAX, ws[0]["psar"],
                            [x["sst"] for x in ws], ws[0]["lat"], hyper_grid=(LS, SS), hyper_mode="marginal",
                            quantiles=LEVELS)
    sw.run()
    ens = EnsembleForecast(sw, 8, LEVELS)
    ens.add(sw)
    d = ens.result()
    r = ens.records
    assert ens.E == 432 and len(d) == 4
    _, rows = ensemble_slots(sw.plan, 8)
    has = np.zeros(ens.E * 8, dtype=bool)
    has[rows] = sw.marginal["n_admissible"] > 0
    count = has.reshape(ens.E, 8).sum(axis=1)
    assert np.array_equal(r["n_members"], count) and (count <= 8).all()
    ok = count > 0
    for f in ("fmean", "fvar", "var_within", "var_between"):
        assert np.isfinite(r[f][ok]).all() and np.isnan(r[f][~ok]).all(), f
    assert np.isnan(r["quantiles"][~ok]).all() and np.isfinite(r["quantiles"][ok]).all()
    assert np.all(r["fvar"][ok] >= r["var_within"][ok]) and np.all(r["var_within"][ok] >= 0)
    assert np.all(np.diff(r["quantiles"][ok], axis=1) >= 0)
    print(f"full size: {ok.sum()} of {ens.E} problems pooled, n_members histogram {np.bincount(count).tolist()}, "
          f"median var_between / fvar {np.median(r['var_between'][ok] / r['fvar'][ok]):.3f}")
