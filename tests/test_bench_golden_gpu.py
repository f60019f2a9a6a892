"""Full-size parity of the BENCHMARKED workloads against outputs of the unmodified reference
(tests/golden/bench_*.npz, written by tests/golden/make_bench_golden.py from /root/reference):

  * bench_north_m0 : BASELINE.json configs[1], `bench.make_workload(0)` -- 144 SIC 57x57 + 36 SST 26x90 networks, 432 forecasts
  * bench_north_m1 : the perturbed-SIC ensemble member `bench.make_workload(1)` (configs[4])
  * bench_south_feb: BASELINE.json configs[2], `bench.make_workload_south(0)` -- 36 SIC 81x81 networks, 108 forecasts

Bars: every network's `V` (dict keys, member cells, list order) bit-exact; tau <= 1e-9 relative; node series <= 1e-9
relative where the fixture stores them (the networks of five years), per-area sums of squares within the bound that
implies for every network; GP outputs
within max(1e-9, 64 2^s eps, 8 cond(K) eps) relative (the last two terms are the conditioning of the reference's own
arithmetic, SURVEY.md H3/H4); predictor counts equal; `info = -1` exactly where the reference's forecast() raises.
The CPU half (not marked gpu) guards the input generators and re-pins the oracle on a few of the full-size networks.
"""
import os
import sys
import warnings

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

import bench  # noqa: E402
from seaiceextentforecasting_b200.config import CONFIGS  # noqa: E402

GOLD = os.path.join(HERE, "golden")
FILES = {"north0": "bench_north_m0.npz", "north1": "bench_north_m1.npz", "south": "bench_south_feb.npz"}
EPS = 2.0 ** -53


def workload(kind):
    return bench.make_workload_south(0) if kind == "south" else bench.make_workload(int(kind[-1]))


def input_digest(w):
    import hashlib
    h = hashlib.sha256()
    for name in sorted(w["sic"]):
        h.update(np.ascontiguousarray(w["sic"][name]).tobytes())
    for reg in sorted(w["sie"]):
        h.update(np.ascontiguousarray(w["sie"][reg], dtype=np.float64).tobytes())
    if w.get("sst") is not None:
        h.update(np.ascontiguousarray(w["sst"]).tobytes())
    h.update(np.ascontiguousarray(w["psar"]).tobytes())
    return h.hexdigest()


class Fixture:
    def __init__(self, kind):
        self.g = g = np.load(os.path.join(GOLD, FILES[kind]))
        self.names = [str(n) for n in g["config_names"]]
        self.fmin, self.fmax = int(g["fmin"]), int(g["fmax"])
        nk = g["V_nkeys"].astype(np.int64)
        self.key_off = np.concatenate([[0], np.cumsum(nk)])
        lens = g["V_lens"].astype(np.int64)
        per_job_cells = np.array([lens[self.key_off[j]:self.key_off[j + 1]].sum() for j in range(len(nk))])
        self.cell_off = np.concatenate([[0], np.cumsum(per_job_cells)])
        T = g["job_year"].astype(np.int64) - 1979 + 1
        jobs = g["anom_jobs"].astype(np.int64)           # networks whose node series are stored in full
        self.anom_off = dict(zip(jobs.tolist(), np.concatenate([[0], np.cumsum(nk[jobs] * T[jobs])]).tolist()))
        self.index = {(int(c), int(y)): j for j, (c, y) in enumerate(zip(g["job_cfg"], g["job_year"]))}

    def network(self, cfg_index, year):
        """-> keys [nA], lens [nA], cells [n, 2] (list order), tau, anomaly [nA, T] (None where the fixture keeps only
        the norms) of one reference network build."""
        g, j = self.g, self.index[(cfg_index, year)]
        k0, k1 = self.key_off[j], self.key_off[j + 1]
        T = year - 1979 + 1
        anom = None
        if j in self.anom_off:
            a0 = self.anom_off[j]
            anom = g["anom"][a0:a0 + (k1 - k0) * T].reshape(k1 - k0, T)
        return (g["V_keys"][k0:k1], g["V_lens"][k0:k1], g["V_cells"][self.cell_off[j]:self.cell_off[j + 1]],
                float(g["job_tau"][j]), anom)

    def anom_norms(self, cfg_index, year):
        """-> per-area sum of squares [nA] and largest |value| of the node series of one reference network build."""
        j = self.index[(cfg_index, year)]
        return self.g["anom_sumsq"][self.key_off[j]:self.key_off[j + 1]], float(self.g["anom_absmax"][j])


def have(kind):
    return os.path.exists(os.path.join(GOLD, FILES[kind]))


KINDS = [k for k in FILES if have(k)]


def test_fixtures_present():
    assert have("north0") and have("south"), "run tests/golden/make_bench_golden.py (authoring container)"


@pytest.mark.parametrize("kind", KINDS)
def test_workload_generators_reproduce_the_fixture_inputs(kind):
    fx = Fixture(kind)
    assert input_digest(workload(kind)) == str(fx.g["input_sha256"])
    nprob = len(fx.g["gp_fmean"])
    assert nprob == 3 * (fx.fmax - fx.fmin + 1) * len(fx.names)


@pytest.mark.parametrize("kind,cfg_index,year", [("north0", -1, 1985), ("north0", -1, 1999), ("north0", 1, 1985),
                                                 ("north0", 3, 1987), ("south", 0, 1985)])
def test_oracle_equals_reference_on_full_size_networks(kind, cfg_index, year):
    """The oracle restatement against the reference's own output on networks of the benchmarked size (the cheapest
    ones: short windows / the SST grid; the generator asserts the same on every 8th network of the sweep)."""
    if not have(kind):
        pytest.skip("fixture not generated")
    from oracle import sweep as osweep
    fx, w = Fixture(kind), workload(kind)
    keys, lens, cells, tau, anom = fx.network(cfg_index, year)
    assert anom is not None, "make_bench_golden.ANOM_YEARS must keep this network's node series"
    if cfg_index < 0:
        field, latlon, weight = w["sst"], True, w["lat"]
    else:
        field, latlon, weight = w["sic"][fx.names[cfg_index]], False, w["psar"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        V, an, otau = osweep.build_network(field, year, latlon, weight)
    assert list(V) == [int(k) for k in keys]
    assert [len(V[k]) for k in V] == [int(x) for x in lens]
    assert np.array_equal(np.array([c for k in V for c in V[k]]), cells.astype(np.int64))
    assert otau == tau
    assert np.array_equal(np.array([an[k] for k in V]), anom)


def gp_tol(rec, cond):
    return max(1e-9, 64.0 * 2.0 ** int(rec["expm_s"]) * EPS, 8.0 * float(cond) * EPS)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_benchmarked_sweep_matches_reference(lib_built, kind):
    from seaiceextentforecasting_b200.forecast import RetrospectiveSweep
    fx, w = Fixture(kind), workload(kind)
    g = fx.g
    assert input_digest(w) == str(g["input_sha256"])
    sw = RetrospectiveSweep(fx.names, w["sic"], w["sie"], fx.fmin, fx.fmax, w["psar"], w["sst"], w["lat"],
                            max_pred=max(384, (int(g["gp_n_pred"].max()) + 3) // 4 * 4))
    out = sw.run()
    raw = sw.raw
    assert len(raw) == len(g["gp_fmean"])

    # ---- networks: V bit-exact (keys, membership, list order), tau, node series
    def check_engine(eng, jobs):
        assert (eng.status.cpu().numpy() == 0).all()
        nA = eng.n_areas.cpu().numpy()
        keys = eng.area_key.cpu().numpy()
        starts = eng.area_start.cpu().numpy()
        cells = eng.area_cells.cpu().numpy()
        tau = eng.tau.cpu().numpy()
        anom = eng.anomaly.cpu().numpy()
        for b, (ci, year) in enumerate(jobs):
            rkeys, rlens, rcells, rtau, ranom = fx.network(ci, year)
            n = int(nA[b])
            assert n == len(rkeys), (kind, ci, year, n, len(rkeys))
            assert np.array_equal(keys[b, :n], rkeys), (kind, ci, year, "dict keys / order")
            assert np.array_equal(np.diff(starts[b, :n + 1]), rlens), (kind, ci, year, "area sizes")
            flat = cells[b, :starts[b, n]]
            assert np.array_equal(np.stack([flat // eng.Y, flat % eng.Y], 1), rcells.astype(np.int64)), \
                (kind, ci, year, "member cells / list order")
            assert abs(tau[b] - rtau) <= 1e-9 * abs(rtau), (kind, ci, year, tau[b], rtau)
            T = year - 1979 + 1
            got = anom[b, :n, :T]
            if ranom is not None:
                assert np.abs(got - ranom).max() <= 1e-9 * np.abs(ranom).max(), (kind, ci, year, "node series")
            # every network: per-area sums of squares within what that elementwise bound implies (|g^2 - r^2| <=
            # e (2 max|r| + e), e = 1e-9 max|r|, summed over T samples: 2e-9 T max|r|^2; 3e-9 leaves room for rounding)
            sumsq, amax = fx.anom_norms(ci, year)
            assert np.abs((got * got).sum(axis=1) - sumsq).max() <= 3e-9 * T * amax ** 2, (kind, ci, year, "node norms")

    check_engine(sw.sic, sw.plan.jobs)
    if sw.sst is not None:
        check_engine(sw.sst, [(-1, y) for y in sw.plan.sst_years])

    # ---- forecasts
    ref = {(int(c), int(k), int(y)): i for i, (c, k, y) in enumerate(zip(g["gp_cfg"], g["gp_region"], g["gp_year"]))}
    n_fail = 0
    worst = 0.0
    for p, (ci, k, year) in enumerate(sw.plan.prob_meta):
        i = ref[(ci, k, year)]
        rec = raw[p]
        name, reg = fx.names[ci], CONFIGS[fx.names[ci]].regions[k]
        if g["gp_failed"][i]:
            assert rec["info"] == -1, (name, reg, year, rec)            # the reference's forecast() raises here
            assert np.isnan(rec["fmean"])
            n_fail += 1
            continue
        assert rec["info"] == 0, (name, reg, year, rec)
        assert rec["n_pred"] == g["gp_n_pred"][i], (name, reg, year, rec["n_pred"], g["gp_n_pred"][i])
        t = gp_tol(rec, g["gp_cond"][i])
        rf, rv = g[f"raw_{name}_{reg}_fmean"][year - fx.fmin], g[f"raw_{name}_{reg}_fvar"][year - fx.fmin]
        scale = max(abs(rf), np.sqrt(abs(rv)))         # the predictive standard deviation is the mean's natural scale
        assert abs(rec["fmean"] - rf) <= t * scale, (name, reg, year, rec["fmean"], rf, t)
        assert abs(rec["fvar"] - rv) <= t * max(abs(rv), scale ** 2), (name, reg, year, rec["fvar"], rv, t)
        assert abs(rec["sigma_f"] - g["gp_sigma_f"][i]) <= t * abs(g["gp_sigma_f"][i]), (name, reg, year)
        # nlML = y'a/2 + sum(log L_ii) + n log(2 pi)/2 with y'a = n by construction of sigma_f: the three terms are O(n)
        # and cancel, so the bound scales with their magnitudes, not with the (possibly tiny) total
        n = year - 1979
        c0 = 0.5 * n + 0.5 * n * np.log(2 * np.pi)
        nl_scale = c0 + abs(g["gp_nlml"][i] - c0)
        assert abs(rec["nlml"] - g["gp_nlml"][i]) <= t * nl_scale, (name, reg, year, rec["nlml"], g["gp_nlml"][i], t)
        if t <= 1e-6:
            worst = max(worst, abs(rec["fmean"] - rf) / scale)
        # the reference's own output format (3 d.p.) wherever the bound is below the rounding step
        if t * max(scale, abs(g[f"raw_{name}_{reg}_fmean_rt"][year - fx.fmin])) < 5e-4:
            for suf in ("_fmean", "_fvar", "_fmean_rt"):
                assert abs(out[name][reg + suf][year - fx.fmin] - g[f"rnd_{name}_{reg}{suf}"][year - fx.fmin]) \
                    <= 1e-3 + 1e-12, (name, reg, year, suf)
    assert n_fail == int(g["gp_failed"].sum())
    print(f"{kind}: {len(raw)} forecasts, {n_fail} reference failures reproduced, worst well-conditioned fmean "
          f"deviation {worst:.2e} relative")
