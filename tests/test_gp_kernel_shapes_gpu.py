"""k_gp_forecast at every tile, panel and tier boundary of its shape-dependent code, against the extended-precision
reference oracle/gp_ext.py (pinned on the CPU by tests/test_gp_ext_reference.py).

The problems go straight to GpBatch, so each test chooses the leading dimension `ld` = max_pred: forecast() always
sizes it to the problem.  Series use Tstride = 64, so every n up to the kernel's limit fits.  With rule 'all' and no
SST, Np is exactly the number of SIC series.

Every record field is compared with the reference evaluated at the (m, s) the kernel reports, so the two differ only
in rounding, within  max(2^-40, 64 2^s u, 8 cond(K) u)  relative (u = 2^-53): fmean against the predictive standard
deviation, fvar against its square, nlml against the sum of its terms' magnitudes, each gradient component against
|trace(K^-1 dK)| / 2 + |alpha^T dK alpha| / 2.  The reported (m, s) must be oracle.expm_spec.pick's, n_pred and info
exact.  Each group prints its worst error-to-bound ratio."""
import dataclasses

import numpy as np
import pytest

from oracle import expm_spec as es
from oracle import gp as og
from oracle import gp_ext as ge
from seaiceextentforecasting_b200.config import RULE_ALL, RULE_POS, RULE_POS_SIG

pytestmark = pytest.mark.gpu

TSTRIDE = 64
RULE_NAME = {RULE_POS: "pos", RULE_ALL: "all", RULE_POS_SIG: "pos_sig"}
VALUE_FIELDS = ("fmean", "fvar", "sigma_f", "nlml", "g_ell", "g_sig", "n_pred", "expm_m", "expm_s", "info")
PADE = [(3, 0), (5, 0), (7, 0), (9, 0), (13, 0), (13, 1), (13, 5), (13, 20)]

# Smem of csrc/gp.cu (k_gp_forecast's shared memory), in doubles: As[2][64 * 20], Bs[2][16 * 68], then the CTA-wide
# K[64 * 65] -- the grid mode's per-warp workspaces -- in front of W.  Each warp needs n (n | 1) + 4 * 64 doubles, so
# nwu = min(8, avail / that) warps evaluate sigma values at once (warp_sigma_fit's callers, gp.cu)
_SMEM_AVAIL = 2 * 64 * 20 + 2 * 16 * 68 + 64 * 65


def nwu_of(n):
    return min(8, _SMEM_AVAIL // (n * (n | 1) + 4 * 64))


@dataclasses.dataclass
class Case:
    key: str
    y: np.ndarray
    sic: dict
    sst: dict = None
    rule: int = RULE_ALL
    alpha: float = 0.05
    zscore: bool = True
    ell: float = 1e-2
    sig: float = 1.0
    want_grad: bool = False
    max_pred: int = 520

    @property
    def n(self):
        return len(self.y)


class Series:
    """anomaly [J][MA][TSTRIDE], n_areas [J], MA, Tstride: the attributes GpBatch reads from a NetworkBatch."""

    def __init__(self, sets):
        import torch
        from seaiceextentforecasting_b200.engine import h2d
        ma = max([1] + [len(s) for s in sets])
        arr = np.zeros((len(sets), ma, TSTRIDE))
        for j, s in enumerate(sets):
            for a, v in enumerate(s.values()):
                v = np.asarray(v, dtype=np.float64)[:TSTRIDE]
                arr[j, a, :len(v)] = v
        self.anomaly = h2d(arr)
        self.n_areas = torch.tensor([len(s) for s in sets], dtype=torch.int32, device="cuda")
        self.MA, self.Tstride = ma, TSTRIDE


def _inputs(cases):
    from seaiceextentforecasting_b200.engine import r_crit_pearson
    from seaiceextentforecasting_b200.forecast import GP_PROBLEM_DTYPE
    prob = np.zeros(len(cases), dtype=GP_PROBLEM_DTYPE)
    ys, sst_sets, off = [], [], 0
    for p, c in enumerate(cases):
        prob[p]["job_sic"] = p
        prob[p]["job_sst"] = -1 if c.sst is None else len(sst_sets)
        if c.sst is not None:
            sst_sets.append(c.sst)
        prob[p]["n"], prob[p]["y_off"] = c.n, off
        prob[p]["rule"], prob[p]["zscore"], prob[p]["want_grad"] = c.rule, int(c.zscore), int(c.want_grad)
        prob[p]["r_sel"] = r_crit_pearson(c.n, c.alpha) if c.rule == RULE_POS_SIG else 0.0
        prob[p]["ell"], prob[p]["sig"] = c.ell, c.sig
        ys.append(np.asarray(c.y, dtype=np.float64))
        off += c.n
    return prob, np.concatenate(ys), Series([c.sic for c in cases]), Series(sst_sets) if sst_sets else None


def launch(cases, max_pred):
    """One sie_gp_forecast launch of all `cases` at leading dimension max_pred -> GP_RESULT_DTYPE [len(cases)]."""
    import torch
    from seaiceextentforecasting_b200.engine import h2d
    from seaiceextentforecasting_b200.forecast import GpBatch
    prob, y, sic, sst = _inputs(cases)
    gp = GpBatch(len(cases), max_pred=max_pred)
    assert gp.max_pred == max_pred
    gp.run(h2d(prob.view(np.uint8)), h2d(y), sic, sst)
    rec = gp.results().copy()
    del gp
    torch.cuda.synchronize()
    return rec


def launch_grid(cases, sigs, max_pred):
    """One sie_gp_hyper_grid launch: problem p at l = cases[p].ell, every sigma of `sigs` -> records [P][n_sig]."""
    import torch
    from seaiceextentforecasting_b200.engine import h2d
    from seaiceextentforecasting_b200.forecast import GP_RESULT_DTYPE, GpBatch
    prob, y, sic, sst = _inputs(cases)
    gp = GpBatch(len(cases), max_pred=max_pred)
    out = torch.empty(len(cases) * len(sigs) * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    gp.run_grid(h2d(prob.view(np.uint8)), h2d(np.asarray(sigs, dtype=np.float64)), len(sigs), h2d(y), sic, sst, out)
    rec = out.cpu().numpy().view(GP_RESULT_DTYPE).reshape(len(cases), len(sigs)).copy()
    del gp
    torch.cuda.synchronize()
    return rec


# ------------------------------------------------------------------------------------------------------------------
# the reference side
# ------------------------------------------------------------------------------------------------------------------
_REF = {}
_FIT = {}


def fit(c, m, s, sig):
    """reference(c, m, s)'s Problem.fit(sig), computed once."""
    k = (c.key, int(m), int(s), float(sig))
    if k not in _FIT:
        _FIT[k] = reference(c, m, s)[0].fit(sig)
    return _FIT[k]


def reference(c, m, s):
    """(ge.Problem at (m, s), n_pred, float64 Laplacian M), computed once per (case, m, s)."""
    k = (c.key, int(m), int(s))
    if k not in _REF:
        Xfull = og.select_predictors(np.asarray(c.y, dtype=np.float64), c.sic, c.sst, RULE_NAME[c.rule], c.alpha)
        M = og.design(Xfull, c.zscore)[2] if Xfull.ndim == 2 and Xfull.shape[1] >= 2 else None
        pr = ge.Problem(Xfull, c.y, c.zscore, c.ell, m, s, c.want_grad) if M is not None and m else None
        _REF[k] = (pr, Xfull.shape[1] if Xfull.ndim == 2 else 0, M)
    return _REF[k]


class Ratios:
    """Error-to-bound ratios of one group: `add` records them, `check` prints the worst and asserts all <= 1."""

    def __init__(self, group):
        self.group, self.items = group, []

    def add(self, where, field, err, bound):
        self.items.append((float(err) / bound, where, field, float(err), bound))

    def check(self):
        assert self.items, self.group
        worst = max(self.items)
        print(f"\n[{self.group}] {len(self.items)} comparisons, worst error/bound {worst[0]:.3g} "
              f"({worst[1]} {worst[2]}: error {worst[3]:.3g}, bound {worst[4]:.3g})")
        bad = [i for i in self.items if not i[0] <= 1.0]
        assert not bad, bad[:10]


def check_record(c, r, ratios, sig=None, where=None):
    """Compare one kernel record with the reference at the record's (m, s); returns the reported (m, s)."""
    where = where or c.key
    sig = c.sig if sig is None else sig
    _, n_pred, M = reference(c, r["expm_m"], r["expm_s"])
    assert r["n_pred"] == n_pred, (where, r["n_pred"], n_pred)
    assert r["info"] == 0, (where, r["info"])
    m, s, _ = es.pick(c.ell * M)
    if (m, s) != (int(r["expm_m"]), int(r["expm_s"])):
        assert ge.pick_margin(c.ell * M) < 1e-12, (where, (m, s), (r["expm_m"], r["expm_s"]))
    ref = fit(c, r["expm_m"], r["expm_s"], sig)
    assert ref["info"] == 0, where
    t = ge.bound(r["expm_s"], ref["cond"])
    for f, scale in scales(ref, c.want_grad).items():
        ratios.add(where, f, abs(float(r[f]) - float(ref[f])) / scale, t)
    return int(r["expm_m"]), int(r["expm_s"])


def scales(ref, want_grad):
    """Per-field error scales: fmean against the predictive standard deviation, fvar against its square, nlml and the
    gradient components against the magnitudes of their terms."""
    sd = max(abs(float(ref["fmean"])), np.sqrt(abs(float(ref["fvar"]))), 1e-3)
    out = {"fmean": sd, "fvar": sd ** 2, "sigma_f": abs(float(ref["sigma_f"])), "nlml": max(1.0, float(ref["nlml_mag"]))}
    if want_grad:
        out["g_ell"] = max(1.0, float(ref["mag_ell"]))
        out["g_sig"] = max(1.0, float(ref["mag_sig"]))
    return out


def round4(x):
    return (x + 3) // 4 * 4


# ------------------------------------------------------------------------------------------------------------------
# the cases
# ------------------------------------------------------------------------------------------------------------------
def np_sweep_cases():
    out = []
    for Np in ge.NP_SWEEP:
        for zscore in (True, False):
            y, sic, ell, sig = ge.shape_problem(Np, 41, zscore)
            out.append(Case(f"sweep Np={Np} {'z' if zscore else 'raw'}", y, sic, zscore=zscore, ell=ell, sig=sig))
    return out


# Np of each row-slice count of the |A|^p power iteration (8 / 4 / 4 / 2 / 1 slices): its || |A|^(2m+1) ||_1 decides
# (m, s) near the lower end of each (m, s) interval of l
PADE_EDGE_NP = (17, 33, 64, 65, 129)
PADE_MID_NP = (33, 129, 257, 520)


def pade_cases():
    """Each (m, s) at the log-midpoint of its interval of l, and 5 % into it from the lower end (at the slice counts):
    there the backward-error check || |A|^(2m+1) ||_1 is what moved l M up to (m, s), and it does so with a margin
    (~0.05 in log2 of that norm) that a power iteration summing only part of its row slices falls short of."""
    out = []
    for Np in sorted(set(PADE_MID_NP) | set(PADE_EDGE_NP)):
        y, sic, _, _ = ge.shape_problem(Np, 41, True, seed=1)
        M = og.design(og.select_predictors(y, sic, None, "all"), True)[2]
        spots = ([("mid", 0.5)] if Np in PADE_MID_NP else []) + ([("low", 0.05)] if Np in PADE_EDGE_NP else [])
        for m, s in (PADE if Np < 520 else [(3, 0), (13, 20)]):
            for where, at in spots:
                ell = ge.ell_for(M, m, s, at=at)
                assert ell is not None, (Np, m, s, where)
                out.append(Case(f"pade {where} Np={Np} (m,s)=({m},{s})", y, sic, ell=ell))
    return out


N_EDGES = (2, 3, 31, 32, 33, 62, 63)


def n_edge_cases():
    out = []
    for Np in (17, 129):
        for n in N_EDGES:
            y, sic, ell, sig = ge.shape_problem(Np, n, True)
            out.append(Case(f"n={n} Np={Np}", y, sic, ell=ell, sig=sig))
    y, sic, ell, sig = ge.shape_problem(100, 41, True)
    out.append(Case("Np=max_pred=100", y, sic, ell=ell, sig=sig, max_pred=100))
    return out


def rejected_cases():
    """(case, expected info): n + 1 > 64 samples, Np above max_pred, fewer than two predictors."""
    y, sic, _ = ge.series(5, 64, 17)
    y2, sic2, _ = ge.series(6, 41, 104)
    y3, sic3, _ = ge.series(7, 41, 1)
    return [(Case("n=64", y, sic), -2), (Case("Np=max_pred+4", y2, sic2, max_pred=100), -2),
            (Case("Np=1", y3, sic3), -1), (Case("Np=0", y3, {}), -1)]


def many_candidates_cases():
    """700 SIC and 300 SST series (four 256-wide chunks of the compaction), rules 'pos' and 'pos_sig'.  Every series is
    regenerated until its float64 Pearson r is at least 0.05 away from 0 and from r_sel, so selection is no
    rounding decision; 40 % of the SIC series correlate positively and half the SST series negatively."""
    from seaiceextentforecasting_b200.engine import r_crit_pearson
    n = 41
    rng = np.random.default_rng(2024)
    common = rng.standard_normal((3, n + 1))
    y = np.round(0.3 * (common[0, :n] - common[1, :n]) + 0.2 * rng.standard_normal(n), 3)
    r_sel = r_crit_pearson(n, 0.05)

    def draw(sign, amp):
        while True:
            x = amp * (sign * rng.uniform(0.1, 1.0) * np.concatenate([y, [0.0]]) / np.std(y)
                       + 0.5 * rng.standard_normal(3) @ common + rng.standard_normal(n + 1))
            r = np.corrcoef(y, x[:n])[0, 1]
            if np.sign(r) == sign and abs(r) > 0.05 and abs(r - r_sel) > 0.05:
                return x

    sic = {2 * a + 1: draw(1.0 if rng.uniform() < 0.4 else -1.0, 1.0) for a in range(700)}
    sst = {a: draw(-1.0 if rng.uniform() < 0.5 else 1.0, 0.1) for a in range(300)}
    out = []
    for rule in (RULE_POS, RULE_POS_SIG):
        Xfull = og.select_predictors(y, sic, sst, RULE_NAME[rule], 0.05)
        M = og.design(Xfull, True)[2]
        out.append(Case(f"1000 candidates rule={RULE_NAME[rule]}", y, sic, sst, rule=rule, ell=1.5 / es.norm1(M)))
    return out


def gradient_cases():
    out = []
    for Np in (33, 129, 257):
        y, sic, ell, sig = ge.shape_problem(Np, 41, True, seed=2, c=1.5)
        out.append(Case(f"grad Np={Np}", y, sic, ell=ell, sig=sig, want_grad=True))
    return out


GRID_N = (29, 30, 35, 36, 39, 40, 43, 44, 51, 52, 63)
GRID_NSIG = (1, 9, 20)


def grid_cases():
    out = []
    for Np in (17, 129):
        for n in GRID_N:
            y, sic, ell, _ = ge.shape_problem(Np, n, True, seed=3)
            out.append(Case(f"grid n={n} Np={Np}", y, sic, ell=ell, want_grad=True, max_pred=round4(Np)))
    return out


def grid_sigs(n_sig):
    return np.array([1.0]) if n_sig == 1 else np.logspace(-1, 2, n_sig)


@pytest.fixture(scope="module")
def alone(lib_built):
    """Every forecast case of groups 1-4 launched on its own at its own max_pred (the sweep also at a padded ld)."""
    cases = {g: f() for g, f in (("sweep", np_sweep_cases), ("pade", pade_cases), ("n", n_edge_cases),
                                 ("candidates", many_candidates_cases), ("grad", gradient_cases))}
    rec = {}
    for g, cs in cases.items():
        for c in cs:
            if g == "sweep":
                Np = len(c.sic)
                rec[c.key] = launch([c], round4(max(Np, 4)))[0]
                rec[c.key + " padded"] = launch([c], 384 if Np <= 384 else 520)[0]
            else:
                rec[c.key] = launch([c], c.max_pred)[0]
    return cases, rec


def test_np_sweep(alone):
    cases, rec = alone
    ratios = Ratios("Np sweep, tight and padded ld")
    seen = set()
    for c in cases["sweep"]:
        Np = len(c.sic)
        for suffix in ("", " padded"):
            r = rec[c.key + suffix]
            if Np < 2:
                assert r["info"] == -1
                continue
            check_record(c, r, ratios, where=c.key + suffix)
            seen.add(Np)
    ratios.check()
    assert seen == set(ge.NP_SWEEP) - {0, 1}


def test_pade_order_and_scaling(alone):
    cases, rec = alone
    ratios = Ratios("Pade order and scaling")
    seen = set()
    for c in cases["pade"]:
        want = tuple(int(v) for v in c.key.split("(m,s)=(")[1].rstrip(")").split(","))
        got = check_record(c, rec[c.key], ratios)
        assert got == want, (c.key, got)
        seen.add((c.key.split()[1], len(c.sic), got))
    ratios.check()
    want = {("mid", Np, ms) for Np in PADE_MID_NP[:3] for ms in PADE} | {("mid", 520, (3, 0)), ("mid", 520, (13, 20))}
    assert seen == want | {("low", Np, ms) for Np in PADE_EDGE_NP for ms in PADE}


def test_n_edges(alone):
    cases, rec = alone
    ratios = Ratios("n edges")
    seen = set()
    for c in cases["n"]:
        check_record(c, rec[c.key], ratios)
        seen.add((c.n, len(c.sic)))
    ratios.check()
    assert {(n, Np) for n in N_EDGES for Np in (17, 129)} | {(41, 100)} <= seen


def test_rejected_problems(lib_built):
    for c, info in rejected_cases():
        r = launch([c], c.max_pred)[0]
        assert r["info"] == info, (c.key, r["info"])
    # the same problems side by side in one launch
    cs = rejected_cases()
    rec = launch([c for c, _ in cs], 100)
    assert [int(v) for v in rec["info"]] == [info for _, info in cs]


def test_many_candidates(alone):
    cases, rec = alone
    ratios = Ratios("more than 256 candidates")
    for c in cases["candidates"]:
        r = rec[c.key]
        assert 256 < len(c.sic) + len(c.sst) and 64 < r["n_pred"] <= 520
        check_record(c, r, ratios)
    ratios.check()


def test_gradient(alone):
    cases, rec = alone
    ratios = Ratios("MLII gradient")
    for c in cases["grad"]:
        check_record(c, rec[c.key], ratios)
    ratios.check()


@pytest.fixture(scope="module")
def grid_runs(lib_built):
    cases = grid_cases()
    runs = {}
    for n_sig in GRID_NSIG:
        sigs = grid_sigs(n_sig)
        runs[n_sig] = [launch_grid([c], sigs, c.max_pred)[0] for c in cases]
    return cases, runs


def test_hyper_grid(grid_runs):
    cases, runs = grid_runs
    assert {nwu_of(c.n) for c in cases} == set(range(2, 9))
    ratios = Ratios("hyper-parameter grid")
    vs_forecast = Ratios("hyper-parameter grid vs forecast records")
    for n_sig, recs in runs.items():
        sigs = grid_sigs(n_sig)
        for c, g in zip(cases, recs):
            single = launch([dataclasses.replace(c, sig=float(s)) for s in sigs], c.max_pred)
            for k, s in enumerate(sigs):
                where = f"{c.key} n_sig={n_sig} sig={s:.3g}"
                check_record(c, g[k], ratios, sig=s, where=where)
                assert (g[k]["n_pred"], g[k]["expm_m"], g[k]["expm_s"], g[k]["info"]) == \
                    (single[k]["n_pred"], single[k]["expm_m"], single[k]["expm_s"], single[k]["info"])
                ref = fit(c, g[k]["expm_m"], g[k]["expm_s"], s)
                t = ge.bound(g[k]["expm_s"], ref["cond"])
                for f, scale in scales(ref, True).items():
                    vs_forecast.add(where, f, abs(float(g[k][f]) - float(single[k][f])) / scale, t)
    ratios.check()
    vs_forecast.check()


# ------------------------------------------------------------------------------------------------------------------
# batch and padding invariance
# ------------------------------------------------------------------------------------------------------------------
def same_bits(a, b):
    """Records equal bit for bit in every field but the cycle counters -> list of differing fields."""
    diff = []
    for f in VALUE_FIELDS:
        x, y = np.asarray(a[f]), np.asarray(b[f])
        if x.dtype.kind == "f":
            x, y = x.view(np.int64), y.view(np.int64)
        if not np.array_equal(x, y):
            diff.append(f)
    return diff


def test_batch_and_padding_invariance(alone):
    """Groups 1-4 in one launch, four copies of each (P > 2 x 148 CTAs, so the scratch slab of a CTA is reused by a
    smaller problem after a larger one: the order kernel starts the large problems first), at max_pred = 520 and 384:
    every record is bit-identical to the same problem launched on its own at its own max_pred.  At 384 the problems
    with more predictors report info = -2."""
    cases, rec = alone
    flat = [c for g in ("sweep", "pade", "n", "candidates", "grad") for c in cases[g]]
    batch = flat * 4
    assert len(batch) > 2 * 148
    for max_pred in (520, 384):
        out = launch(batch, max_pred)
        for i, c in enumerate(batch):
            r = out[i]
            ref = rec[c.key]
            if ref["n_pred"] > max_pred:
                assert r["info"] == -2 and r["n_pred"] == ref["n_pred"], c.key
                continue
            assert not same_bits(r, ref), (max_pred, i, c.key, same_bits(r, ref))


def test_grid_batch_and_padding_invariance(grid_runs):
    """Case 6's grid problems in one launch, at the tight ld and at max_pred = 520: bit-identical grid records."""
    cases, runs = grid_runs
    for n_sig, recs in runs.items():
        for max_pred in (132, 520):
            out = launch_grid(cases, grid_sigs(n_sig), max_pred)
            for c, g, alone_g in zip(cases, out, recs):
                for k in range(n_sig):
                    assert not same_bits(g[k], alone_g[k]), (n_sig, max_pred, c.key, k, same_bits(g[k], alone_g[k]))
