"""Host-side mirror of the script-level helpers every reference script re-defines -- `detrend`, `networks`,
`forecast` (+ nested `MLII`), `skill` -- with explicit arguments instead of module globals, plus the batched
retrospective sweep that is the headline workload (north/retrospective_forecasts/*_retro.py: years
fmin..fmax x init months x 3 regions).  All arithmetic runs in libsie_b200's kernels.

Reference lines: detrend north/June1st.py:179-194 (retro: June1st_retro.py:178-195); networks :196-206;
forecast :208-288; MLII :235-257; read_SIE de-trending June1st_retro.py:58-69; skill :293-314.
"""
from __future__ import annotations

import collections
import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from .config import CONFIGS, RULE_POS_SIG, ForecastConfig
from .engine import NetworkBatch, _ptr, _stream, h2d, r_crit_pearson, r_crit_ttest, require_cuda

FIRST_YEAR = 1979

GP_PROBLEM_DTYPE = np.dtype([("job_sic", "<i4"), ("job_sst", "<i4"), ("n", "<i4"), ("y_off", "<i4"),
                             ("rule", "<i4"), ("zscore", "<i4"), ("want_grad", "<i4"), ("pad_", "<i4"),
                             ("r_sel", "<f8"), ("ell", "<f8"), ("sig", "<f8")])
GP_RESULT_DTYPE = np.dtype([("fmean", "<f8"), ("fvar", "<f8"), ("sigma_f", "<f8"), ("nlml", "<f8"),
                            ("g_ell", "<f8"), ("g_sig", "<f8"), ("n_pred", "<i4"), ("expm_m", "<i4"),
                            ("expm_s", "<i4"), ("info", "<i4"), ("cycles_total", "<i8"), ("cycles_expm", "<i8")])
assert GP_PROBLEM_DTYPE.itemsize == C.sizeof(_lib.SieGpProblem)
assert GP_RESULT_DTYPE.itemsize == C.sizeof(_lib.SieGpResult)


# ------------------------------------------------------------------------------------------------
# single-call helpers (reference call surface)
# ------------------------------------------------------------------------------------------------
def detrend(data):
    """`detrend(dataset)` (north/June1st.py:179-194): (X,Y,T) -> (dt (X,Y,T), trend (X,Y,2))."""
    require_cuda()
    data = np.ascontiguousarray(data, dtype=np.float64)
    X, Y, T = data.shape
    n_upper = int((~np.isnan(data).any(axis=2)).sum())
    eng = NetworkBatch(X, Y, T, 1, latlon=False, n_upper=n_upper, keep_R=False, max_areas=1)
    fields = h2d(data.reshape(1, X * Y, T))
    jf = torch.zeros(1, dtype=torch.int32, device="cuda")
    jT = torch.full((1,), T, dtype=torch.int32, device="cuda")
    eng.detrend_zscore(fields, jf, jT, do_detrend=True)
    return (eng.dt[0].cpu().numpy().reshape(X, Y, T), eng.trend[0].cpu().numpy().reshape(X, Y, 2))


def networks(dt, area=None, lat=None, latlon=True, significance=0.01):
    """`networks(dataset, latlon)` (north/June1st.py:196-206) -> (nodes = V, anoms = anomaly)."""
    from .ComplexNetworks import Network
    net = Network(data=dt)
    Network.tau(net, significance)
    Network.area_level(net, latlon_grid=latlon)
    if latlon:
        Network.intra_links(net, lat=lat)
    else:
        Network.intra_links(net, area=area)
    return net.V, net.anomaly


def sie_detrend_tables(sie, fmin, fmax):
    """The de-trending arithmetic of `read_SIE` (north/retrospective_forecasts/June1st_retro.py:58-69): one OLS
    fit per end-year on the prefix window; `dt` rounded to 3 d.p., `trend` = [slope, intercept] un-rounded.
    O(years^2) scalar work on the host (not a kernel)."""
    rows = fmax - (fmin - 1) + 1
    trend = np.zeros((rows, 2))
    dt = np.zeros((rows, fmax - FIRST_YEAR + 1))
    sie = np.asarray(sie, dtype=np.float64)
    for year in range(fmin - 1, fmax + 1):
        n = year - FIRST_YEAR + 1
        x = np.arange(n, dtype=np.float64)
        y = sie[:n]
        xm, ym = x.mean(), y.mean()
        slope = np.mean((x - xm) * (y - ym)) / np.mean((x - xm) ** 2)
        icpt = ym - slope * xm
        trend[year - (fmin - 1)] = (slope, icpt)
        dt[year - (fmin - 1), :n] = y - (slope * x + icpt)
    return dt.round(3), trend


def skill(obs_rt, forecast_rt, obs_dt, forecast_dt):
    """`skill()` (north/retrospective_forecasts/June1st_retro.py:293-314): 1 - MSE/MSE_clim, 3 d.p."""
    a = np.mean((obs_rt - forecast_rt) ** 2)
    b = np.mean((obs_rt - np.nanmean(obs_rt)) ** 2)
    c = np.mean((obs_dt - forecast_dt) ** 2)
    d = np.mean((obs_dt - np.nanmean(obs_dt)) ** 2)
    return (1 - (a / b)).round(3), (1 - (c / d)).round(3)


# ------------------------------------------------------------------------------------------------
# batched GP
# ------------------------------------------------------------------------------------------------
def _series_args(sic, sst):
    """(anomaly, n_areas, MA, Tstride) of the SIC node series, then of the SST ones (null / 0 without SST): the series
    arguments of sie_gp_forecast and sie_gp_hyper_grid."""
    if sst is None:
        return _ptr(sic.anomaly), _ptr(sic.n_areas), sic.MA, sic.Tstride, C.c_void_p(0), C.c_void_p(0), 0, 0
    return (_ptr(sic.anomaly), _ptr(sic.n_areas), sic.MA, sic.Tstride,
            _ptr(sst.anomaly), _ptr(sst.n_areas), sst.MA, sst.Tstride)


class GpBatch:
    """P GP problems over one or two anomaly sets held by NetworkBatch objects."""

    def __init__(self, P, max_pred=256):
        require_cuda()
        self.lib = _lib.load()
        self.P = int(P)
        self.max_pred = int((max_pred + 3) // 4 * 4)
        self.scratch_bytes = int(self.lib.sie_gp_scratch_bytes(self.P, self.max_pred, 64))
        self.scratch = torch.empty((self.scratch_bytes + 7) // 8, dtype=torch.float64, device="cuda")
        self.out = torch.empty(self.P * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")

    def run(self, prob_dev, y_dev, sic: NetworkBatch, sst: NetworkBatch | None, pr=None, out=None):
        """`pr = (p0, p1)`: run only that range of problems (records p0..p1-1 of prob_dev / out); each range needs its
        own GpBatch when ranges run concurrently (the scratch holds the work queue); `out`: result buffer of the
        whole problem list (default: this batch's own)."""
        p0, p1 = (0, self.P) if pr is None else (int(pr[0]), int(pr[1]))
        out = self.out if out is None else out
        isz = GP_PROBLEM_DTYPE.itemsize
        osz = GP_RESULT_DTYPE.itemsize
        rc = self.lib.sie_gp_forecast(_ptr(prob_dev[p0 * isz:]), p1 - p0, _ptr(y_dev), *_series_args(sic, sst),
                                      self.max_pred, _ptr(out[p0 * osz:]), _ptr(self.scratch), self.scratch_bytes,
                                      _stream())
        _lib.check(rc, "sie_gp_forecast")

    def run_grid(self, prob_dev, sig_grid_dev, n_sig, y_dev, sic, sst, out, n=None):
        """Hyper-parameter grid: problem p fixes l = prob[p].ell; every sig_grid[k] is evaluated from the same
        expm / X Sigma X^T (sie_gp_hyper_grid).  `n`: run the first n <= P problems of prob_dev (default: P).  `out`:
        uint8 device buffer of n * n_sig result records."""
        n = self.P if n is None else int(n)
        assert 0 < n <= self.P
        rc = self.lib.sie_gp_hyper_grid(_ptr(prob_dev), n, _ptr(sig_grid_dev), int(n_sig), _ptr(y_dev),
                                        *_series_args(sic, sst), self.max_pred, _ptr(out), _ptr(self.scratch),
                                        self.scratch_bytes, _stream())
        _lib.check(rc, "sie_gp_hyper_grid")

    def results(self):
        return self.out.cpu().numpy().view(GP_RESULT_DTYPE)


_ELL_COL = GP_PROBLEM_DTYPE.fields["ell"][1] // 8        # `ell` as a float64 column of a problem record
assert GP_PROBLEM_DTYPE.itemsize % 8 == 0 and GP_PROBLEM_DTYPE.fields["ell"][1] % 8 == 0


def expand_problems(prob_dev, ell_dev, out):
    """`out` (uint8 device buffer of P * n_ell problem records) <- np.repeat(prob, n_ell) with copy i of every problem
    at l = ell_dev[i]: the problem list sie_gp_hyper_grid evaluates on an (l, sigma_n~) grid.  Built on the device from
    the first P records of `prob_dev` by copies into the preallocated `out` (no host round trip, no allocation), so a
    captured step replays it."""
    isz = GP_PROBLEM_DTYPE.itemsize
    nl = ell_dev.numel()
    P = out.numel() // (isz * nl)
    out.view(P, nl, isz).copy_(prob_dev[:P * isz].view(P, 1, isz).expand(P, nl, isz))
    out.view(torch.float64).view(P, nl, isz // 8)[:, :, _ELL_COL].copy_(ell_dev.view(1, nl).expand(P, nl))


def grid_select(grid_dev, prob_dev, P, ell_dev, sig_dev, tuned_dev, best_dev):
    """sie_gp_grid_select on the current stream: best_dev [P] (int32) <- flat index i * n_sig + j of the smallest
    admissible nlML of every problem's grid records grid_dev [P][n_ell][n_sig] (-1: none admissible), tuned_dev [P]
    <- prob_dev with (l, sigma_n~) = (ell_dev[i], sig_dev[j])."""
    rc = _lib.load().sie_gp_grid_select(_ptr(grid_dev), _ptr(prob_dev), int(P), _ptr(ell_dev), ell_dev.numel(),
                                        _ptr(sig_dev), sig_dev.numel(), _ptr(tuned_dev), _ptr(best_dev), _stream())
    _lib.check(rc, "sie_gp_grid_select")


class _GridBuffers:
    """Device buffers of one (ells x sigs) hyper-parameter grid over a sweep's P problems."""

    def __init__(self, ells, sigs, P):
        self.ells, self.sigs = ells, sigs
        self.ell_dev, self.sig_dev = h2d(ells), h2d(sigs)
        self.prob = torch.empty(P * len(ells) * GP_PROBLEM_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        self.out = torch.empty(P * len(ells) * len(sigs) * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        self.gp = None                # GpBatch of hyper_grid() (the whole problem list in one launch)


# (l, sigma_n~) a tuned sweep forecast with, and the flat grid index i * n_sig + j they came from (-1: the script's own)
SELECTION_DTYPE = np.dtype([("ell", "<f8"), ("sig", "<f8"), ("best", "<i4")])


def selection_records(tuned, best):
    sel = np.empty(len(best), dtype=SELECTION_DTYPE)
    sel["ell"], sel["sig"], sel["best"] = tuned["ell"], tuned["sig"], best
    return sel


# SieGpMarginal (include/sie_b200.h): what sie_gp_grid_marginal reports about each problem's grid posterior
GP_MARGINAL_DTYPE = np.dtype([("ess", "<f8"), ("w_max", "<f8"), ("n_admissible", "<i4"), ("argmax", "<i4")])
assert GP_MARGINAL_DTYPE.itemsize == C.sizeof(_lib.SieGpMarginal)
DEFAULT_QUANTILES = (0.05, 0.5, 0.95)


def _with_quantiles(recs, dtype, quant):
    """recs: `dtype` [N] (or its bytes), quant: float64 [N][n_q] -> `dtype`'s fields plus `quantiles` [N]."""
    recs = np.asarray(recs).view(dtype).reshape(-1)
    quant = np.asarray(quant, dtype=np.float64).reshape(-1)
    quant = quant.reshape(len(recs), quant.size // max(1, len(recs)))
    rec = np.empty(len(recs), dtype=np.dtype(dtype.descr + [("quantiles", "<f8", (quant.shape[1],))]))
    for f in dtype.names:
        rec[f] = recs[f]
    rec["quantiles"] = quant
    return rec


def marginal_dtype(n_q):
    """Per-problem record of a marginalised forecast: GP_MARGINAL_DTYPE's fields plus `quantiles`, a float64 sub-array
    of the n_q predictive quantiles (detrended).  Its length is the number of levels, hence a function of n_q."""
    return np.dtype(GP_MARGINAL_DTYPE.descr + [("quantiles", "<f8", (int(n_q),))])


def marginal_records(stats, quant):
    """stats: GP_MARGINAL_DTYPE [P] (or its bytes), quant: float64 [P][n_q] -> marginal_dtype(n_q) [P]."""
    return _with_quantiles(stats, GP_MARGINAL_DTYPE, quant)


def check_levels(quantiles):
    """-> the quantile levels as float64; raises ValueError unless every level lies strictly inside (0, 1)."""
    q = np.ascontiguousarray(quantiles, dtype=np.float64).reshape(-1)
    if not np.all((q > 0.0) & (q < 1.0)):
        raise ValueError(f"quantile levels must lie strictly between 0 and 1, got {q.tolist()}")
    return q


def grid_marginal(grid_dev, P, n_grid, q_dev, out_dev, stats_dev, quant_dev):
    """sie_gp_grid_marginal on the current stream: out_dev [P] (GP records) <- the marginal-likelihood-weighted mixture
    of every problem's grid records grid_dev [P][n_grid], stats_dev [P] (GP_MARGINAL_DTYPE) <- ESS, largest weight,
    |A| and its index, quant_dev [P][n_q] <- the mixture's quantiles at the levels q_dev [n_q] (q_dev None: none)."""
    n_q = 0 if q_dev is None else q_dev.numel()
    null = C.c_void_p(0)
    rc = _lib.load().sie_gp_grid_marginal(_ptr(grid_dev), int(P), int(n_grid), _ptr(q_dev) if n_q else null, n_q,
                                          _ptr(out_dev), _ptr(stats_dev), _ptr(quant_dev) if n_q else null, _stream())
    _lib.check(rc, "sie_gp_grid_marginal")


# SieGpEnsemble (include/sie_b200.h): one ensemble problem's pooled predictive distribution (sie_gp_ensemble)
GP_ENSEMBLE_DTYPE = np.dtype([("fmean", "<f8"), ("fvar", "<f8"), ("var_within", "<f8"), ("var_between", "<f8"),
                              ("n_members", "<i4"), ("pad_", "<i4")])
assert GP_ENSEMBLE_DTYPE.itemsize == C.sizeof(_lib.SieGpEnsemble) == 40


def ensemble_records(pooled, quant):
    """pooled: GP_ENSEMBLE_DTYPE [E] (or its bytes), quant: float64 [E][n_q] -> GP_ENSEMBLE_DTYPE's fields plus
    `quantiles` (float64 [n_q], detrended) per ensemble problem."""
    return _with_quantiles(pooled, GP_ENSEMBLE_DTYPE, quant)


def gp_ensemble_scratch_bytes(E, M, n_grid):
    return int(_lib.load().sie_gp_ensemble_scratch_bytes(int(E), int(M), int(n_grid)))


def gp_ensemble(rec_dev, E, M, n_grid, q_dev, out_dev, quant_dev, scratch_dev):
    """sie_gp_ensemble on the current stream: out_dev [E] (GP_ENSEMBLE_DTYPE) <- the pool of the M members' records
    rec_dev [E][M][n_grid] of every ensemble problem, quant_dev [E][n_q] <- its quantiles at the levels q_dev [n_q]
    (q_dev None: none).  scratch_dev: at least gp_ensemble_scratch_bytes(E, M, n_grid) bytes."""
    n_q = 0 if q_dev is None else q_dev.numel()
    null = C.c_void_p(0)
    rc = _lib.load().sie_gp_ensemble(_ptr(rec_dev), int(E), int(M), int(n_grid), _ptr(q_dev) if n_q else null, n_q,
                                     _ptr(out_dev), _ptr(quant_dev) if n_q else null, _ptr(scratch_dev),
                                     scratch_dev.numel() * scratch_dev.element_size(), _stream())
    _lib.check(rc, "sie_gp_ensemble")


def ensemble_slots(plan, n_members):
    """The ensemble problems of a single-rank SweepPlan and where its records go in an ensemble store
    [E][n_members][n_grid]: (meta int64 [E][3] = the sorted (config index, region index, year) triples, rows int64 [P]
    = e * n_members + member of every problem, in the plan's current problem order, partition_sst's included)."""
    meta = np.array(sorted({tuple(int(v) for v in m) for m in plan.prob_meta}), dtype=np.int64).reshape(-1, 3)
    e_of = {tuple(m): e for e, m in enumerate(meta.tolist())}
    rows = np.array([e_of[tuple(int(v) for v in m)] * int(n_members) + int(mb)
                     for m, mb in zip(plan.prob_meta, plan.prob_member)], dtype=np.int64)
    return meta, rows


class _SeriesSet:
    """Node series of ONE network given as a dict (the reference's `dataset['anoms']`), packed the way GpBatch reads a
    NetworkBatch: anomaly [1][nA][n+1], n_areas [1]."""

    def __init__(self, anoms, n):
        keys = list(anoms)
        arr = np.zeros((1, max(1, len(keys)), n + 1))
        for a, k in enumerate(keys):
            arr[0, a] = np.asarray(anoms[k], dtype=np.float64)[:n + 1]
        self.anomaly = h2d(arr)
        self.n_areas = torch.tensor([len(keys)], dtype=torch.int32, device="cuda")
        self.MA = arr.shape[1]
        self.Tstride = n + 1


class _OneProblem:
    """One forecast problem from node series given as dicts (the reference's `dataset['anoms']`) on the device: its
    targets `y`, node series `s1` (SIC) and `s2` (SST, None without), host problem record `prob` [1] (l, sigma_n~ left
    0) and `gp`, a GpBatch of P problems sized for its predictors."""

    def __init__(self, y, anoms_sic, anoms_sst, rule, alpha, zscore, want_grad, P=1):
        require_cuda()
        y = np.asarray(y, dtype=np.float64).reshape(-1)
        n = y.size
        self.y = h2d(y)
        self.s1 = _SeriesSet(anoms_sic, n)
        self.s2 = _SeriesSet(anoms_sst, n) if anoms_sst is not None else None
        self.prob = np.zeros(1, dtype=GP_PROBLEM_DTYPE)
        self.prob["job_sic"] = 0
        self.prob["job_sst"] = 0 if anoms_sst is not None else -1
        self.prob["n"] = n
        self.prob["rule"] = rule
        self.prob["zscore"] = int(zscore)
        self.prob["want_grad"] = int(want_grad)
        self.prob["r_sel"] = r_crit_pearson(n, alpha) if rule == RULE_POS_SIG else 0.0
        npred = self.s1.MA + (self.s2.MA if self.s2 is not None else 0)
        self.gp = GpBatch(P, max_pred=max(4, npred))


def forecast(y, anoms_sic, anoms_sst=None, rule=0, alpha=0.05, zscore=False, ell=1.0, sig=1.0, want_grad=False):
    """One GP forecast from node series given as dicts (the reference's `dataset['anoms']`), i.e. the body of
    `forecast()` for one region (north/June1st.py:214-277).  Returns the raw result record."""
    one = _OneProblem(y, anoms_sic, anoms_sst, rule, alpha, zscore, want_grad)
    one.prob["ell"] = ell
    one.prob["sig"] = sig
    one.gp.run(h2d(one.prob.view(np.uint8)), one.y, one.s1, one.s2)
    return one.gp.results()[0]


def _grid_on_device(y, anoms_sic, anoms_sst, rule, alpha, zscore, ells, sigs, want_grad):
    """One problem's (l, sigma_n~) grid records, left on the device: (uint8 buffer of [len(ells)][len(sigs)] records,
    ells, sigs); ells / sigs None are the reference's grids."""
    ells = np.logspace(-7, 2, 20) if ells is None else np.asarray(ells, dtype=np.float64)
    sigs = np.logspace(-3, 9, 20) if sigs is None else np.asarray(sigs, dtype=np.float64)
    one = _OneProblem(y, anoms_sic, anoms_sst, rule, alpha, zscore, want_grad, P=len(ells))
    prob = np.repeat(one.prob, len(ells))
    prob["ell"] = ells
    out = torch.empty(len(ells) * len(sigs) * GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    one.gp.run_grid(h2d(prob.view(np.uint8)), h2d(sigs), len(sigs), one.y, one.s1, one.s2, out)
    return out, ells, sigs


def hyper_grid(y, anoms_sic, anoms_sst=None, rule=0, alpha=0.05, zscore=False, ells=None, sigs=None, want_grad=False):
    """Grid search over the reference's hyper-parameter grids `ls = np.logspace(-7,2,20)`, `ss = np.logspace(-3,9,20)`
    (north/June1st.py:210-211; the `minimize(MLII, ...)` call at :259-262 is commented out there): negative log marginal
    likelihood of MLII() for every (l, sigma_n~) pair, one expm per l.
    Returns (records [len(ells)][len(sigs)], (i, j) of the smallest finite nlML)."""
    out, ells, sigs = _grid_on_device(y, anoms_sic, anoms_sst, rule, alpha, zscore, ells, sigs, want_grad)
    rec = out.cpu().numpy().view(GP_RESULT_DTYPE).reshape(len(ells), len(sigs))
    nl = np.where((rec["info"] == 0) & np.isfinite(rec["nlml"]), rec["nlml"], np.inf)
    best = np.unravel_index(int(np.argmin(nl)), nl.shape)
    return rec, (int(best[0]), int(best[1]))


def marginal_forecast(y, anoms_sic, anoms_sst=None, rule=0, alpha=0.05, zscore=False, ells=None, sigs=None,
                      quantiles=DEFAULT_QUANTILES):
    """The forecast averaged over the (l, sigma_n~) grid (hyper_grid's problem and grids), every grid point weighted by
    its marginal likelihood, on the device (sie_gp_grid_marginal).  Returns (record, stats, quantiles): the GP record
    with the mixture's fmean / fvar and nlml = -log of the grid-averaged marginal likelihood (the other fields are the
    largest-weight point's), GP_MARGINAL_DTYPE stats (ESS, largest weight, |A|, its flat index), and the mixture's
    predictive quantiles at `quantiles` (detrended; NaN where no grid point is admissible)."""
    q = check_levels(quantiles)
    out, ells, sigs = _grid_on_device(y, anoms_sic, anoms_sst, rule, alpha, zscore, ells, sigs, False)
    rec = torch.empty(GP_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    stats = torch.empty(GP_MARGINAL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    quant = torch.empty(max(1, q.size), dtype=torch.float64, device="cuda")
    grid_marginal(out, 1, len(ells) * len(sigs), h2d(q) if q.size else None, rec, stats, quant)
    return (rec.cpu().numpy().view(GP_RESULT_DTYPE)[0], stats.cpu().numpy().view(GP_MARGINAL_DTYPE)[0],
            quant.cpu().numpy()[:q.size])


def mlii(theta, y, anoms_sic, anoms_sst=None, rule=0, alpha=0.05, zscore=False):
    """`MLII(hyperparameters)` (north/June1st.py:235-257): theta = (log l, log sigma_n~) ->
    (nlML, [d/dtheta1, d/dtheta2]); (inf, [inf, inf]) when the kernel matrix is not SPD."""
    r = forecast(y, anoms_sic, anoms_sst, rule, alpha, zscore, float(np.exp(theta[0])), float(np.exp(theta[1])),
                 want_grad=True)
    if r["info"] != 0:
        return np.inf, np.asarray([np.inf, np.inf])
    return np.float64(r["nlml"]), np.asarray([r["g_ell"], r["g_sig"]])


class MliiObjective:
    """`MLII(hyperparameters)` of one forecast problem as a callable for an optimiser: the node series and targets are
    uploaded once, every call evaluates the negative log marginal likelihood and its gradient on the device."""

    def __init__(self, y, anoms_sic, anoms_sst=None, rule=0, alpha=0.05, zscore=False):
        self.one = _OneProblem(y, anoms_sic, anoms_sst, rule, alpha, zscore, True)
        self.evaluations = 0

    def record(self, theta):
        one = self.one
        one.prob["ell"] = float(np.exp(theta[0]))
        one.prob["sig"] = float(np.exp(theta[1]))
        one.gp.run(h2d(one.prob.view(np.uint8)), one.y, one.s1, one.s2)
        self.evaluations += 1
        return one.gp.results()[0]

    def __call__(self, theta):
        r = self.record(theta)
        if r["info"] != 0 or not np.isfinite(r["nlml"]):
            return np.inf, np.asarray([np.inf, np.inf])            # the `except` branch of MLII, north/June1st.py:254-256
        return float(r["nlml"]), np.asarray([r["g_ell"], r["g_sig"]], dtype=np.float64)


def optimise_hyperparameters(y, anoms_sic, anoms_sst=None, rule=0, alpha=0.05, zscore=False, ell0=None, sig0=None,
                             from_grid=False):
    """The hyper-parameter optimisation the reference leaves commented out (north/June1st.py:259-262):
        theta = minimize(MLII, x0=[log(l_init), log(sigma_init)], method='CG', jac=True, options={'disp': False}).x
    with MLII and its gradient evaluated on the device.  `from_grid`: start from the minimum of the 20 x 20
    (l, sigma_n~) grid of :210-211 instead of (ell0, sig0).  Returns (l, sigma_n~, scipy OptimizeResult)."""
    from scipy.optimize import minimize
    if from_grid:
        ells, sigs = np.logspace(-7, 2, 20), np.logspace(-3, 9, 20)
        _, (i, j) = hyper_grid(y, anoms_sic, anoms_sst, rule, alpha, zscore, ells, sigs)
        ell0, sig0 = ells[i], sigs[j]
    obj = MliiObjective(y, anoms_sic, anoms_sst, rule, alpha, zscore)
    res = minimize(obj, x0=[np.log(ell0), np.log(sig0)], method="CG", jac=True, options={"disp": False})
    res.evaluations = obj.evaluations
    return float(np.exp(res.x[0])), float(np.exp(res.x[1])), res


# ------------------------------------------------------------------------------------------------
# retrospective sweep
# ------------------------------------------------------------------------------------------------
class SweepPlan:
    """Host-only bookkeeping of a retrospective sweep: which network builds (jobs) and which GP problems exist,
    in the year/row indexing of the reference scripts (June1st_retro.py:199-290; south January1st_retro.py:173-182
    for the previous-year variant).  `members` > 1: an ensemble of input realisations (perturbed SIC / SST fields,
    shared SIE targets; BASELINE.json configs[4]) in ONE batch -- member m's networks read field m * n_configs + ci.
    `rank`/`world` shard whole (member, config, year) tasks -- a task owns its network build(s) and its three regional
    forecasts, so shards exchange nothing."""

    def __init__(self, config_names, sie, fmin, fmax, significance=0.01, rank=0, world=1, members=1):
        self.cfgs = [CONFIGS[c] if isinstance(c, str) else c for c in config_names]
        self.fmin, self.fmax = int(fmin), int(fmax)
        self.years = list(range(self.fmin, self.fmax + 1))
        self.significance = significance
        self.rank, self.world = int(rank), int(world)
        self.members = int(members)
        self.use_sst = any(c.use_sst for c in self.cfgs)
        ncfg = len(self.cfgs)
        # tasks in a fixed global order, longest windows first (the slowest network builds: the device pops jobs in
        # this order, LPT) so round-robin shards are balanced too
        tasks = [(m, ci, year) for year in reversed(self.years) for m in range(self.members) for ci in range(ncfg)]
        self.all_tasks = tasks
        self.tasks = [t for i, t in enumerate(tasks) if i % self.world == self.rank]
        self.jobs_m, self.job_index = [], {}        # SIC network builds: (member, cfg index, network year)
        self.sst_jobs, self.sst_index = [], {}      # SST network builds: (member, target year)
        for m, ci, year in self.tasks:
            cfg = self.cfgs[ci]
            ny = year - 1 if cfg.prev_year_network else year
            if (m, ci, ny) not in self.job_index:
                self.job_index[(m, ci, ny)] = len(self.jobs_m)
                self.jobs_m.append((m, ci, ny))
            if cfg.use_sst and (m, year) not in self.sst_index:
                self.sst_index[(m, year)] = len(self.sst_jobs)
                self.sst_jobs.append((m, year))
        self.jobs = [(ci, ny) for _, ci, ny in self.jobs_m]          # (cfg index, network year) per SIC job
        self.job_member = np.array([m for m, _, _ in self.jobs_m], dtype=np.int32)
        self.sst_years = [y for _, y in self.sst_jobs]
        self.sst_member = np.array([m for m, _ in self.sst_jobs], dtype=np.int32)
        self.job_field = np.array([m * ncfg + ci for m, ci, _ in self.jobs_m], dtype=np.int32)
        self.job_T = np.array([ny - FIRST_YEAR + 1 for _, _, ny in self.jobs_m], dtype=np.int32)
        self.rcrit = np.array([r_crit_ttest(int(T), significance) for T in self.job_T])
        self.sst_T = np.array([y - FIRST_YEAR + 1 for y in self.sst_years], dtype=np.int32)
        self.sst_rcrit = np.array([r_crit_ttest(int(T), significance) for T in self.sst_T])
        self.sie = {k: np.asarray(v, dtype=np.float64) for k, v in sie.items()}
        self.sie_dt, self.sie_trend = {}, {}
        for reg, series in self.sie.items():
            self.sie_dt[reg], self.sie_trend[reg] = sie_detrend_tables(series, self.fmin, self.fmax)
        probs, ys, self.prob_meta, prob_member = [], [], [], []
        y_off = 0
        for m, ci, year in self.tasks:
            cfg = self.cfgs[ci]
            for k, reg in enumerate(cfg.regions):
                row = year - (self.fmin - 1) - 1
                if cfg.prev_year_network:
                    y = self.sie_dt[reg][row, 1:year - FIRST_YEAR]          # south January1st_retro.py:175
                else:
                    y = self.sie_dt[reg][row, 0:year - FIRST_YEAR]          # June1st_retro.py:220
                n = y.size
                ny = year - 1 if cfg.prev_year_network else year
                p = np.zeros(1, dtype=GP_PROBLEM_DTYPE)
                p["job_sic"] = self.job_index[(m, ci, ny)]
                p["job_sst"] = self.sst_index[(m, year)] if cfg.use_sst else -1
                p["n"] = n
                p["y_off"] = y_off
                p["rule"] = cfg.rule[k]
                p["zscore"] = int(cfg.zscore)
                p["r_sel"] = r_crit_pearson(n, cfg.alpha) if cfg.rule[k] == RULE_POS_SIG else 0.0
                p["ell"] = cfg.ell[k]
                p["sig"] = cfg.sig[k]
                probs.append(p)
                ys.append(y)
                y_off += n
                self.prob_meta.append((ci, k, year))
                prob_member.append(m)
        self.prob_member = np.array(prob_member, dtype=np.int32)
        self.prob = np.concatenate(probs) if probs else np.zeros(0, dtype=GP_PROBLEM_DTYPE)
        self.y = np.concatenate(ys) if ys else np.zeros(0)
        self.P = len(probs)

    def partition_sst(self, ranges):
        """Stable partition of the problems inside every range (p0, p1): those that read no SST network first, the
        SST-reading ones last.  Records are self-contained (job indices, y_off), so this only permutes `prob` and
        `prob_meta` together; assemble() finds results through `prob_meta`.  Returns the split point of every range."""
        perm = np.arange(self.P)
        splits = []
        for (p0, p1) in ranges:
            idx = np.arange(p0, p1)
            uses = self.prob["job_sst"][idx] >= 0
            perm[p0:p1] = np.concatenate([idx[~uses], idx[uses]])
            splits.append(int(p0 + (~uses).sum()))
        self.prob = np.ascontiguousarray(self.prob[perm])
        self.prob_meta = [self.prob_meta[i] for i in perm]
        self.prob_member = self.prob_member[perm]
        return splits

    def assemble(self, raw, meta=None, member=None, selection=None, marginal=None):
        """-> {config: {region_fmean / _fvar / _fmean_rt: array(years)}} like the reference's GPR dict
        (June1st_retro.py:284-290, rounded to 3 d.p.), the un-rounded values under '<region>_raw_*'.
        `raw`/`meta`/`member` may be the concatenation over all ranks (after a gather).  With `members` > 1 the result
        is a list of such dicts, one per ensemble member.  `selection` (SELECTION_DTYPE, aligned with `raw`; tuned
        sweeps): also '<region>_ell' / '_sig', the hyper-parameters each forecast used, and '<region>_grid_index', the
        flat grid index they came from (-1: the script's own setting was kept).  `marginal` (marginal_dtype(n_q),
        aligned with `raw`; marginalised sweeps): also '<region>_grid_index' (the largest-weight grid point, -1: none
        admissible), '_ess', '_w_max', '_quantiles' (array(years, n_q), detrended) and '_quantiles_rt' (the same
        re-trended like '_raw_fmean_rt')."""
        meta = self.prob_meta if meta is None else meta
        member = self.prob_member if member is None else np.asarray(member)
        raw = np.asarray(raw)
        if self.members > 1:
            marr = np.asarray(meta, dtype=np.int64).reshape(-1, 3)
            return [self._assemble_one(raw[member == mm], marr[member == mm],
                                       None if selection is None else np.asarray(selection)[member == mm],
                                       None if marginal is None else np.asarray(marginal)[member == mm])
                    for mm in range(self.members)]
        return self._assemble_one(raw, meta, selection, marginal)

    def _assemble_one(self, raw, meta, selection=None, marginal=None, ensemble=None):
        m = np.asarray(meta, dtype=np.int64).reshape(-1, 3)
        out = {}
        if m.shape[0] == 0:
            return out
        ci_a, k_a, year_a = m[:, 0], m[:, 1], m[:, 2]
        fmean_raw, fvar_raw = raw["fmean"].astype(np.float64), raw["fvar"].astype(np.float64)
        fmean = np.round(fmean_raw, 3)
        fvar = np.round(fvar_raw, 3)
        for ci, cfg in enumerate(self.cfgs):
            for k, reg in enumerate(cfg.regions):
                sel = np.nonzero((ci_a == ci) & (k_a == k))[0]
                if sel.size == 0:
                    continue
                g = out.setdefault(cfg.name, {})
                years = year_a[sel]
                row = years - (self.fmin - 1) - 1
                tr = self.sie_trend[reg][row]                        # (slope, intercept) of that year's window
                line_last = (years - FIRST_YEAR) * tr[:, 0] + tr[:, 1]   # lineT[-1], June1st_retro.py:285-286
                i = years - self.fmin
                items = [("_fmean", fmean[sel]), ("_fvar", fvar[sel]), ("_fmean_rt", np.round(fmean[sel] + line_last, 3)),
                         ("_raw_fmean", fmean_raw[sel]), ("_raw_fvar", fvar_raw[sel]),
                         ("_raw_fmean_rt", fmean_raw[sel] + line_last)]
                if selection is not None:
                    items += [("_ell", selection["ell"][sel]), ("_sig", selection["sig"][sel]),
                              ("_grid_index", selection["best"][sel])]
                if marginal is not None:
                    qs = marginal["quantiles"][sel]
                    items += [("_grid_index", marginal["argmax"][sel]), ("_ess", marginal["ess"][sel]),
                              ("_w_max", marginal["w_max"][sel]), ("_quantiles", qs),
                              ("_quantiles_rt", qs + line_last[:, None])]
                if ensemble is not None:
                    qs = ensemble["quantiles"][sel]
                    items += [("_var_within", ensemble["var_within"][sel]),
                              ("_var_between", ensemble["var_between"][sel]),
                              ("_n_members", ensemble["n_members"][sel]), ("_quantiles", qs),
                              ("_quantiles_rt", qs + line_last[:, None])]
                for key, val in items:
                    arr = g.setdefault(reg + key, np.full((len(self.years),) + np.shape(val)[1:], np.nan))
                    arr[i] = val
        return out

    def skill(self, gpr):
        """skill() of the retro scripts (June1st_retro.py:293-314) from an assembled GPR dict."""
        out = {}
        for cfg in self.cfgs:
            rt, dt_ = [], []
            for reg in cfg.regions:
                obs_dt = np.array([self.sie_dt[reg][t - (self.fmin - 1), t - FIRST_YEAR] for t in self.years])
                obs_rt = self.sie[reg][self.fmin - FIRST_YEAR:self.fmax - FIRST_YEAR + 1]
                a, b = skill(obs_rt, gpr[cfg.name][reg + "_fmean_rt"], obs_dt, gpr[cfg.name][reg + "_fmean"])
                rt.append(a)
                dt_.append(b)
            out[cfg.name] = (rt, dt_)
        return out


def _members(x, n):
    """One member's input or a list (tuple) of them -> a list; a single input stands for all n members."""
    return list(x) if isinstance(x, (list, tuple)) else [x] * n


# One GP launch of a sweep step: its wave, its problems p0..p1-1, whether it reads SST networks (it then also waits for
# them and runs on its wave's SST stream) and the GpBatch whose scratch it runs on
_Launch = collections.namedtuple("_Launch", "wave p0 p1 sst gp")
# A step's schedule: its waves (job range, SST job range, problem range) and its GP launches in enqueue order
_Plan = collections.namedtuple("_Plan", "waves launches")


class RetrospectiveSweep:
    """years fmin..fmax x the given init-month configs x 3 regions, in one device-resident batch.

    sic_fields : dict config-name -> (X, Y, Tfull) raw monthly SIC of that init's data month, or a LIST of such dicts:
                 one per ensemble member (perturbed realisations, BASELINE.json configs[4]); all members run in one
                 device batch, so the latency-bound domain-growth chains of different members overlap
    sst_field  : (Xs, Ys, Tfull) raw May SST (only used by configs with use_sst) or None; a list (one per member) when
                 sic_fields is a list
    sie        : dict region -> (Tfull,) September (or target-month) extent
    psar / sst_lat : weights for intra_links (cell area for the polar grid, latitude grid for SST)
    hyper_grid : None (every forecast at its script's (l, sigma_n~)) or (ells, sigs): tuned sweep -- every forecast at
                 the minimum of MLII's nlML over the ells x sigs grid of its own problem (type-II maximum likelihood on
                 the grid, the search north/June1st.py:210-211 / :259-262 sets up), chosen on the device within the step;
                 a problem with no admissible grid point keeps its script's setting
    hyper_mode : with hyper_grid: "argmin" (the default: the tuned sweep above) or "marginal" -- every forecast is the
                 average of its problem's forecasts at all grid points, each weighted by its marginal likelihood
                 (sie_gp_grid_marginal: a uniform prior over the admissible grid points; the variance includes the
                 spread of the grid means); the step runs the grid and that one reduction, no second forecast
    quantiles  : marginal mode: levels in (0, 1) of the predictive quantiles to compute from each forecast's mixture
                 (self.marginal["quantiles"], '<region>_quantiles' of the assembled dict)
    """

    def __init__(self, config_names, sic_fields, sie, fmin, fmax, psar, sst_field=None, sst_lat=None,
                 significance=0.01, max_areas=None, max_pred=384, rank=0, world=1, wave_T=(12,), keep_R=True,
                 hyper_grid=None, hyper_mode=None, quantiles=()):
        if hyper_mode is not None and hyper_grid is None:
            raise ValueError("hyper_mode needs a hyper_grid")
        hyper_mode = "argmin" if hyper_mode is None else hyper_mode
        if hyper_mode not in ("argmin", "marginal"):
            raise ValueError(f"hyper_mode must be 'argmin' or 'marginal', got {hyper_mode!r}")
        levels = check_levels(quantiles)
        if levels.size and hyper_mode != "marginal":
            raise ValueError("quantiles are computed by marginal sweeps only (hyper_mode='marginal')")
        require_cuda()
        member_fields = _members(sic_fields, 1)
        self.members = len(member_fields)
        self.plan = plan = SweepPlan(config_names, sie, fmin, fmax, significance, rank, world, members=self.members)
        self.cfgs, self.years, self.fmin, self.fmax = plan.cfgs, plan.years, plan.fmin, plan.fmax
        self.X, self.Y, self.Tfull = np.shape(member_fields[0][self.cfgs[0].name])
        assert self.Tfull >= self.fmax - FIRST_YEAR + 1
        self.sic_host = self._stack_sic(member_fields)      # [member * n_configs + ci]
        self.psar_host = np.sqrt(np.asarray(psar, dtype=np.float64)).reshape(-1)     # ComplexNetworks.py:298-299
        self.use_sst = plan.use_sst and len(plan.sst_years) > 0
        # node capacity: a cell is a node of window T when its first T samples are NaN-free (detrend() fits the prefix),
        # so the count is largest for the SHORTEST window of the sweep -- a cell whose only NaN lies in a later year
        # is a node of the early windows
        Tmin = int(plan.job_T.min()) if len(plan.job_T) else self.Tfull
        n_upper = int(max((~np.isnan(f[:, :Tmin]).any(axis=1)).sum() for f in self.sic_host))
        # keep_R=False: the correlation matrices are never stored (tau-only K2); domain growth recomputes every
        # correlation it consumes from the unit-norm rows -- for grids whose N x N matrices do not fit in HBM
        self.sic = NetworkBatch(self.X, self.Y, self.Tfull, max(1, len(plan.jobs)), latlon=False, n_upper=n_upper,
                                max_areas=max_areas, keep_R=keep_R)
        self.sst = None
        if self.use_sst:
            self.Xs, self.Ys = np.shape(_members(sst_field, 1)[0])[:2]
            self.sst_host = self._stack_sst(sst_field)
            self.lat_host = np.sqrt(np.cos(np.radians(np.asarray(sst_lat, dtype=np.float64)))).reshape(-1)  # :296-297
            Tmin_s = int(plan.sst_T.min())
            n_up = int(max((~np.isnan(f[:, :Tmin_s]).any(axis=1)).sum() for f in self.sst_host))
            self.sst = NetworkBatch(self.Xs, self.Ys, self.Tfull, len(plan.sst_years), latlon=True, n_upper=n_up,
                                    max_areas=max_areas, keep_R=keep_R)
        self.P = plan.P
        self.n_forecasts = plan.P
        self._grids = {}                       # (ells, sigs) -> _GridBuffers (hyper_grid() and the tuned step)
        self.tune = None
        self.hyper_mode = hyper_mode if hyper_grid is not None else None
        self.levels = levels
        self.selection = None                  # tuned mode: SELECTION_DTYPE [P] of the step last read back
        self.marginal = None                   # marginal mode: marginal_dtype(n_q) [P] of the step last read back
        if hyper_grid is not None:
            ells, sigs = (np.ascontiguousarray(a, dtype=np.float64).reshape(-1) for a in hyper_grid)
            if ells.size < 1 or sigs.size < 1 or self.P < 1:
                raise ValueError("hyper_grid needs at least one l and one sigma_n~ value and a sweep with problems")
            self.tune = self._grid_buffers(ells, sigs)
            if hyper_mode == "argmin":
                self._tuned = torch.empty(self.P * GP_PROBLEM_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
                self._best = torch.empty(self.P, dtype=torch.int32, device="cuda")
            else:
                self._q_dev = h2d(levels) if levels.size else None
                self._mstats = torch.empty(self.P * GP_MARGINAL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
                self._quant = torch.empty(max(1, self.P * levels.size), dtype=torch.float64, device="cuda")
        # Waves.  Jobs and GP problems are ordered by descending year, so splitting the window lengths at `wave_T` edges
        # gives contiguous job / problem ranges: wave 0 = the longest windows (slowest domain growth, small GP problems),
        # the last wave = the shortest windows (networks finish early; their many small areas give the expensive
        # 100-160-predictor GP problems).  Every wave runs its chain on its own stream and its GP starts as soon as ITS
        # networks are done, overlapping the domain growth of the longer-window waves.
        edges = sorted({int(e) for e in (wave_T if isinstance(wave_T, (tuple, list)) else (wave_T,))}, reverse=True)
        self.wave_T = tuple(edges)
        T = plan.job_T
        prob_T = plan.job_T[plan.prob["job_sic"]] if plan.P else np.zeros(0, dtype=np.int32)

        def cuts(values):                      # descending `values` -> range boundaries [0, c1, c2, ..., len]
            values = np.asarray(values)
            return [0] + [int((values > e).sum()) for e in edges] + [len(values)]

        jc, pc = cuts(T), cuts(prob_T)
        sc = cuts(plan.sst_T) if self.use_sst else [0] * (len(edges) + 2)
        ok = plan.P > 0 and bool((np.diff(T) <= 0).all()) and bool((np.diff(prob_T) <= 0).all())
        if self.use_sst:
            ok = ok and bool((np.diff(plan.sst_T) <= 0).all())
        self.waves = []                        # (job range, sst range, problem range), longest windows first
        for w in range(len(edges) + 1):
            jr, sr, pr = (jc[w], jc[w + 1]), (sc[w], sc[w + 1]), (pc[w], pc[w + 1])
            if jr[1] > jr[0] or pr[1] > pr[0]:
                self.waves.append((jr, sr, pr))
        if ok and self.use_sst and plan.P:     # a wave's problems may only read SST networks of the same or a shorter-window wave
            for (jr, sr, pr) in self.waves:
                ps = plan.prob["job_sst"][pr[0]:pr[1]]
                ok = ok and bool((ps[ps >= 0] >= sr[0]).all())
        if ok and plan.P:                      # ... and SIC networks of the same or a shorter-window wave (previous-year configs)
            for (jr, sr, pr) in self.waves:
                ok = ok and bool((plan.prob["job_sic"][pr[0]:pr[1]] >= jr[0]).all())
        self.multi_wave = bool(ok and len(self.waves) > 1)
        # The launch plan of a step, built here so that compute() only walks it and allocates nothing: the waves (job,
        # SST job and problem ranges) and the GP launches in enqueue order.  Within a wave of a multi-wave step the
        # problems that read no SST network come first: they only wait for the wave's SIC networks, the SST-reading ones
        # (June) also for its SST networks, which finish later - two GP launches per wave instead of one that waits for
        # everything (13.0 -> 12.5 ms, DESIGN.md section 6).  Records are self-contained (y_off), so this is a
        # permutation of plan.prob / plan.prob_meta; assemble() looks results up through prob_meta.
        self.gp_sst = self.multi_wave and self.use_sst          # the SST split is on
        ranges = [pr for (_, _, pr) in self.waves]
        splits = plan.partition_sst(ranges) if self.gp_sst else [p1 for (_, p1) in ranges]
        # a grid-mode launch runs (p1 - p0) * n_ell grid problems on its batch, whose scratch also serves its forecast
        n_ell = 1 if self.tune is None else len(self.tune.ells)
        # the launch from problem 0 runs on self.gp, sized for all P so that the one-wave plan reuses it; self.gp.out
        # receives every launch's records
        self.gp = GpBatch(max(1, self.P) * n_ell, max_pred=max_pred)
        self._one_wave = _Plan([((0, self.sic.B), (0, self.sst.B if self.use_sst else 0), (0, self.P))],
                               [_Launch(0, 0, self.P, self.use_sst, self.gp)] if self.P else [])
        self._plan = self._one_wave
        if self.multi_wave:
            launches = []
            for w in range(len(ranges) - 1, -1, -1):
                p0, p1 = ranges[w]
                for lo, hi, sst in ((p0, splits[w], False), (splits[w], p1, True)):
                    if hi > lo:
                        gp = self.gp if lo == 0 else GpBatch((hi - lo) * n_ell, max_pred=max_pred)
                        launches.append(_Launch(w, lo, hi, sst, gp))
            self._plan = _Plan(self.waves, launches)
        self._streams = [(torch.cuda.Stream(priority=-1), torch.cuda.Stream(priority=-1)) for _ in self._plan.waves]
        plans = (self._plan, self._one_wave)   # steps run one at a time: the plans share their domain-growth scratch
        self.sic.prepare(*[[jr for (jr, _, _) in p.waves] for p in plans])
        if self.use_sst:
            self.sst.prepare(*[[sr for (_, sr, _) in p.waves] for p in plans])
        self._graph = None
        self.use_graph = False                 # opt-in: see compute()
        # pinned staging buffers so every step pays a real host->device copy
        self._pin = {name: torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
                     for name, arr in self._host_inputs().items()}
        self.dev = self._device_inputs()
        self._dev2, self._copy_stream = None, None     # run_many's second input set and its copy stream
        self._h2d_done = None                  # event after the last enqueued copy out of self._pin (load_inputs)
        # what a step reads back, each sliced to the bytes read (decoded by _decode); pinned host copies per slot:
        # 0 / 1 for run_many's two steps in flight, 2 for download()
        self._d2h = [self.gp.out[:self.P * GP_RESULT_DTYPE.itemsize]]
        if self.hyper_mode == "argmin":
            self._d2h += [self._tuned, self._best]
        elif self.hyper_mode == "marginal":
            self._d2h += [self._mstats, self._quant[:self.P * levels.size]]
        self._pinned = [None] * 3

    def _stack_sic(self, sic_fields):
        """One member's {config name: (X, Y, Tfull) SIC field}, or a list of them -> float64 [members * n_configs][X * Y]
        [Tfull]; raises ValueError unless the member count and shapes are the sweep's."""
        member_fields = _members(sic_fields, 1)
        if len(member_fields) != self.members:
            raise ValueError(f"{len(member_fields)} members given, the sweep was built for {self.members}")
        for mf in member_fields:
            for c in self.cfgs:
                if np.shape(mf[c.name]) != (self.X, self.Y, self.Tfull):
                    raise ValueError(f"{c.name}: SIC field of shape {np.shape(mf[c.name])}, expected "
                                     f"{(self.X, self.Y, self.Tfull)}")
        return np.stack([np.ascontiguousarray(mf[c.name], dtype=np.float64).reshape(self.X * self.Y, self.Tfull)
                         for mf in member_fields for c in self.cfgs])

    def _stack_sst(self, sst_field):
        """One (Xs, Ys, Tfull) SST field shared by every member, or one per member -> float64 [members][Xs * Ys][Tfull];
        raises ValueError unless the field count and shapes are the sweep's."""
        sst_members = _members(sst_field, self.members)
        if len(sst_members) != self.members:
            raise ValueError(f"{len(sst_members)} SST fields given, the sweep was built for {self.members} members")
        if any(np.shape(f) != (self.Xs, self.Ys, self.Tfull) for f in sst_members):
            raise ValueError(f"SST fields must have the shape {(self.Xs, self.Ys, self.Tfull)}")
        return np.stack([np.ascontiguousarray(f, dtype=np.float64).reshape(self.Xs * self.Ys, self.Tfull)
                         for f in sst_members])

    def _device_inputs(self):
        """A device buffer for every pinned input."""
        return {k: torch.empty_like(t, device="cuda") for k, t in self._pin.items()}

    def _host_inputs(self):
        p = self.plan
        d = {"sic": self.sic_host, "job_field": p.job_field, "job_T": p.job_T, "rcrit": p.rcrit,
             "psar": self.psar_host, "prob": p.prob.view(np.uint8), "y": p.y}
        if self.use_sst:
            d.update({"sst": self.sst_host, "sst_T": p.sst_T, "sst_rcrit": p.sst_rcrit, "lat": self.lat_host,
                      "sst_field_idx": p.sst_member.astype(np.int32)})
        return d

    def h2d_bytes(self):
        return int(sum(t.numel() * t.element_size() for t in self._pin.values()))

    def d2h_bytes(self):
        return int(sum(t.numel() * t.element_size() for t in self._d2h))

    def upload(self):
        """Host -> device copy of every input (pinned, async on the current stream) into device buffers that keep their
        addresses, so the captured step (compute) can be replayed on fresh inputs."""
        for k, t in self._pin.items():
            self.dev[k].copy_(t, non_blocking=True)
        self._h2d_done = torch.cuda.Event()
        self._h2d_done.record()
        return self.dev

    def load_inputs(self, sic_fields, sst_field=None):
        """Replace the sweep's input fields (same shapes and member count as the constructor's) for the next upload():
        an ensemble far larger than one device batch streams through the same device buffers batch by batch instead of
        re-allocating them (the stored correlation matrices alone are ~29 GB for 8 north members).  Rewrites the pinned
        host buffers in place once every copy still reading them has finished.  `sst_field` None keeps the current SST
        inputs.  The node capacity stays the constructor's: a batch with more ocean cells raises in check_status()."""
        sic = self._stack_sic(sic_fields)
        sst = self._stack_sst(sst_field) if self.use_sst and sst_field is not None else None
        if self._h2d_done is not None:
            self._h2d_done.synchronize()
        self.sic_host = sic
        self._pin["sic"].numpy()[...] = sic
        if sst is not None:
            self.sst_host = sst
            self._pin["sst"].numpy()[...] = sst

    def compute(self, marks=None, waves=None):
        """Enqueue the whole hot path on the current stream (no host sync).  `marks`: optional list that receives
        (stage name, torch.cuda.Event) pairs recorded after each stage, for per-kernel timing.  `waves`: None = the
        launch plan's waves (short/long-window waves on separate streams when the sweep is multi-wave), 1 = one wave:
        one SIC chain and one SST chain on two streams and one GP launch that waits for both, 0 = that one wave with
        every stage on the current stream (clean per-stage timing).
        With `use_graph` the default call (no marks, default waves) is captured once into a CUDA graph -
        ~55 kernels on up to five streams with their cross-stream dependencies - and replayed afterwards: one launch
        per step instead of ~150 ctypes / stream calls.  Measured on B200 (same box, N = 1 and 2): the replayed step is
        ~5 % SLOWER back to back (13.8 vs 12.9 ms; the graph's branch scheduling loses the issue order the eager
        streams impose) and ~1 % faster end to end, so eager stays the default."""
        if waves not in (None, 0, 1):
            raise ValueError(f"waves must be None, 0 or 1, got {waves!r}")
        if marks is None and waves is None and self.use_graph:
            if self._graph is None:
                self._compute(None, None)               # eager once: sets the kernel attributes
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._compute(None, None)
                self._graph = g
            self._graph.replay()
            return
        self._compute(marks, waves)

    def _compute(self, marks, waves):
        d = self.dev
        plan_waves, launches = self._plan if waves is None else self._one_wave
        nw = len(plan_waves)
        sfx = [""] if nw == 1 else [str(w) for w in range(nw)]        # stage tags: sic / sst / gp, or sic0, gps1, ...
        main = torch.cuda.current_stream()
        streams = [(main, main)] if waves == 0 else self._streams[:nw]

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append((name, ev))

        def chain(tag, eng, fields, job_field, job_T, rcrit, scale, jr):
            mark(tag + ".start")
            eng.detrend_zscore(fields, job_field, job_T, do_detrend=True, jr=jr)
            mark(tag + ".detrend_zscore")
            eng.corr_tau(rcrit, store_R=eng.R is not None, jr=jr)
            mark(tag + ".corr_tau")
            eng.area_level(jr=jr)
            mark(tag + ".area_level")
            eng.intra_links(scale, jr=jr)
            mark(tag + ".intra_links")

        if self.tune is not None:               # before any side stream forks from `main`
            expand_problems(d["prob"], self.tune.ell_dev, self.tune.prob)
        for (s1, s2) in streams:
            s1.wait_stream(main)
            s2.wait_stream(main)
        sdone = [None] * nw                     # SST networks of wave w complete (None: the wave has none)
        done = [None] * nw
        # enqueue order = issue order: SIC chains from the longest windows (the critical path) to the shortest, then
        # the SST chains from the shortest to the longest (measured best of the orders tried, tools/timeline.py; splitting
        # the chains into fronts K1+K2 / backs K3-K6 with high-priority fronts or explicit front-before-back events was
        # 5-12 % slower in steady state: the long-window area CTAs must never wait for an SM)
        seq = [("s", w) for w in range(nw)] + [("t", w) for w in range(nw - 1, -1, -1)]
        for kind, w in seq:
            jr, sr, _ = plan_waves[w]
            if kind == "s":
                with torch.cuda.stream(streams[w][0]):
                    if jr[1] > jr[0]:
                        chain("sic" + sfx[w], self.sic, d["sic"], d["job_field"], d["job_T"], d["rcrit"], d["psar"], jr)
                    ev = torch.cuda.Event()
                    ev.record()
                    done[w] = ev
            elif sr[1] > sr[0]:
                with torch.cuda.stream(streams[w][1]):
                    chain("sst" + sfx[w], self.sst, d["sst"], d["sst_field_idx"], d["sst_T"], d["sst_rcrit"], d["lat"],
                          sr)
                    ev = torch.cuda.Event()
                    ev.record()
                    sdone[w] = ev
        # GP of wave w: needs its own networks and those of the shorter-window waves (previous-year configurations);
        # a launch that reads SST networks also waits for those
        for launch in launches:
            w = launch.wave
            tag = ("gps" if launch.sst and nw > 1 else "gp") + sfx[w]
            st = streams[w][launch.sst]
            with torch.cuda.stream(st):
                for v in range(w, nw):
                    st.wait_event(done[v])
                    if launch.sst and sdone[v] is not None:
                        st.wait_event(sdone[v])
                mark(tag + ".start")
                self._gp_run(launch, mark, tag)
                mark(tag)
        for (s1, s2) in streams:                # the step is complete on `main` once every wave has finished
            main.wait_stream(s1)
            main.wait_stream(s2)

    def _gp_run(self, launch, mark, tag):
        """One GP launch of the step on the current stream over its problems p0..p1-1, results into self.gp.out.
        Tuned sweep: sie_gp_hyper_grid over the range's expanded problems, sie_gp_grid_select, then sie_gp_forecast of
        the selected problems -- three launches in stream order on the launch's batch, no host sync.  Marginal sweep:
        the grid, then sie_gp_grid_marginal straight into self.gp.out and the range's stats / quantiles."""
        d, p0, p1, gp = self.dev, launch.p0, launch.p1, launch.gp
        if self.tune is None:
            gp.run(d["prob"], d["y"], self.sic, self.sst, (p0, p1), out=self.gp.out)
            return
        g, nl, ns = self.tune, len(self.tune.ells), len(self.tune.sigs)
        isz, osz = GP_PROBLEM_DTYPE.itemsize, GP_RESULT_DTYPE.itemsize
        grid = g.out[p0 * nl * ns * osz:]
        gp.run_grid(g.prob[p0 * nl * isz:], g.sig_dev, ns, d["y"], self.sic, self.sst, grid, n=(p1 - p0) * nl)
        mark(tag + ".grid")
        if self.hyper_mode == "marginal":
            nq = self.levels.size
            grid_marginal(grid, p1 - p0, nl * ns, self._q_dev, self.gp.out[p0 * osz:],
                          self._mstats[p0 * GP_MARGINAL_DTYPE.itemsize:], self._quant[p0 * nq:])
            return
        grid_select(grid, d["prob"][p0 * isz:], p1 - p0, g.ell_dev, g.sig_dev, self._tuned[p0 * isz:], self._best[p0:])
        gp.run(self._tuned, d["y"], self.sic, self.sst, (p0, p1), out=self.gp.out)

    def _grid_buffers(self, ells, sigs):
        key = (ells.tobytes(), sigs.tobytes())
        if key not in self._grids:
            self._grids[key] = _GridBuffers(ells, sigs, self.P)
        return self._grids[key]

    def grid_records(self):
        """Tuned sweep: the grid records [P][n_ell][n_sig] of the last step (host; synchronises)."""
        g = self.tune
        return g.out.cpu().numpy().view(GP_RESULT_DTYPE).reshape(self.P, len(g.ells), len(g.sigs))

    def best_index(self):
        """Tuned sweep: flat grid index i * n_sig + j each problem of the last step forecast at, -1 where no grid point
        was admissible and the script's own (l, sigma_n~) was kept (host int32 [P]; synchronises)."""
        return self._best.cpu().numpy()

    def tuned_problems(self):
        """Tuned sweep: the problem records the last step forecast with (host GP_PROBLEM_DTYPE [P]; synchronises)."""
        return self._tuned.cpu().numpy().view(GP_PROBLEM_DTYPE)

    def hyper_grid(self, ells=None, sigs=None):
        """BASELINE.json configs[4] on this member: every GP problem of the sweep (year x init x region) evaluated on
        the reference's `ls` x `ss` hyper-parameter grid (north/June1st.py:210-211), from the node series the last
        compute() left on the device.  One CTA per (problem, l): expm and X Sigma X^T once, the Cholesky fit / nlML for
        every sigma.  Returns records [P][len(ells)][len(sigs)] (host)."""
        ells = np.logspace(-7, 2, 20) if ells is None else np.asarray(ells, dtype=np.float64)
        sigs = np.logspace(-3, 9, 20) if sigs is None else np.asarray(sigs, dtype=np.float64)
        nl, ns = len(ells), len(sigs)
        g = self._grid_buffers(ells, sigs)
        if g.gp is None:
            g.gp = GpBatch(self.P * nl, max_pred=self.gp.max_pred)
        expand_problems(self.dev["prob"], g.ell_dev, g.prob)
        g.gp.run_grid(g.prob, g.sig_dev, ns, self.dev["y"], self.sic, self.sst, g.out)
        return g.out.cpu().numpy().view(GP_RESULT_DTYPE).reshape(self.P, nl, ns)

    def kernel_launches(self):
        """Kernels of libsie_b200 enqueued by one compute(): 12 per network chain (K1: 3, K2: 4, K3-K5: 2, K6: 3) + 2 per
        GP launch (tuned sweep: 5 -- grid 2, select 1, forecast 2; marginal sweep: 3 -- grid 2, marginal 1)."""
        per_gp = 2 if self.tune is None else (5 if self.hyper_mode == "argmin" else 3)
        chains = sum((jr[1] > jr[0]) + (sr[1] > sr[0]) for (jr, sr, _) in self._plan.waves)
        return 12 * chains + per_gp * len(self._plan.launches)

    def _read_back(self, slot):
        """Enqueue (current stream) the copies of the step's outputs self._d2h into pinned set `slot` -> the set."""
        bufs = self._pinned[slot]
        if bufs is None:
            bufs = self._pinned[slot] = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in self._d2h]
        for b, t in zip(bufs, self._d2h):
            b.copy_(t, non_blocking=True)
        return bufs

    def _decode(self, bufs):
        """Host copies of self._d2h -> self.raw (a copy: the pinned buffers are reused), self.selection (tuned sweep),
        self.marginal (marginal sweep)."""
        host = [b.numpy() for b in bufs]
        self.raw = host[0].view(GP_RESULT_DTYPE).copy()
        if self.hyper_mode == "argmin":
            self.selection = selection_records(host[1].view(GP_PROBLEM_DTYPE), host[2])
        elif self.hyper_mode == "marginal":
            self.marginal = marginal_records(host[1], host[2])

    def download(self):
        """Device -> host read of the GP results (synchronises).  Raises if any network build or GP problem ran out of
        the capacity this sweep was sized for (a silent NaN forecast would look like a reference failure).  Tuned
        sweep: also reads the selected (l, sigma_n~) and grid indices into self.selection; marginal sweep: the grid
        posterior's stats and the quantiles into self.marginal."""
        bufs = self._read_back(2)
        torch.cuda.current_stream().synchronize()
        self._decode(bufs)
        self.check_status(self.raw)
        return self.raw

    def run(self):
        self.upload()
        self.compute()
        return self.plan.assemble(self.download(), selection=self.selection, marginal=self.marginal)

    def run_many(self, n):
        """Generator over `n` sweeps run back to back (a perturbed-input ensemble, bench.py's end-to-end loop): every
        step does its own host -> device copy of the inputs, the whole hot path and a device -> host read of its results,
        but step i's read lands in a pinned buffer and is assembled on the host while step i+1 is already on the
        device, so host work (launch enqueue, assemble) is off the device's critical path, and step i+1's inputs are
        copied from the pinned buffers into a second set of device buffers on a copy stream while step i computes.
        Yields the same dict as run() per step; `self.raw` holds the records of the step just yielded."""
        pending = None

        def finish(ev, k):
            ev.synchronize()
            self._decode(self._pinned[k])
            if (self.raw["info"] == -2).any():
                self.check_status(self.raw)
            return self.plan.assemble(self.raw, selection=self.selection, marginal=self.marginal)

        # inputs are double-buffered on the device: step i+1's host -> device copy runs on a copy stream while step i
        # computes (with CUDA-graph replay the captured step reads fixed addresses: single buffer, copy in stream order)
        n = int(n)
        overlap = not self.use_graph
        if overlap:
            if self._dev2 is None:
                self._dev2 = self._device_inputs()
                self._copy_stream = torch.cuda.Stream()
            devs = [self.dev, self._dev2]
            main = torch.cuda.current_stream()
            up_ev, done_ev = [None, None], [None, None]

            def upload_to(k):
                cs = self._copy_stream
                if done_ev[k] is not None:
                    cs.wait_event(done_ev[k])           # the step that last read this buffer is finished
                else:
                    cs.wait_stream(main)
                with torch.cuda.stream(cs):
                    for key, t in self._pin.items():
                        devs[k][key].copy_(t, non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(cs)
                self._h2d_done = ev
                return ev

            if n > 0:
                up_ev[0] = upload_to(0)
        for i in range(n):
            if overlap:
                k = i & 1
                main.wait_event(up_ev[k])
                self.dev = devs[k]
                if i + 1 < n:
                    up_ev[k ^ 1] = upload_to(k ^ 1)
                self.compute()
                done_ev[k] = torch.cuda.Event()
                done_ev[k].record(main)
            else:
                self.upload()
                self.compute()
            self._read_back(i & 1)
            ev = torch.cuda.Event()
            ev.record()
            if pending is not None:
                yield finish(*pending)
            pending = (ev, i & 1)
        if pending is not None:
            yield finish(*pending)
        self.check_status()                    # every step ran the same inputs: one check of the job statuses suffices

    def check_status(self, raw=None):
        """Raises SieError when a network build exceeded the node / area capacity (status SIE_JOB_CAPACITY, SIC or SST
        engine) or a GP problem the predictor capacity `max_pred` (info = -2); returns the SIC status array.  A job
        over capacity produces no areas, so its forecasts come back as info = -1 / NaN: indistinguishable from a
        reference failure unless checked here."""
        st = self.sic.status.cpu().numpy()
        for tag, eng in (("SIC", self.sic), ("SST", self.sst)):
            if eng is None:
                continue
            bad = np.nonzero(eng.status.cpu().numpy() == _lib.SIE_JOB_CAPACITY)[0]
            if bad.size:
                raise _lib.SieError(f"capacity exceeded in {tag} network builds {bad.tolist()[:8]} (nodes > {eng.ldn} "
                                    f"or areas > {eng.MA}): construct the sweep with larger capacities")
        if raw is not None:
            bad = np.nonzero(np.asarray(raw["info"]) == -2)[0]
            if bad.size:
                raise _lib.SieError(f"GP problems {bad.tolist()[:8]} selected more than max_pred = {self.gp.max_pred} "
                                    "predictors (or n + 1 > 64 samples): construct the sweep with a larger max_pred")
        return st


class EnsembleForecast:
    """The ensemble forecast of a perturbed-input ensemble: every member's predictive distribution of each (config,
    region, year) pooled into one on the device (sie_gp_ensemble), each member with weight 1 / M' (M' = members with a
    forecast there).  It carries the input uncertainty on top of the GP and hyper-parameter uncertainty that each
    member's record holds: fvar = var_within (mean member variance) + var_between (spread of the member means).

    sweep      : a single-rank RetrospectiveSweep; fixes the configs, years, SIE targets, hyper mode and grid every added
                 sweep must share.  What is pooled per member: the forecast record of plain and tuned ("argmin")
                 sweeps (n_grid = 1), all n_ell * n_sig grid records of marginalised sweeps (n_grid = the grid size;
                 each member then enters as its grid marginal)
    n_members  : member slots; every slot must be filled by add() before result()
    quantiles  : levels in (0, 1) of the pooled distribution's quantiles

    Device memory, allocated once here: the record store, 80 * E * n_members * n_grid bytes (E = configs x regions x
    years; 14.2 GB for the 4-init north sweep at 1024 members x the 400-point grid), and the kernel's scratch,
    24 * E * n_members * n_grid bytes (4.2 GB there).  The ensemble streams through one sweep batch by batch:
    sweep.load_inputs(batch) -> upload() -> compute() -> add(sweep, first_member), then result()."""

    def __init__(self, sweep, n_members, quantiles=DEFAULT_QUANTILES):
        if sweep.plan.world > 1:
            raise NotImplementedError("an ensemble forecast pools the members of a single-rank sweep (world = 1)")
        self.n_members = int(n_members)
        if self.n_members < 1:
            raise ValueError(f"n_members must be positive, got {n_members}")
        self.levels = check_levels(quantiles)
        self.plan = sweep.plan
        self._key = self._signature(sweep)
        self.n_grid = len(sweep.tune.ells) * len(sweep.tune.sigs) if sweep.hyper_mode == "marginal" else 1
        self.meta, _ = ensemble_slots(self.plan, self.n_members)
        self.E = len(self.meta)
        self._rb = self.n_grid * GP_RESULT_DTYPE.itemsize
        self.store = torch.empty(self.E * self.n_members * self._rb, dtype=torch.uint8, device="cuda")
        self._filled = np.zeros(self.E * self.n_members, dtype=bool)
        self._rows = weakref.WeakKeyDictionary()          # sweep -> (host rows, device rows) of its problems
        self._q_dev = h2d(self.levels) if self.levels.size else None
        self._out = torch.empty(self.E * GP_ENSEMBLE_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        self._quant = torch.empty(max(1, self.E * self.levels.size), dtype=torch.float64, device="cuda")
        self._scratch = torch.empty(gp_ensemble_scratch_bytes(self.E, self.n_members, self.n_grid), dtype=torch.uint8,
                                    device="cuda")
        self.records = None                               # ensemble_records of the last result()

    @staticmethod
    def _signature(sweep):
        p = sweep.plan
        grid = None if sweep.tune is None else (sweep.tune.ells.tobytes(), sweep.tune.sigs.tobytes())
        return (tuple(c.name for c in p.cfgs), tuple(p.years), tuple((k, v.tobytes()) for k, v in sorted(p.sie.items())),
                sweep.hyper_mode, grid)

    def add(self, sweep, first_member=0):
        """Enqueue (current stream, no host sync) the copy of the records of `sweep`'s last compute() into member slots
        first_member + 0 .. sweep.members - 1.  Raises ValueError for a sweep with other configs, years, SIE targets,
        hyper mode or grid, or slots beyond n_members."""
        if sweep.plan.world > 1:
            raise NotImplementedError("an ensemble forecast pools the members of a single-rank sweep (world = 1)")
        if self._signature(sweep) != self._key:
            raise ValueError("the sweep's configs, years, SIE targets, hyper mode or grid differ from the ensemble's")
        first = int(first_member)
        if first < 0 or first + sweep.members > self.n_members:
            raise ValueError(f"members {first}..{first + sweep.members - 1} do not fit the {self.n_members} slots")
        rows = self._rows.get(sweep)
        if rows is None:
            host = ensemble_slots(sweep.plan, self.n_members)[1]
            rows = self._rows[sweep] = (host, h2d(host))
        host, dev = rows
        src = sweep.tune.out if sweep.hyper_mode == "marginal" else sweep.gp.out
        self.store.view(self.E * self.n_members, self._rb).index_copy_(
            0, dev + first if first else dev, src[:sweep.P * self._rb].view(sweep.P, self._rb))
        self._filled[host + first] = True

    def result(self):
        """Pool the store on the device and read it back (synchronises) -> the dict of a member's assembled forecast
        ('<region>_fmean / _fvar / _fmean_rt' at 3 d.p., '_raw_*') for the ensemble forecast, plus '_var_within',
        '_var_between', '_n_members', '_quantiles' and '_quantiles_rt' (re-trended like '_raw_fmean_rt').  NaN where no
        member has a forecast.  SweepPlan.skill() reads it unchanged."""
        if not self._filled.all():
            miss = np.argwhere(~self._filled.reshape(self.E, self.n_members))
            raise RuntimeError(f"{len(miss)} (problem, member) slots were never added, e.g. member {miss[0][1]}")
        gp_ensemble(self.store, self.E, self.n_members, self.n_grid, self._q_dev, self._out, self._quant, self._scratch)
        nq = self.levels.size
        self.records = ensemble_records(self._out.cpu().numpy(), self._quant.cpu().numpy()[:self.E * nq])
        return self.plan._assemble_one(self.records, self.meta, ensemble=self.records)
