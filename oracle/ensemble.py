"""ORACLE (test infrastructure, NOT product code) -- numpy / scipy statement of the ensemble pool of GP forecasts
(include/sie_b200.h, sie_gp_ensemble): the predictive distributions of M input-perturbed members of one problem pooled
into one, every member with weight 1 / M'.  Member m's distribution is its grid marginal (oracle/marginal.py) over
its n_grid records (n_grid = 1: the record's Gaussian).

    A_m  = member m's admissible records (info == 0, finite nlml), M' = #{m : A_m non-empty}
    w_mk = member m's marginal-likelihood weights (oracle/marginal.py), mu_m = sum_k w_mk mu_mk,
    v_m  = sum_k w_mk (v_mk + (mu_mk - mu_m)^2)
    fmean = sum mu_m / M',  var_within = sum v_m / M',  var_between = sum (mu_m - fmean)^2 / M',
    fvar = var_within + var_between
    F(x) = sum_m sum_k (w_mk / M') Phi((x - mu_mk) / sqrt(v_mk))   (the flattened two-level mixture)

Only `tests/` and the measurement tools may import this module.
"""
from __future__ import annotations

import numpy as np

from oracle import marginal as om


def ensemble(fmean, fvar, nlml, info, levels=()):
    """One problem's records ([M][n_grid] arrays) -> dict(fmean, fvar, var_within, var_between, n_members, quantiles,
    member_mean [M], member_var [M] (NaN for a member without an admissible record), w [M][n_grid] (the flattened
    two-level weights), mu, var [M][n_grid] (0 outside the admissible records)).  M' = 0: NaN moments and quantiles."""
    fmean, fvar, nlml = (np.atleast_2d(np.asarray(a, dtype=np.float64)) for a in (fmean, fvar, nlml))
    info = np.atleast_2d(np.asarray(info))
    levels = np.asarray(levels, dtype=np.float64).reshape(-1)
    M = fmean.shape[0]
    w = np.zeros(fmean.shape)
    mm, mv = np.full(M, np.nan), np.full(M, np.nan)
    ok = np.zeros(M, dtype=bool)
    for m in range(M):
        wm, _ = om.weights(nlml[m], info[m])
        if wm is None:
            continue
        r = om.marginal(fmean[m], fvar[m], nlml[m], info[m])
        mm[m], mv[m] = r["fmean"], r["fvar"]
        w[m] = wm
        ok[m] = True
    n = int(ok.sum())
    adm = w > 0
    mu, var = np.where(adm, fmean, 0.0), np.where(adm, fvar, 0.0)
    if n == 0:
        nan = np.nan
        return dict(fmean=nan, fvar=nan, var_within=nan, var_between=nan, n_members=0,
                    quantiles=np.full(levels.size, nan), member_mean=mm, member_var=mv, w=w, mu=mu, var=var)
    w = w / n
    f = float(np.mean(mm[ok]))
    vw = float(np.mean(mv[ok]))
    vb = float(np.mean((mm[ok] - f) ** 2))
    q = np.array([om.mixture_quantile(t, w, mu, var) for t in levels])
    return dict(fmean=f, fvar=vw + vb, var_within=vw, var_between=vb, n_members=n, quantiles=q, member_mean=mm,
                member_var=mv, w=w, mu=mu, var=var)
