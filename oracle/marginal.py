"""ORACLE (test infrastructure, NOT product code) -- numpy / scipy statement of the grid marginal of a GP forecast
(include/sie_b200.h, sie_gp_grid_marginal): the forecasts at every (l, sigma_n~) grid point of one problem averaged
with weights proportional to their marginal likelihoods (profile likelihood: nlML profiles sigma_f out), a uniform
prior over the admissible grid points.

    A   = {k : info_k == 0 and nlml_k finite}
    w_k = exp(-nlml_k - logsumexp(-nlml_A))                      (0 outside A)
    fmean = sum w mu,  fvar = sum w (v + (mu - fmean)^2),  nlml = -logsumexp(-nlml_A) + log|A|
    F(x) = sum w Phi((x - mu) / sqrt(v))   (v <= 0: a point mass at mu), Phi = scipy.special.ndtr

Only `tests/` and the measurement tools may import this module.
"""
from __future__ import annotations

import numpy as np
from scipy.special import logsumexp, ndtr


def admissible(nlml, info):
    nlml = np.asarray(nlml, dtype=np.float64).reshape(-1)
    return (np.asarray(info).reshape(-1) == 0) & np.isfinite(nlml)


def weights(nlml, info):
    """-> (w [n], log S where S = sum over A of exp(-nlml)); w = 0 outside A.  (None, nan) when A is empty."""
    nlml = np.asarray(nlml, dtype=np.float64).reshape(-1)
    adm = admissible(nlml, info)
    if not adm.any():
        return None, np.nan
    lse = logsumexp(-nlml[adm])
    w = np.zeros(nlml.size)
    w[adm] = np.exp(-nlml[adm] - lse)
    return w, lse


def mixture_cdf(x, w, mu, var):
    """F(x) = sum w Phi((x - mu) / sqrt(var)), a component with var <= 0 a point mass at mu (right-continuous)."""
    w, mu, var = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (w, mu, var))
    pos = w > 0
    w, mu, var = w[pos], mu[pos], var[pos]
    sd = np.sqrt(np.where(var > 0, var, 1.0))
    phi = np.where(var > 0, ndtr((x - mu) / sd), (x >= mu).astype(np.float64))
    return float(np.sum(w * phi))


def mixture_quantile(q, w, mu, var):
    """inf {x : F(x) >= q} by bisection on [min(mu - 40 sd), max(mu + 40 sd)] over the components with w > 0, keeping
    F(lo) < q <= F(hi), at most 128 halvings or until the midpoint equals an end; returns hi."""
    w, mu, var = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (w, mu, var))
    pos = w > 0
    sd = np.sqrt(np.maximum(var[pos], 0.0))
    lo, hi = float(np.min(mu[pos] - 40 * sd)), float(np.max(mu[pos] + 40 * sd))
    if mixture_cdf(lo, w, mu, var) >= q:
        return lo
    if mixture_cdf(hi, w, mu, var) < q:
        return hi
    for _ in range(128):
        c = 0.5 * lo + 0.5 * hi
        if c == lo or c == hi:
            break
        if mixture_cdf(c, w, mu, var) >= q:
            hi = c
        else:
            lo = c
    return hi


def marginal(fmean, fvar, nlml, info, levels=()):
    """One problem's grid records (flat [n_grid] arrays) -> dict(fmean, fvar, nlml, ess, w_max, n_admissible, argmax,
    quantiles, w).  With no admissible point: NaN moments / stats / quantiles, n_admissible 0, argmax -1."""
    fmean, fvar, nlml = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (fmean, fvar, nlml))
    levels = np.asarray(levels, dtype=np.float64).reshape(-1)
    w, lse = weights(nlml, info)
    if w is None:
        nan = np.nan
        return dict(fmean=nan, fvar=nan, nlml=nan, ess=nan, w_max=nan, n_admissible=0, argmax=-1,
                    quantiles=np.full(levels.size, nan), w=None)
    adm = admissible(nlml, info)
    mu = np.where(adm, fmean, 0.0)
    var = np.where(adm, fvar, 0.0)
    fm = float(np.sum(w * mu))
    fv = float(np.sum(w * (var + (mu - fm) ** 2)))
    argmax = int(np.argmin(np.where(adm, nlml, np.inf)))
    q = np.array([mixture_quantile(t, w, mu, var) for t in levels])
    return dict(fmean=fm, fvar=fv, nlml=float(-lse + np.log(adm.sum())), ess=float(1.0 / np.sum(w ** 2)),
                w_max=float(w.max()), n_admissible=int(adm.sum()), argmax=argmax, quantiles=q, w=w)
