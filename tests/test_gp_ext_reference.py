"""The extended-precision GP reference (oracle/gp_ext.py) pinned on the CPU, before any kernel is compared with it:

  * its Pade expm against exact matrix exponentials (40-digit mpmath eigendecompositions of the symmetric M), at
    every Pade order the kernel can pick;
  * its fmean / fvar / sigma_f / nlml / MLII gradient against the float64 oracle (scipy / LAPACK) on every shape of
    tests/test_gp_kernel_shapes_gpu.py's Np sweep, within the bound the kernel is held to there -- so that bound is
    not tighter than float64 arithmetic can reach."""
import mpmath
import numpy as np
import pytest

from oracle import expm_spec as es
from oracle import gp as og
from oracle import gp_ext as ge

U_LD = float(np.finfo(np.longdouble).eps) / 2
ORDERS = [(3, 0), (5, 0), (7, 0), (9, 0), (13, 0), (13, 1), (13, 5), (13, 20)]


def exact_expm(A):
    """expm of a symmetric matrix at 40 digits: Q diag(exp(lambda)) Q^T."""
    with mpmath.workdps(40):
        lam, Q = mpmath.eigsy(mpmath.matrix(A.tolist()))
        R = Q * mpmath.diag([mpmath.exp(x) for x in lam]) * Q.T
        return np.array([[np.longdouble(mpmath.nstr(R[i, j], 30)) for j in range(A.shape[1])]
                         for i in range(A.shape[0])])


@pytest.mark.parametrize("Np", [4, 9, 16])
@pytest.mark.parametrize("m,s", ORDERS)
def test_pade_expm_matches_exact(Np, m, s):
    y, sic, _ = ge.series(Np, 41, Np)
    _, _, M = og.design(og.select_predictors(y, sic, None, "all"), True)
    ell = ge.ell_for(M, m, s)
    assert ell is not None, (Np, m, s)
    A = ell * M
    assert es.pick(A)[:2] == (m, s)
    X = exact_expm(A)
    scale = np.abs(X).max()
    # at pick's (m, s) the Pade truncation has backward error <= u (float64) by construction; expm of a symmetric
    # matrix has relative condition number ||A||_2, so the forward error stays below max(1, ||A||_2) u
    err = float(np.abs(ge.pade_expm(A, m, s) - X).max() / scale)
    assert err <= 2.0 * max(1.0, np.linalg.norm(A, 2)) * ge.U64, (err, np.linalg.norm(A, 2))
    if s <= 3:
        # 64 more halvings of the truncation error (s + 6) put it below long-double rounding: what is left is the
        # long-double arithmetic itself, ~2^(s + 6) squarings' worth of its rounding
        err6 = float(np.abs(ge.pade_expm(A, 13, s + 6) - X).max() / scale)
        assert err6 <= 1000 * U_LD, err6


@pytest.mark.parametrize("zscore", [True, False])
@pytest.mark.parametrize("Np", ge.NP_SWEEP)
def test_reference_matches_float64_oracle(Np, zscore):
    """The bound the kernel tests use, max(2^-40, 64 2^s u, 8 cond(K) u), also holds between this reference and the
    float64 oracle on every shape of the Np sweep: float64 arithmetic can meet it."""
    n = 41
    y, sic, ell, sig = ge.shape_problem(Np, n, zscore)
    Xfull = og.select_predictors(y, sic, None, "all")
    assert Xfull.shape[1] == Np
    X, Xs, M = og.design(Xfull, zscore)
    m, s, _ = es.pick(ell * M)
    r = ge.Problem(Xfull, y, zscore, ell, m, s, want_grad=True).fit(sig)
    o = og.gp_fit_predict(X, Xs, y[:, None], M, ell, sig)
    nl, g = og.mlii(np.log([ell, sig]), X, y[:, None], M)
    assert r["info"] == 0
    t = ge.bound(s, r["cond"])
    sd = max(abs(float(r["fmean"])), np.sqrt(abs(float(r["fvar"]))), 1e-3)
    checks = [("fmean", o["fmean"], sd), ("fvar", o["fvar"], sd ** 2), ("sigma_f", o["sigma_f"], abs(r["sigma_f"])),
              ("nlml", o["nlml"], max(1.0, r["nlml_mag"])), ("nlml", nl, max(1.0, r["nlml_mag"])),
              ("g_ell", g[0], max(1.0, r["mag_ell"])), ("g_sig", g[1], max(1.0, r["mag_sig"]))]
    for name, val, scale in checks:
        err = abs(float(val - r[name])) / float(scale)
        assert err <= t, (name, err, t, (m, s), r["cond"])
