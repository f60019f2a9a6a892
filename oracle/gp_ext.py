"""ORACLE (test infrastructure, NOT product code) -- `oracle.gp.gp_fit_predict` and `oracle.gp.mlii` restated in
extended precision (np.longdouble: a 64-bit mantissa on x86-64, u = 2^-64, about 2000 times finer than float64).

The float64 oracle delegates to scipy / LAPACK, whose own rounding is of the same size as the GP kernel's, so a
disagreement between the two says nothing about which one is wrong.  This restatement holds none of that error:

  * the float64 series and targets convert exactly to long double; the design matrix (optional z-score over all n + 1
    rows) and the graph Laplacian M are formed in long double;
  * predictor selection is a decision, not a value: it uses the float64 `oracle.gp.select_predictors`, so test data
    must keep every |r| and r - r_sel well away from zero;
  * expm(l M) is the Pade approximant of `oracle.expm_spec` at a GIVEN (m, s) -- the (m, s) the kernel reports -- so
    the reference and the kernel differ only in rounding, not in truncation; (V - U) X = V + U is solved by a
    partial-pivot LU written here (numpy's LAPACK is float64 only), then squared s times;
  * both Cholesky factorisations and every triangular solve are written here too.

tests/test_gp_ext_reference.py pins it against exact (40-digit mpmath) matrix exponentials and against the float64
oracle.  Only `tests/` may import this module."""
from __future__ import annotations

import numpy as np

from . import expm_spec
from . import gp as og

LD = np.longdouble
U64 = 2.0 ** -53                      # float64 unit roundoff, the unit of the kernel's error bounds
PI = LD("3.141592653589793238462643383279502884")


def design(Xfull, zscore):
    """`oracle.gp.design` in long double: (X [n][Np], Xs [Np], M [Np][Np])."""
    X = np.asarray(Xfull, dtype=np.float64).astype(LD)
    if zscore:
        mu = X.sum(axis=0) / LD(X.shape[0])
        d = X - mu
        X = d / np.sqrt((d * d).sum(axis=0) / LD(X.shape[0]))
    Xs, X = X[-1, :].copy(), X[:-1, :]
    Xc = X - X.sum(axis=0) / LD(X.shape[0])
    M = np.abs(Xc.T @ Xc / LD(X.shape[0]))
    np.fill_diagonal(M, LD(0))
    np.fill_diagonal(M, -M.sum(axis=0))
    return X, Xs, M


def pade_expm(A, m, s):
    """expm(A) by the degree-m Pade approximant with 2^-s scaling and s squarings (oracle/expm_spec.py's formulas)."""
    A = np.asarray(A).astype(LD)
    n = A.shape[0]
    eye = np.eye(n, dtype=LD)
    b = [LD(c) for c in expm_spec.B[m]]
    sc = LD(2) ** -int(s)
    A = A * sc
    A2 = A @ A
    A4 = A2 @ A2
    A6 = A4 @ A2
    if m == 13:
        U = A @ (A6 @ (b[13] * A6 + b[11] * A4 + b[9] * A2) + b[7] * A6 + b[5] * A4 + b[3] * A2 + b[1] * eye)
        V = A6 @ (b[12] * A6 + b[10] * A4 + b[8] * A2) + b[6] * A6 + b[4] * A4 + b[2] * A2 + b[0] * eye
    else:
        pw = [eye, A2, A4, A6, A4 @ A4][:m // 2 + 1]
        U = A @ sum(b[2 * i + 1] * p for i, p in enumerate(pw))
        V = sum(b[2 * i] * p for i, p in enumerate(pw))
    X = lu_solve(V - U, V + U)
    for _ in range(int(s)):
        X = X @ X
    return X


def lu_solve(P, Q):
    """P X = Q by Gaussian elimination with partial pivoting (any float dtype; P, Q are not modified)."""
    P = P.copy()
    Q = Q.copy()
    n = P.shape[0]
    for k in range(n):
        p = k + int(np.argmax(np.abs(P[k:, k])))
        if p != k:
            P[[k, p]] = P[[p, k]]
            Q[[k, p]] = Q[[p, k]]
        lk = P[k + 1:, k] / P[k, k]
        P[k + 1:, k:] -= np.outer(lk, P[k, k:])
        Q[k + 1:] -= np.outer(lk, Q[k])
    for k in range(n - 1, -1, -1):
        Q[k] = (Q[k] - P[k, k + 1:] @ Q[k + 1:]) / P[k, k]
    return Q


def cholesky(K):
    """Lower Cholesky factor, or None when a pivot is not positive."""
    n = K.shape[0]
    L = np.zeros_like(K)
    for j in range(n):
        d = K[j, j] - L[j, :j] @ L[j, :j]
        if not d > 0:
            return None
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (K[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return L


def fwd(L, b):
    """L^-1 b (b a vector or a matrix of columns)."""
    x = np.zeros_like(b)
    for i in range(L.shape[0]):
        x[i] = (b[i] - L[i, :i] @ x[:i]) / L[i, i]
    return x


def bwd(L, b):
    """L^-T b."""
    x = np.zeros_like(b)
    for i in range(L.shape[0] - 1, -1, -1):
        x[i] = (b[i] - L[i + 1:, i] @ x[i + 1:]) / L[i, i]
    return x


class Problem:
    """One forecast problem in long double: the design of `oracle.gp.design`, and expm(l M) at a given (m, s).
    `fit(sig)` is gp_fit_predict / MLII at that sigma_n~, reusing the expm (as the kernel's grid mode does)."""

    def __init__(self, Xfull, y, zscore, ell, m, s, want_grad=False):
        self.y = np.asarray(y, dtype=np.float64).astype(LD)
        self.n = self.y.size
        self.X, self.Xs, self.M = design(Xfull, zscore)
        self.ell, self.m, self.s = float(ell), int(m), int(s)
        self.E = pade_expm(LD(ell) * self.M, m, s)
        XE = self.X @ self.E
        self.W = XE @ self.X.T
        self.kxs_raw = XE @ self.Xs
        self.kss_raw = self.Xs @ self.E @ self.Xs
        self.G1 = self.X @ (self.M @ self.E) @ self.X.T if want_grad else None

    def fit(self, sig):
        """-> dict: fmean, fvar, sigma_f, nlml, nlml_mag (|y^T alpha| / 2 + sum |log L_ii| + n log(2 pi) / 2), cond
        (2-norm condition number of K, float64), info (0, or the 1-based failing Cholesky pivot), and with the gradient
        g_ell, g_sig and mag_ell, mag_sig: |trace(K^-1 dK)| / 2 + |alpha^T dK alpha| / 2 of each component."""
        n, y, W = self.n, self.y, self.W
        sig = LD(sig)
        eye = np.eye(n, dtype=LD)
        out = {"cond": float(np.linalg.cond(np.asarray(W + sig * eye, dtype=np.float64)))}
        L = cholesky(W + sig * eye)
        if L is None:
            out["info"] = 1
            return out
        sf = (y @ bwd(L, fwd(L, y))) / LD(n)
        sn = sf * sig
        K = sf * W + sn * eye
        L = cholesky(K)
        if L is None:
            out["info"] = 1
            return out
        alpha = bwd(L, fwd(L, y))
        kx = sf * self.kxs_raw
        v = fwd(L, kx)
        logdet = np.log(np.diag(L))
        half_log2pi = LD(n) * np.log(LD(2) * PI) / LD(2)
        out.update(info=0, sigma_f=sf, fmean=kx @ alpha, fvar=sf * self.kss_raw + sn - v @ v,
                   nlml=(y @ alpha) / LD(2) + logdet.sum() + half_log2pi,
                   nlml_mag=abs(y @ alpha) / LD(2) + np.abs(logdet).sum() + half_log2pi)
        if self.G1 is not None:
            for name, dK in (("ell", sf * self.G1 + sn * eye), ("sig", sf * W + sf * eye)):
                tr = np.trace(bwd(L, fwd(L, dK)))
                quad = alpha @ dK @ alpha
                out["g_" + name] = tr / LD(2) - quad / LD(2)
                out["mag_" + name] = abs(tr) / LD(2) + abs(quad) / LD(2)
        return out


def problem(y, anoms_sic, anoms_sst, rule, alpha, zscore, ell, m, s, want_grad=False):
    """Problem of the reference's forecast(): float64 selection (`oracle.gp.select_predictors`, rule 'pos' / 'all' /
    'pos_sig'), then the long-double design and expm(l M) at (m, s).  Returns (Problem, n_pred)."""
    Xfull = og.select_predictors(np.asarray(y, dtype=np.float64), anoms_sic, anoms_sst, rule, alpha)
    return Problem(Xfull, y, zscore, ell, m, s, want_grad), Xfull.shape[1]


def bound(s, cond):
    """Relative error bound of a kernel result against this reference: max(2^-40, 64 2^s u, 8 cond(K) u), u = 2^-53.
    2^s u: s squarings amplify rounding by ~2^s; cond(K) u: two backward-stable Cholesky solves."""
    return max(2.0 ** -40, 64.0 * 2.0 ** int(s) * U64, 8.0 * float(cond) * U64)


def series(seed, n, n_sic, n_sst=0, scale=1.0, sst_scale=0.1):
    """Synthetic node series built like tests/test_gp_gpu.py's: three common factors plus noise; returns
    (y [n], sic {key: [n + 1]}, sst {key: [n + 1]} or None).  y is rounded to 3 d.p. like the scripts' targets."""
    rng = np.random.default_rng(seed)
    common = rng.standard_normal((3, n + 1))
    sic = {2 * a + 1: scale * (rng.standard_normal(3) * 0.8 @ common + rng.standard_normal(n + 1))
           for a in range(n_sic)}
    sst = None
    if n_sst:
        sst = {a: sst_scale * (rng.standard_normal(3) @ common + rng.standard_normal(n + 1)) for a in range(n_sst)}
    y = np.round(0.3 * (common[0, :n] - common[1, :n]) + 0.2 * rng.standard_normal(n), 3)
    return y, sic, sst


def pick_margin(A):
    """The smallest relative distance, over every comparison `oracle.expm_spec.pick(A)` makes on its way to (m, s),
    between a compared quantity and its threshold (for the ceil()s: of the quantity to the nearest power of 2 that
    moves the result).  Below ~1e-12 a device that forms the same quantities in another summation order may take
    the other branch."""
    import math
    absA = np.abs(A)
    normA = expm_spec.norm1(A)
    margins = []

    def near(x, t):
        margins.append(abs(x - t) / abs(t))
        return x < t

    def ell(a, na, idx, m):
        t = expm_spec.absnorm_power(a, 2 * m + 1)
        if not t > 0:
            return 0
        val = math.log2(t / na / expm_spec.COEFF[idx]) / (2 * m)
        if not np.isfinite(val):
            return 1 << 20
        margins.append(abs(val - round(val)) * 2 * m * math.log(2.0))
        return max(int(math.ceil(val)), 0)

    A2 = A @ A
    A4 = A2 @ A2
    A6 = A4 @ A2
    d4, d6 = expm_spec.norm1(A4) ** 0.25, expm_spec.norm1(A6) ** (1 / 6.)
    eta0 = max(d4, d6)
    if near(eta0, expm_spec.THETA[0]) and ell(absA, normA, 0, 3) == 0:
        return min(margins)
    if near(eta0, expm_spec.THETA[1]) and ell(absA, normA, 1, 5) == 0:
        return min(margins)
    d8 = expm_spec.norm1(A4 @ A4) ** 0.125
    eta2 = max(d6, d8)
    if near(eta2, expm_spec.THETA[2]) and ell(absA, normA, 2, 7) == 0:
        return min(margins)
    if near(eta2, expm_spec.THETA[3]) and ell(absA, normA, 3, 9) == 0:
        return min(margins)
    eta4 = min(eta2, max(d8, expm_spec.norm1(A4 @ A6) ** 0.1))
    q = math.log2(eta4 / expm_spec.THETA[4])
    if q > -1.0:
        margins.append(abs(q - round(q)) * math.log(2.0))
    s = max(int(math.ceil(q)), 0)
    ell(absA * 2.0 ** -s, normA * 2.0 ** -s, 4, 13)
    return min(margins)


def _rank(m, s):
    return (m if m < 13 else 13 + s)


def ell_for(M, m, s, at=0.5, lo=1e-12, hi=1e8):
    """l > 0 at which `oracle.expm_spec.pick(l M)` gives (m, s): the (m, s) order rises with l; the interval of l
    that gives (m, s) is bracketed by bisection over log l and the point a fraction `at` into it (in log l) returned,
    by default its log-midpoint.  None if no l gives it."""
    target = _rank(m, s)
    nm = expm_spec.norm1(M)
    rank = lambda x: _rank(*expm_spec.pick(np.exp(x) / nm * M)[:2])   # x = log(l ||M||_1)

    def edge(strict):                   # smallest x with rank(x) > target (strict) or >= target
        a, b = np.log(lo), np.log(hi)
        for _ in range(20):
            c = 0.5 * (a + b)
            r = rank(c)
            if r > target or (not strict and r == target):
                b = c
            else:
                a = c
        return b

    x0, x1 = edge(False), edge(True)
    if not x1 > x0:
        return None
    ell = float(np.exp(x0 + at * (x1 - x0)) / nm)
    return ell if expm_spec.pick(ell * M)[:2] == (m, s) else None


def shape_problem(Np, n, zscore, seed=0, c=None):
    """Forecast problem with exactly Np series under rule 'all' and no SST: (y, sic, ell, sig).  ell = c / ||M||_1
    (c cycles through 0.05, 1.5, 6 with Np: Pade orders 5..13 at s = 0..2), sig keeps cond(K) ~ 1e2..1e3 for both
    the z-scored and the raw (x 30) series."""
    y, sic, _ = series(1000 * Np + 7 * n + seed, n, Np, scale=1.0 if zscore else 30.0)
    if Np < 2:
        return y, sic, 1e-2, 1.0
    _, _, M = og.design(og.select_predictors(y, sic, None, "all"), zscore)
    c = (0.05, 1.5, 6.0)[Np % 3] if c is None else c
    return y, sic, c / expm_spec.norm1(M), 1.0 if zscore else 900.0


# Np values on both sides of every shape boundary of k_gp_forecast: 16-wide LU panels, 64 x 64 GEMM tiles, the 8 / 4 /
# 2 / 1 row slices of the |A|^p power iteration (Np <= 32 / 64 / 128 / above), a second 256-thread pass of the column
# loops and of the predictor compaction, and the 520-row LU panel capacity
NP_SWEEP = (2, 3, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 300, 383, 384, 519, 520)
