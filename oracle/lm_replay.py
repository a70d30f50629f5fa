"""TEST INFRASTRUCTURE ONLY -- scalar restatement of the survey-mode Levenberg-Marquardt update
(``rbvfit_b200/csrc/rbv_lm.cuh``, DESIGN.md section 16).

Python floats are IEEE doubles and each operation below is rounded once, as the kernel's ``__dadd_rn`` /
``__dsub_rn`` / ``__dmul_rn`` / ``__ddiv_rn`` / ``__dsqrt_rn`` are; the loops run in the kernel's orders.  Driven by a
one-sightline ``GpuLikelihood.lnlike_and_fisher`` (whose rows are bit-identical to the survey-mode Fisher rows), it
gives the device's x, chi^2, n_evals and status bit for bit.  Driven by any other ``fisher_fn`` (the Fisher oracle),
it is a second implementation of ``rbvfit_b200.lm.levenberg_marquardt``'s rules.
"""
from __future__ import annotations

import math
from typing import NamedTuple

import numpy as np

STATUS_FAILED, STATUS_MAX_EVALS, STATUS_FTOL, STATUS_XTOL = -1, 0, 1, 2


class ReplayResult(NamedTuple):
    x: np.ndarray
    chi2: float
    cov: np.ndarray
    n_evals: int
    status: int
    flags: int             # bit 0: F_ff not positive definite at the end (cov left NaN)


def _clip(v, lo, hi):
    return min(max(v, lo), hi)


def free_set(x, g, F, lb, ub):
    return [i for i in range(len(x))
            if F[i][i] > 0.0 and not ((x[i] <= lb[i] and g[i] < 0.0) or (x[i] >= ub[i] and g[i] > 0.0))]


def cholesky(F, idx, lam=None):
    """Lower factor of F_ff (+ lam diag F_ff), or None when a pivot is not > 0."""
    m = len(idx)
    L = [[0.0] * m for _ in range(m)]
    for j in range(m):
        f = F[idx[j]][idx[j]]
        s = f if lam is None else f + lam * f
        for k in range(j):
            s = s - L[j][k] * L[j][k]
        if not s > 0.0:
            return None
        d = math.sqrt(s)
        L[j][j] = d
        for i in range(j + 1, m):
            t = F[idx[i]][idx[j]]
            for k in range(j):
                t = t - L[i][k] * L[j][k]
            L[i][j] = t / d
    return L


def covariance(x, g, F, lb, ub):
    """(cov, flags) as the kernel's finish step writes them."""
    n = len(x)
    cov = np.full((n, n), np.nan)
    idx = free_set(x, g, F, lb, ub)
    m = len(idx)
    if m == 0:
        return cov, 0
    L = cholesky(F, idx)
    if L is None:
        return cov, 1
    Li = [[0.0] * m for _ in range(m)]
    for c in range(m):
        for i in range(c, m):
            t = 1.0 if i == c else 0.0
            for k in range(c, i):
                t = t - L[i][k] * Li[k][c]
            Li[i][c] = t / L[i][i]
    for i in range(m):
        for j in range(m):
            t = 0.0
            for k in range(max(i, j), m):
                t = t + Li[k][i] * Li[k][j]
            cov[idx[i], idx[j]] = t
    return cov, 0


def _finite(v, g, F):
    return math.isfinite(v) and bool(np.all(np.isfinite(g))) and bool(np.all(np.isfinite(F)))


def run(fisher_fn, theta0, lb, ub, max_evals=200, ftol=1e-10, xtol=1e-10) -> ReplayResult:
    """``fisher_fn(theta) -> (lnlike, grad, F)``; the kernel's iteration, one evaluation per candidate."""
    lb = [float(v) for v in lb]
    ub = [float(v) for v in ub]
    n = len(lb)
    xc = [_clip(float(v), lb[i], ub[i]) for i, v in enumerate(np.asarray(theta0, dtype=np.float64))]

    def evaluate(point):
        ll, g, F = fisher_fn(np.array(point))
        g, F = np.asarray(g, dtype=np.float64), np.asarray(F, dtype=np.float64)
        return -2.0 * float(ll), [float(v) for v in g], [[float(v) for v in row] for row in F]

    chi2, g, F = evaluate(xc)
    n_evals = 1
    x = list(xc)
    if not _finite(chi2, g, F):
        return ReplayResult(np.array(x), chi2, np.full((n, n), np.nan), n_evals, STATUS_FAILED, 0)
    lam, nu = 0.1, 2.0

    def finish(status):
        cov, flags = covariance(x, g, F, lb, ub)
        return ReplayResult(np.array(x), chi2, cov, n_evals, status, flags)

    while True:
        while True:                                    # propose the next candidate
            idx = free_set(x, g, F, lb, ub)
            if not idx:
                return finish(STATUS_XTOL)
            L = cholesky(F, idx, lam)
            if L is None:
                lam = lam * nu
                nu = nu * 2.0
                if lam > 1e30:
                    return finish(STATUS_FAILED)
                continue
            m = len(idx)
            y = [0.0] * m
            for i in range(m):
                t = g[idx[i]]
                for k in range(i):
                    t = t - L[i][k] * y[k]
                y[i] = t / L[i][i]
            for i in range(m - 1, -1, -1):
                t = y[i]
                for k in range(i + 1, m):
                    t = t - L[k][i] * y[k]
                y[i] = t / L[i][i]
            step = dict(zip(idx, y))
            sd = sx = 0.0
            xc = [0.0] * n
            for i in range(n):
                v = _clip(x[i] + step.get(i, 0.0), lb[i], ub[i])
                xc[i] = v
                dd = v - x[i]
                sd = sd + dd * dd
                sx = sx + x[i] * x[i]
            if math.sqrt(sd) <= xtol * (math.sqrt(sx) + xtol):
                return finish(STATUS_XTOL)
            if n_evals >= max_evals:
                return finish(STATUS_MAX_EVALS)
            break
        chi2_n, g_n, F_n = evaluate(xc)
        n_evals += 1
        gd = q = 0.0
        for i in range(n):
            di = xc[i] - x[i]
            gd = gd + g[i] * di
            t = 0.0
            for j in range(n):
                t = t + F[i][j] * (xc[j] - x[j])
            q = q + di * t
        pred = 2.0 * gd - q
        actual = chi2 - chi2_n
        rho = actual / pred if (_finite(chi2_n, g_n, F_n) and pred > 0.0) else -1.0
        if rho > 0.0:
            t = 2.0 * rho - 1.0
            lam = lam * max(1.0 / 3.0, 1.0 - t * t * t)
            nu = 2.0
            x, g, F = xc, g_n, F_n
            chi2_old, chi2 = chi2, chi2_n
            if actual <= ftol * abs(chi2_old):
                return finish(STATUS_FTOL)
        else:
            lam = lam * nu
            nu = nu * 2.0
