"""Bounded Levenberg-Marquardt on chi^2 = -2 lnlike, driven by the device's Gauss-Newton matrix.

``fisher_fn(theta) -> (lnlike, grad, F)`` is one evaluation: the value, its gradient g = d lnlike / d theta and the
Gauss-Newton matrix F = sum_p w_p dM_p/dtheta_i dM_p/dtheta_j (``GpuLikelihood.lnlike_and_fisher``).  With
chi^2 = -2 lnlike + const, grad chi^2 = -2 g and the Gauss-Newton approximation of its Hessian is 2 F, so the damped
step solves (F_ff + lambda diag(F_ff)) delta_f = g_f over the free parameters f.  Every candidate costs one call,
which is both the acceptance test and the next linearisation.  Pure numpy: the same driver runs on any callable.
"""
from __future__ import annotations

import warnings
from typing import NamedTuple

import numpy as np

STATUS_FAILED, STATUS_MAX_EVALS, STATUS_FTOL, STATUS_XTOL = -1, 0, 1, 2


class LMResult(NamedTuple):
    x: np.ndarray          # best point
    chi2: float            # -2 lnlike at x (chi^2 up to the constant sum_p log w_p)
    cov: np.ndarray        # inv(F_ff) over the free set; NaN rows / columns for pinned or unconstrained parameters
    n_evals: int           # fisher_fn calls
    status: int            # STATUS_*: > 0 converged
    message: str


def free_set(theta, grad, fisher, lb, ub):
    """Parameters the data constrain (F_ii > 0) minus those on a bound whose gradient points out of the box."""
    d = np.diag(fisher)
    pinned = ((theta <= lb) & (grad < 0)) | ((theta >= ub) & (grad > 0))
    return (d > 0) & ~pinned


def covariance(fisher, free):
    """inv(F_ff) embedded in an ndim x ndim matrix of NaN (the Delta chi^2 = 1 covariance); pinv with a warning when
    F_ff is not positive definite."""
    n = fisher.shape[0]
    cov = np.full((n, n), np.nan)
    idx = np.flatnonzero(free)
    if idx.size == 0:
        return cov
    Ff = fisher[np.ix_(idx, idx)]
    try:
        L = np.linalg.cholesky(Ff)
        Linv = np.linalg.solve(L, np.eye(idx.size))
        inv = Linv.T @ Linv
    except np.linalg.LinAlgError:
        warnings.warn("Fisher matrix is not positive definite on the free parameters: covariance from pinv")
        inv = np.linalg.pinv(Ff)
    cov[np.ix_(idx, idx)] = inv
    return cov


def _damped_step(Ff, gf, lam):
    A = Ff + lam * np.diag(np.diag(Ff))
    L = np.linalg.cholesky(A)
    return np.linalg.solve(L.T, np.linalg.solve(L, gf))


def levenberg_marquardt(fisher_fn, theta0, lb, ub, max_evals=200, ftol=1e-10, xtol=1e-10) -> LMResult:
    """Maximise lnlike inside [lb, ub] from ``theta0`` (clipped into the box).  Stops when an accepted step lowers
    chi^2 by at most ``ftol`` * |chi^2|, when a step is at most ``xtol`` * (|theta| + xtol) long, or after
    ``max_evals`` calls of ``fisher_fn``.  The damping follows Nielsen's rule on rho = actual / predicted reduction,
    predicted = 2 g.delta - delta.F.delta; a candidate with non-finite chi^2 is rejected."""
    lb = np.asarray(lb, dtype=np.float64)
    ub = np.asarray(ub, dtype=np.float64)
    x = np.clip(np.asarray(theta0, dtype=np.float64), lb, ub)
    ll, g, F = fisher_fn(x)
    n_evals = 1
    chi2 = -2.0 * float(ll)
    if not (np.isfinite(chi2) and np.all(np.isfinite(g)) and np.all(np.isfinite(F))):
        return LMResult(x, chi2, np.full((x.size, x.size), np.nan), n_evals, STATUS_FAILED,
                        "lnlike, gradient or Fisher matrix not finite at the start")
    lam, nu = 0.1, 2.0          # 1e-3 lets the first Gauss-Newton step of C4 clip a b onto its bound
    status, message = STATUS_MAX_EVALS, "maximum number of evaluations reached"
    while True:
        free = free_set(x, g, F, lb, ub)
        if not free.any():
            status, message = STATUS_XTOL, "no free parameter left"
            break
        idx = np.flatnonzero(free)
        Ff, gf = F[np.ix_(idx, idx)], g[idx]
        try:
            step = _damped_step(Ff, gf, lam)
        except np.linalg.LinAlgError:
            lam *= nu
            nu *= 2.0
            if lam > 1e30:
                status, message = STATUS_FAILED, "damped system could not be factorised"
                break
            continue
        delta = np.zeros_like(x)
        delta[idx] = step
        xn = np.clip(x + delta, lb, ub)
        delta = xn - x
        small = np.linalg.norm(delta) <= xtol * (np.linalg.norm(x) + xtol)
        if small:
            status, message = STATUS_XTOL, "step below xtol"
            break
        if n_evals >= max_evals:
            break
        ll_n, g_n, F_n = fisher_fn(xn)
        n_evals += 1
        chi2_n = -2.0 * float(ll_n)
        pred = 2.0 * float(g @ delta) - float(delta @ F @ delta)
        actual = chi2 - chi2_n
        ok = np.isfinite(chi2_n) and np.all(np.isfinite(g_n)) and np.all(np.isfinite(F_n)) and pred > 0
        rho = actual / pred if ok else -1.0
        if rho > 0:
            x, g, F = xn, g_n, F_n
            chi2_old, chi2 = chi2, chi2_n
            lam *= max(1.0 / 3.0, 1.0 - (2.0 * rho - 1.0) ** 3)
            nu = 2.0
            if actual <= ftol * abs(chi2_old):
                status, message = STATUS_FTOL, "relative chi^2 decrease below ftol"
                break
        else:
            lam *= nu
            nu *= 2.0
    cov = covariance(F, free_set(x, g, F, lb, ub))
    return LMResult(x, chi2, cov, n_evals, status, message)
