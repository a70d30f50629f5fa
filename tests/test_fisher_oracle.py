"""CPU: the Jacobian / Fisher oracle (oracle/voigt_fisher_oracle.py) against Richardson differences of the forward
model and against the gradient oracle, and the bounded Levenberg-Marquardt driver (rbvfit_b200.lm) run on the oracle
against scipy's least_squares."""
import os
import sys

import numpy as np
import pytest

from golden_util import Golden

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gradient_oracle import gradient_cases  # noqa: E402

CASES = ["C1", "C1_f32err", "C1_coslsf", "C1_smallb", "C3", "C4", "piecewise", "C1_ndim_gt_3C"]


def _case(name):
    return next(c for c in gradient_cases() if c[0] == name)


@pytest.mark.parametrize("case", CASES)
def test_oracle_jacobian_vs_richardson(case):
    from oracle import voigt_fisher_oracle as vf
    _name, comp, theta = _case(case)
    worst = 0.0
    for d in comp.values():
        ncol = 3 * d["model"].total_components
        J = vf.model_jacobian(d, theta)
        fd = vf.model_jacobian_fd(d, theta)
        assert np.all(J[ncol:] == 0.0) and np.all(fd[ncol:] == 0.0)
        for i in range(ncol):
            scale = np.max(np.abs(J[i]))
            err = np.max(np.abs(J[i] - fd[i]))
            if scale == 0.0:
                assert err == 0.0
                continue
            worst = max(worst, err / scale)
    print(case, "max |J - FD| / max|J_col|", worst)
    assert worst <= 1e-6


@pytest.mark.parametrize("case", CASES)
def test_oracle_jtr_vs_gradient_oracle(case):
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_grad_oracle as vg
    from oracle import voigt_oracle as vo
    _name, comp, theta = _case(case)
    ll, g, F = vf.lnlike_fisher(comp, theta)
    assert ll == vo.lnlike(comp, theta)
    ref = vg.lnlike_grad(comp, theta)
    G = vg.grad_scale(comp, theta)
    ncol = 3 * next(iter(comp.values()))["model"].total_components
    assert np.all(g[ncol:] == 0.0) and np.all(F[ncol:] == 0.0) and np.all(F[:, ncol:] == 0.0)
    err = np.abs(g[:ncol] - ref[:ncol]) / G[:ncol]
    print(case, "max |J^T r - grad| / G", err.max())
    assert err.max() <= 1e-12


def _residuals(comp):
    """least_squares form of the same chi^2: residuals (D - M) sqrt(w) and their Jacobian -J sqrt(w)."""
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_oracle as vo

    def fun(x):
        return np.concatenate([(d["flux"] - vo.model_flux(d["model"], x, d["wave"])) * np.sqrt(d["inv_sigma2"])
                               for d in comp.values()])

    def jac(x):
        return np.concatenate([-(vf.model_jacobian(d, x) * np.sqrt(d["inv_sigma2"])[None, :]).T
                               for d in comp.values()])
    return fun, jac


def _chi2(comp, x):
    from oracle import voigt_oracle as vo
    return float(sum(np.sum((d["flux"] - vo.model_flux(d["model"], x, d["wave"])) ** 2 * d["inv_sigma2"])
                     for d in comp.values()))


@pytest.mark.parametrize("case", ["C1", "C4"])
def test_lm_on_oracle_vs_least_squares(case):
    import scipy.optimize as op
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_grad_oracle as vg
    from oracle import voigt_oracle as vo
    from rbvfit_b200.lm import levenberg_marquardt
    g = Golden(case)
    comp = g.oracle_compiled()
    lb, ub = g.lb.astype(float), g.ub.astype(float)
    theta0 = np.clip(g.thetas[0], lb, ub)
    res = levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), theta0, lb, ub)
    assert res.status > 0, res.message
    fun, jac = _residuals(comp)
    ref = op.least_squares(fun, theta0, jac=jac, bounds=(lb, ub), method="trf", x_scale="jac", ftol=1e-15,
                           xtol=1e-15, gtol=1e-15, max_nfev=2000)
    c_lm, c_ref = _chi2(comp, res.x), _chi2(comp, ref.x)
    sig = np.sqrt(np.diag(res.cov))
    dx = np.abs(res.x - ref.x) / sig
    lbfgs = op.minimize(lambda x: (-2.0 * vo.lnlike(comp, x), -2.0 * vg.lnlike_grad(comp, x)), theta0, jac=True,
                        method="L-BFGS-B", bounds=list(zip(lb, ub)), options={"maxfun": 5000})
    print(case, "chi2 LM", c_lm, "least_squares", c_ref, "L-BFGS-B", _chi2(comp, lbfgs.x),
          "| evaluations: LM", res.n_evals, "least_squares", ref.nfev, "L-BFGS-B", lbfgs.nfev,
          "| max |dx| / sigma", dx.max())
    assert abs(c_lm - c_ref) <= 1e-9 * c_ref
    assert np.all(np.isfinite(sig)) and dx.max() <= 1e-3


def test_lm_bound_pins_parameter():
    from oracle import voigt_fisher_oracle as vf
    from rbvfit_b200.lm import levenberg_marquardt
    g = Golden("C1")
    comp = g.oracle_compiled()
    lb, ub = g.lb.astype(float), g.ub.astype(float)
    theta0 = np.clip(g.thetas[0], lb, ub)
    free = levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), theta0, lb, ub)
    i = 3                                              # b of the second component
    ub2 = ub.copy()
    ub2[i] = free.x[i] - 3.0 * np.sqrt(free.cov[i, i])
    assert ub2[i] > lb[i]
    res = levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), np.minimum(theta0, ub2), lb, ub2)
    assert res.status > 0, res.message
    err = np.sqrt(np.diag(res.cov))
    assert res.x[i] == ub2[i]
    assert np.isnan(err[i]) and np.all(np.isnan(res.cov[i])) and np.all(np.isnan(res.cov[:, i]))
    assert np.all(np.isfinite(np.delete(err, i)))


def test_lm_extra_columns_stay_put():
    from oracle import voigt_fisher_oracle as vf
    from rbvfit_b200.lm import levenberg_marquardt
    _name, comp, theta = _case("C1_ndim_gt_3C")
    g = Golden("C1")
    lb = np.concatenate([g.lb, [-5.0, -5.0]])
    ub = np.concatenate([g.ub, [5.0, 5.0]])
    theta0 = np.clip(theta, lb, ub)
    res = levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), theta0, lb, ub)
    assert res.status > 0, res.message
    err = np.sqrt(np.diag(res.cov))
    assert np.array_equal(res.x[6:], theta0[6:])
    assert np.all(np.isnan(err[6:])) and np.all(np.isfinite(err[:6]))


def test_lm_stops_at_max_evals_and_rejects_bad_start():
    from oracle import voigt_fisher_oracle as vf
    from rbvfit_b200 import lm
    g = Golden("C1")
    comp = g.oracle_compiled()
    lb, ub = g.lb.astype(float), g.ub.astype(float)
    theta0 = np.clip(g.thetas[0], lb, ub)
    res = lm.levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), theta0, lb, ub, max_evals=2)
    assert res.n_evals == 2 and res.status == lm.STATUS_MAX_EVALS
    bad = theta0.copy()
    bad[0] = np.nan
    res = lm.levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), bad, lb, ub)
    assert res.status == lm.STATUS_FAILED and res.n_evals == 1
