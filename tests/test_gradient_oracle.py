"""CPU: the gradient oracle (oracle/voigt_grad_oracle.py) -- H, dH/dx, dH/da against mpmath at 40 digits, and the
adjoint gradient of vfit.lnlike against Richardson-extrapolated central differences of the oracle's lnlike."""
import numpy as np
import pytest

from golden_util import Golden


def derivative_lattice(seed=3):
    """a in [1e-8, 20], |x| in [0, 3e4]: core, near wing and far wing of every damping regime."""
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.uniform(0, 10, 500), np.exp(rng.uniform(np.log(10), np.log(3e4), 200)),
                        [0.0, 1e4, 3e4, 8.0, 6.0]])
    x = x * rng.choice([-1.0, 1.0], x.size)
    a = np.exp(rng.uniform(np.log(1e-8), np.log(20.0), x.size))
    return x, a


def mpmath_derivs(x, a):
    """H, H_x, H_a from w = exp(-z^2) erfc(-iz) and w' = -2 z w + 2i/sqrt(pi) at 40 digits."""
    import mpmath
    out = np.empty((x.size, 3))
    with mpmath.workdps(40):
        for i, (xv, av) in enumerate(zip(x, a)):
            z = mpmath.mpc(float(xv), float(av))
            w = mpmath.exp(-z * z) * mpmath.erfc(-1j * z)
            dw = -2 * z * w + 2j / mpmath.sqrt(mpmath.pi)
            out[i] = float(w.real), float(dw.real), float(-dw.imag)
    return out


def derivative_errors(got, ref):
    """Relative error of H, H_x, H_a against max(|ref|, 1e-3 H)."""
    return [float(np.max(np.abs(got[c] - ref[:, c]) / np.maximum(np.abs(ref[:, c]), 1e-3 * ref[:, 0])))
            for c in range(3)]


def test_oracle_voigt_derivatives_vs_mpmath():
    from oracle import voigt_grad_oracle as vg
    x, a = derivative_lattice()
    ref = mpmath_derivs(x, a)
    err = derivative_errors(vg.voigt_H_derivs(x, a), ref)
    print("oracle H, H_x, H_a max rel err", err)
    assert err[0] <= 1e-12
    # H_x, H_a: scipy's wofz rounding, magnified by the cancellation in w' = -2 z w + 2i/sqrt(pi) where
    # 36 <= |z|^2 < 64 and the series cannot be used (small a: it misses the exp(-x^2) part of Re w): measured 3e-12
    assert err[1] <= 5e-12 and err[2] <= 5e-12


def test_oracle_E_is_the_combination_without_cancellation():
    """E = H + x H_x + a H_a from the differentiated series agrees with the plain combination where nothing cancels,
    and keeps its relative accuracy in the far wing where the plain combination is rounding noise."""
    from oracle import voigt_grad_oracle as vg
    x = np.array([0.5, 3.0, 9.0, 20.0])
    a = np.array([0.01, 0.2, 0.5, 0.05])
    H, Hx, Ha, E = vg.voigt_H_derivs(x, a, with_E=True)
    assert np.allclose(E, H + x * Hx + a * Ha, rtol=1e-10, atol=0)
    # far wing: E ~ (2a/sqrt(pi)) (-q_2 rho^2 + ...) with q_2 = 3/2 + O(a^2): E ~ -3a / (sqrt(pi) x^4)
    x, a = np.array([1e4]), np.array([1e-4])
    _H, _Hx, _Ha, E = vg.voigt_H_derivs(x, a, with_E=True)
    assert abs(E[0] / (-3.0 * a[0] / (np.sqrt(np.pi) * x[0] ** 4)) - 1.0) <= 1e-6


def piecewise_compiled():
    """The piecewise-LSF problem of test_host_logic as oracle instruments with their weight masks."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host_logic import _piecewise_problem
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import lsf
    w, cfg, wave, flux, error, starts, models, lowered = _piecewise_problem()
    entries = lsf.piecewise_lsf_instruments("COS", wave, flux, error, list(zip(starts, models)))
    comp = vo.compile_instruments({n: dict(model=m, wave=d["wave"], flux=d["flux"], error=d["error"])
                                   for (n, d), m in zip(entries.items(), lowered)})
    for n, d in entries.items():
        mask = d["weight_mask"]
        comp[n]["inv_sigma2"] = np.where(mask, comp[n]["inv_sigma2"], 0.0)
        comp[n]["log_inv_sigma2"] = np.where(mask, comp[n]["log_inv_sigma2"], 0.0)
    theta = w["theta_true"] + np.array([0.05, -0.03, 2.0, -1.5, 3.0, -4.0])
    return w, entries, comp, theta


def gradient_cases():
    """(name, oracle compiled instruments, theta) of every configuration the gradient is checked on."""
    out = []
    for case in ("C1", "C1_f32err", "C1_coslsf", "C1_smallb", "C3", "C4"):
        g = Golden(case)
        out.append((case, g.oracle_compiled(), g.thetas[0]))
    _w, _entries, comp, theta = piecewise_compiled()
    out.append(("piecewise", comp, theta))
    g = Golden("C1")
    out.append(("C1_ndim_gt_3C", g.oracle_compiled(), np.concatenate([g.thetas[0], [0.7, -1.3]])))
    return out


@pytest.mark.parametrize("case", ["C1", "C1_f32err", "C1_coslsf", "C1_smallb", "C3", "C4", "piecewise",
                                  "C1_ndim_gt_3C"])
def test_oracle_gradient_vs_richardson(case):
    from oracle import voigt_grad_oracle as vg
    name, comp, theta = next(c for c in gradient_cases() if c[0] == case)
    an = vg.lnlike_grad(comp, theta)
    fd = vg.lnlike_fd(comp, theta)
    G = vg.grad_scale(comp, theta)
    ncol = 3 * next(iter(comp.values()))["model"].total_components
    assert np.all(an[ncol:] == 0.0) and np.all(G[ncol:] == 0.0)
    err = np.abs(an[:ncol] - fd[:ncol]) / G[:ncol]
    print(case, "max |analytic - FD| / G", err.max())
    assert err.max() <= 1e-6
