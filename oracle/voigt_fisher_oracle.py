"""TEST INFRASTRUCTURE ONLY -- numpy/scipy restatement of the model Jacobian and the Gauss-Newton (Fisher) matrix of
``vfit.lnlike`` (DESIGN.md section 15).

Built on ``voigt_grad_oracle`` (its per-line terms) and ``voigt_oracle`` (the forward model and its LSF); both stay
untouched:
  * ``model_jacobian(d, theta)``     dM/dtheta [ndim, P]: per column -F dtau/dtheta_i, then the LSF exactly as
                                     ``voigt_oracle.model_flux`` applies it
  * ``lnlike_fisher(compiled, theta)`` (lnlike, sum_p r_p dM_p/dtheta, sum_p w_p dM_p/dtheta_i dM_p/dtheta_j)
  * ``model_jacobian_fd(d, theta)``  Richardson-extrapolated central differences of ``voigt_oracle.model_flux``
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

from . import voigt_grad_oracle as vg
from . import voigt_oracle as vo


def _apply_lsf(m, col):
    if m.kernel_taps is None:
        return col
    if m.kernel_kind == "gaussian":
        return ndimage.convolve1d(col, m.kernel_taps, mode="nearest")
    return vo.convolve_extend(col, m.kernel_taps)


def model_jacobian(d, theta):
    """dM_p/dtheta_i of one instrument dict of ``voigt_oracle.compile_instruments``: [len(theta), P], rows beyond
    3C are 0."""
    theta = np.asarray(theta, dtype=np.float64)
    m = d["model"]
    t = vg._line_terms(m, theta, d["wave"])
    F = np.exp(-vo.model_flux(m, theta, d["wave"], return_tau=True))
    P = F.size
    dtau = np.zeros((theta.size, P))
    S = t["S"][:, None]
    np.add.at(dtau, m.N_indices, np.log(10.0) * S * t["H"])
    np.add.at(dtau, m.b_indices, -(S / t["b"][:, None]) * t["E"])
    np.add.at(dtau, m.v_indices, (S * t["A"][:, None] / (vg.C_KMS + t["v"][:, None])) * t["Hx"] * t["u"][None, :])
    J = np.zeros((theta.size, P))
    for i in range(3 * m.total_components):
        J[i] = _apply_lsf(m, -F * dtau[i])
    return J


def lnlike_fisher(compiled, theta):
    """(vfit.lnlike, its gradient sum_p r_p dM_p/dtheta, the Gauss-Newton matrix sum_p w_p J_ip J_jp)."""
    theta = np.asarray(theta, dtype=np.float64)
    grad = np.zeros(theta.size)
    fisher = np.zeros((theta.size, theta.size))
    for d in compiled.values():
        J = model_jacobian(d, theta)
        r = (d["flux"] - vo.model_flux(d["model"], theta, d["wave"])) * d["inv_sigma2"]
        grad += J @ r
        fisher += (J * d["inv_sigma2"][None, :]) @ J.T
    return vo.lnlike(compiled, theta), grad, fisher


def model_jacobian_fd(d, theta, steps=None):
    """Richardson-extrapolated central differences of ``voigt_oracle.model_flux`` (error O(h^4)): [len(theta), P]."""
    theta = np.asarray(theta, dtype=np.float64)
    if steps is None:
        steps = np.maximum(1e-3 * np.abs(theta), 1e-4)
    m = d["model"]
    out = np.zeros((theta.size, np.size(d["wave"])))
    for i in range(theta.size):
        def D(h):
            e = np.zeros(theta.size)
            e[i] = h
            return (vo.model_flux(m, theta + e, d["wave"]) - vo.model_flux(m, theta - e, d["wave"])) / (2 * h)
        h = steps[i]
        out[i] = (4.0 * D(h / 2) - D(h)) / 3.0
    return out
