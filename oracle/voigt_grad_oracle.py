"""TEST INFRASTRUCTURE ONLY -- numpy/scipy restatement of the analytic gradient of ``vfit.lnlike``.

Kept beside ``voigt_oracle`` (which stays pinned to the reference fixtures) and built on its forward model:
  * ``voigt_H_derivs(x, a)``   H, dH/dx, dH/da: scipy.special.wofz where |z|^2 is small, the differentiated
                               asymptotic series of w(z) beyond (w' = -2 z w + 2i/sqrt(pi) cancels in the wings)
  * ``lnlike_grad``            the adjoint of DESIGN.md section 14 (one forward and one backward pass)
  * ``grad_scale``             G_i = sum_{l,q} |g_q| |d tau_lq / d theta_i|, the magnitude gradient errors are
                               measured against (d lnL / d theta_i itself cancels near an optimum)
  * ``lnlike_fd``              Richardson-extrapolated central differences of ``voigt_oracle.lnlike``
"""
from __future__ import annotations

import numpy as np
from scipy.special import wofz

from . import voigt_oracle as vo

C_KMS = 299792.458
# wofz and w' = -2 z w + 2i/sqrt(pi) below |z|^2 = 64, or below 36 when a >= 1 (there w' would lose digits to the
# cancellation against 2i/sqrt(pi), and the series has no exponentially small term left to miss); 40 terms of the
# series beyond (truncation ~ exp(-|z|^2) relative to |w|)
_D_WOFZ, _D_WOFZ_BIG_A = 64.0, 36.0
_N_ASYM = 40


def _asym_terms(z):
    """w, w' and w + z w' from w(z) ~ (i/sqrt(pi)) sum_k c_k z^-(2k+1), c_k = (2k-1)!!/2^k."""
    zeta = 1.0 / z
    s = zeta * zeta
    c = np.ones(_N_ASYM)
    for k in range(1, _N_ASYM):
        c[k] = c[k - 1] * (2 * k - 1) * 0.5
    S0 = np.zeros_like(z)
    S1 = np.zeros_like(z)
    S2 = np.zeros_like(z)
    for k in range(_N_ASYM - 1, -1, -1):
        S0 = S0 * s + c[k]
        S1 = S1 * s + (2 * k + 1) * c[k]
        S2 = S2 * s + (-2 * k) * c[k]
    pref = 1j / np.sqrt(np.pi)
    return pref * zeta * S0, -pref * s * S1, pref * zeta * S2


def voigt_H_derivs(x, a, with_E=False):
    """H = Re w(x + i a), H_x, H_a (and E = H + x H_x + a H_a with ``with_E``), elementwise."""
    x, a = np.broadcast_arrays(np.asarray(x, dtype=np.float64), np.asarray(a, dtype=np.float64))
    z = x + 1j * a
    d = x * x + a * a
    near = d < np.where(a >= 1.0, _D_WOFZ_BIG_A, _D_WOFZ)
    w = np.empty(z.shape, dtype=complex)
    dw = np.empty(z.shape, dtype=complex)
    wE = np.empty(z.shape, dtype=complex)
    if near.any():
        zn = z[near]
        wn = wofz(zn)
        dwn = -2.0 * zn * wn + 2j / np.sqrt(np.pi)
        w[near], dw[near], wE[near] = wn, dwn, wn + zn * dwn
    far = ~near
    if far.any():
        w[far], dw[far], wE[far] = _asym_terms(z[far])
    H, Hx, Ha = w.real, dw.real, -dw.imag
    if with_E:
        return H, Hx, Ha, wE.real
    return H, Hx, Ha


def _line_terms(m, theta, wave):
    """Per (line, pixel): S, A, u, H, H_x, E and the component of each line."""
    theta = np.asarray(theta, dtype=np.float64)
    N = 10 ** theta[m.N_indices]
    b = theta[m.b_indices]
    v = theta[m.v_indices]
    lam0 = m.atomic_lambda0
    gam = np.asarray(m.atomic_gamma, dtype=np.float64)
    f = np.asarray(m.atomic_f, dtype=np.float64)
    c_freq = 2.99792458e18
    b_f = b / lam0 * 1e13
    nu0 = c_freq / lam0
    konst = 4.48898479507e3 / (nu0 * b)
    a = gam / (4 * np.pi * b_f)
    zt = m.z_factors * (1 + v / C_KMS) - 1
    A = c_freq * (1 + zt) / b_f
    B = nu0 / b_f
    S = N * f * konst
    u = 1.0 / np.asarray(wave, dtype=np.float64)
    x = A[:, None] * u[None, :] - B[:, None]
    H, Hx, Ha, E = voigt_H_derivs(x, a[:, None], with_E=True)
    return dict(S=S, A=A, b=b, v=v, u=u, H=H, Hx=Hx, E=E)


def _conv_taps(m):
    """Taps of M = taps * F exactly as ``voigt_oracle.model_flux`` applies them (None: no LSF)."""
    if m.kernel_taps is None:
        return None
    t = np.asarray(m.kernel_taps, dtype=np.float64)
    return t / t.sum() if m.kernel_kind == "custom" else t


def _conv(F, taps):
    K = taps.size
    h = K // 2
    P = F.size
    idx = np.arange(P)
    M = np.zeros(P)
    for j in range(K):     # M_p = sum_j taps[j] F[clamp(p + h - j)]  (true convolution, edges replicated)
        M += taps[j] * F[np.clip(idx + h - j, 0, P - 1)]
    return M


def _conv_T(r, taps):
    K = taps.size
    h = K // 2
    P = r.size
    idx = np.arange(P)
    s = np.zeros(P)
    for j in range(K):
        np.add.at(s, np.clip(idx + h - j, 0, P - 1), taps[j] * r)
    return s


def _adjoint(d, theta):
    """g_q = d lnL / d tau_q for one instrument dict of ``voigt_oracle.compile_instruments``."""
    m = d["model"]
    tau = vo.model_flux(m, theta, d["wave"], return_tau=True)
    F = np.exp(-tau)
    taps = _conv_taps(m)
    M = F if taps is None else _conv(F, taps)
    r = (d["flux"] - M) * d["inv_sigma2"]
    s = r if taps is None else _conv_T(r, taps)
    return -F * s


def lnlike_grad(compiled, theta):
    """d vfit.lnlike / d theta (length of theta; columns beyond 3C are 0)."""
    theta = np.asarray(theta, dtype=np.float64)
    grad = np.zeros(theta.size)
    for d in compiled.values():
        m = d["model"]
        g = _adjoint(d, theta)
        t = _line_terms(m, theta, d["wave"])
        TN = t["H"] @ g
        Tb = t["E"] @ g
        Tv = t["Hx"] @ (g * t["u"])
        np.add.at(grad, m.N_indices, np.log(10.0) * t["S"] * TN)
        np.add.at(grad, m.b_indices, -(t["S"] / t["b"]) * Tb)
        np.add.at(grad, m.v_indices, t["S"] * t["A"] * Tv / (C_KMS + t["v"]))
    return grad


def grad_scale(compiled, theta):
    """G_i = sum_{l,q} |g_q| |d tau_lq / d theta_i|."""
    theta = np.asarray(theta, dtype=np.float64)
    G = np.zeros(theta.size)
    for d in compiled.values():
        m = d["model"]
        g = np.abs(_adjoint(d, theta))
        t = _line_terms(m, theta, d["wave"])
        np.add.at(G, m.N_indices, np.log(10.0) * t["S"] * (np.abs(t["H"]) @ g))
        np.add.at(G, m.b_indices, (t["S"] / np.abs(t["b"])) * (np.abs(t["E"]) @ g))
        np.add.at(G, m.v_indices, t["S"] * np.abs(t["A"]) * (np.abs(t["Hx"]) @ (g * t["u"])) / np.abs(C_KMS + t["v"]))
    return G


def lnlike_fd(compiled, theta, steps=None):
    """Richardson-extrapolated central differences of ``voigt_oracle.lnlike`` (error O(h^4))."""
    theta = np.asarray(theta, dtype=np.float64)
    if steps is None:
        steps = np.maximum(1e-3 * np.abs(theta), 1e-4)
    out = np.zeros(theta.size)
    for i in range(theta.size):
        def D(h):
            e = np.zeros(theta.size)
            e[i] = h
            return (vo.lnlike(compiled, theta + e) - vo.lnlike(compiled, theta - e)) / (2 * h)
        h = steps[i]
        out[i] = (4.0 * D(h / 2) - D(h)) / 3.0
    return out
