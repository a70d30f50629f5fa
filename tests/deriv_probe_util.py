"""Per-pixel probes of the derivative kernels (rbv_grad.cuh, rbv_fisher.cuh).

The Jacobian oracle (``oracle.voigt_fisher_oracle.model_jacobian``) is evaluated here on the pixels an LSF needs
around the probed ones only, as ``stream_probe_util.oracle_flux_at`` does for the flux, so a long spectrum costs the
oracle a few thousand pixels per row.

Per-pixel scale.  A Jacobian entry J_ip = sum_m k_m (-F dtau/dtheta_i)[clip(p + h - m)] can be small because it is
far from every line, or because terms of opposite sign cancel.  Errors are measured against the same sum with every
term replaced by its absolute value, so nothing cancels:

    Jhat_ip = sum_m |k_m| F_q sum_{l in c(i)} T_il(q),   q = clip(p + h - m),
    logN column:  T = ln(10) S_l H
    b column:     T = (S_l / b) (H + |x H_x| + a |H_a|)          (E = H + x H_x + a H_a itself crosses 0 near x ~ 1)
    v column:     T = S_l |A_l u| (|H_x| + 1e-3 H) / (c + v)     (H_x itself crosses 0 at line centre)

the per-pixel form of ``voigt_grad_oracle.grad_scale``.

x-conditioning.  x = A u - B is the difference of two numbers of size c / b, so every evaluation of it (oracle,
kernel, mpmath) carries an error of a few eps c / b that has nothing to do with the Voigt tiers.  To first order that
is the change a relative shift of the wavelength grid by n eps makes (A u = B (1 + O(x b / c))), so the allowance for
it is ``x_allowance`` = n eps |lambda dJ/dlambda|, the derivative taken by central differences of the oracle's own
Jacobian.  It matters at b << 1 km/s only (the damping tiers a >= 0.05 of Lyman alpha need b <= 0.12 km/s).

Survey probe.  One sightline per probed pixel p_j (``stream_probe_util.probe_sightlines``: data 2, error 1, weight 1
at p_j only) through ``SightlineBatch.lnlike_and_fisher``: masked pixels add exact zeros, so v = -(2 - M)^2 / 2,
g_i = (2 - M) J_pi and F_ij = J_pi J_pj, hence M = 2 - sqrt(-2 v) and J_pi = g_i / (2 - M) (2 - M in [1, 2])."""
import numpy as np

import stream_probe_util as spu

LN10 = np.log(10.0)
C_KMS = 299792.458


def _stencil(om, P, px):
    """(src [n, K] source pixels of each probed pixel, k [K] normalised taps)."""
    px = np.asarray(px, dtype=np.int64)
    K = spu.n_taps(om)
    if K == 1:
        return px[:, None], np.ones(1)
    taps = np.asarray(om.kernel_taps, dtype=np.float64)
    h = K // 2
    return np.clip(px[:, None] + h - np.arange(K)[None, :], 0, P - 1), taps / taps.sum()


def _columns(om, theta, wn):
    """(F, dtau [len(theta), n], _line_terms) on the pixels ``wn``: the column formulas of
    voigt_fisher_oracle.model_jacobian."""
    from oracle import voigt_grad_oracle as vg
    from oracle import voigt_oracle as vo
    t = vg._line_terms(om, theta, wn)
    F = np.exp(-vo.model_flux(om, theta, wn, return_tau=True))
    S = t["S"][:, None]
    dtau = np.zeros((theta.size, wn.size))
    np.add.at(dtau, om.N_indices, LN10 * S * t["H"])
    np.add.at(dtau, om.b_indices, -(S / t["b"][:, None]) * t["E"])
    np.add.at(dtau, om.v_indices, (S * t["A"][:, None] / (C_KMS + t["v"][:, None])) * t["Hx"] * t["u"][None, :])
    return F, dtau, t


def oracle_jacobian_at(om, theta, wave, px, with_scale=False):
    """The oracle's LSF-applied Jacobian dM_p/dtheta_i [len(theta), len(px)] at pixels ``px`` (columns beyond 3C are
    0); with ``with_scale`` also Jhat (module docstring) of the same shape."""
    from oracle import voigt_grad_oracle as vg
    theta = np.asarray(theta, dtype=np.float64)
    wave = np.asarray(wave, dtype=np.float64)
    src, k = _stencil(om, wave.size, px)
    need = np.unique(src)
    pos = np.searchsorted(need, src)
    F, dtau, t = _columns(om, theta, wave[need])
    J = ((-F * dtau)[:, pos] * k).sum(axis=2)
    if not with_scale:
        return J
    S = t["S"][:, None]
    b_f = t["b"] / om.atomic_lambda0 * 1e13                   # x and a exactly as _line_terms forms them
    a = np.asarray(om.atomic_gamma, dtype=np.float64) / (4 * np.pi * b_f)
    x = t["A"][:, None] * t["u"][None, :] - (2.99792458e18 / om.atomic_lambda0 / b_f)[:, None]
    H, Hx, Ha = vg.voigt_H_derivs(x, a[:, None])
    sc = np.zeros((theta.size, need.size))
    np.add.at(sc, om.N_indices, LN10 * S * H)
    np.add.at(sc, om.b_indices, (S / t["b"][:, None]) * (H + np.abs(x * Hx) + a[:, None] * np.abs(Ha)))
    np.add.at(sc, om.v_indices, (S * np.abs(t["A"][:, None] * t["u"][None, :]) / (C_KMS + t["v"][:, None]))
              * (np.abs(Hx) + 1e-3 * H))
    return J, ((F * sc)[:, pos] * np.abs(k)).sum(axis=2)


def grad_scale_nc(d, theta):
    """Ghat_i = sum_q |g_q| sum_{l in c(i)} T_il(q) with g_q = dlnL/dtau_q and T the terms of Jhat: the gradient's
    magnitude with nothing cancelled.  ``voigt_grad_oracle.grad_scale`` uses |E| and |H_x|, which cross zero near
    x ~ 1 and at line centre, so a b or v column whose lines sit on those zeros has a G_i below the size of the terms
    it is summed from.  ``d``: one instrument dict of ``voigt_oracle.compile_instruments``."""
    from oracle import voigt_grad_oracle as vg
    theta = np.asarray(theta, dtype=np.float64)
    om, wave = d["model"], np.asarray(d["wave"], dtype=np.float64)
    g = np.abs(vg._adjoint(d, theta))
    t = vg._line_terms(om, theta, wave)
    S = t["S"][:, None]
    b_f = t["b"] / om.atomic_lambda0 * 1e13
    a = np.asarray(om.atomic_gamma, dtype=np.float64) / (4 * np.pi * b_f)
    x = t["A"][:, None] * t["u"][None, :] - (2.99792458e18 / om.atomic_lambda0 / b_f)[:, None]
    H, Hx, Ha = vg.voigt_H_derivs(x, a[:, None])
    out = np.zeros(theta.size)
    np.add.at(out, om.N_indices, (LN10 * S * H) @ g)
    np.add.at(out, om.b_indices, ((S / t["b"][:, None]) * (H + np.abs(x * Hx) + a[:, None] * np.abs(Ha))) @ g)
    np.add.at(out, om.v_indices, ((S * np.abs(t["A"][:, None] * t["u"][None, :]) / (C_KMS + t["v"][:, None]))
                                  * (np.abs(Hx) + 1e-3 * H)) @ g)
    return out


def jacobian_scale_at(om, theta, wave, px):
    """Jhat [len(theta), len(px)] (module docstring)."""
    return oracle_jacobian_at(om, theta, wave, px, with_scale=True)[1]


def x_allowance(om, theta, wave, px, n_eps=8.0):
    """The first-order effect of the x-conditioning [len(theta), len(px)] (module docstring):
    n eps sum_m |k_m| F (|lambda d(dtau_i)/dlambda| + |dtau_i| |lambda dtau/dlambda|) at the source pixels.  The
    flux factor and the column carry their own roundings of x (the oracle takes tau from voigt_oracle.model_flux's
    lowering and the columns from _line_terms'), so their effects add in absolute value.  The central-difference
    step moves x by 1e-3 of the narrowest line's Doppler width (x changes by about c / b per unit relative
    wavelength)."""
    from oracle import voigt_oracle as vo
    theta = np.asarray(theta, dtype=np.float64)
    wave = np.asarray(wave, dtype=np.float64)
    src, k = _stencil(om, wave.size, px)
    need = np.unique(src)
    pos = np.searchsorted(need, src)
    wn = wave[need]
    h = 1e-3 * float(np.min(theta[om.b_indices])) / C_KMS
    F, dtau, _t = _columns(om, theta, wn)
    d_col = (_columns(om, theta, wn * (1 + h))[1] - _columns(om, theta, wn * (1 - h))[1]) / (2 * h)
    d_tau = (vo.model_flux(om, theta, wn * (1 + h), return_tau=True)
             - vo.model_flux(om, theta, wn * (1 - h), return_tau=True)) / (2 * h)
    per = F * (np.abs(d_col) + np.abs(dtau) * np.abs(d_tau))
    return n_eps * np.finfo(float).eps * (per[:, pos] * np.abs(k)).sum(axis=2)


def _mp_terms(z):
    """H, H_x, H_a and E = H + x H_x + a H_a = Re(w + z w') of one mpmath complex z, with w = exp(-z^2) erfc(-iz)
    and w' = -2 z w + 2i/sqrt(pi) (the formulas of test_gradient_oracle.mpmath_derivs).  E is formed in mpmath: in
    the far wing it is ~x^-2 times smaller than its terms, which a double-precision sum of H, x H_x and a H_a would
    leave at eps x^2 relative."""
    import mpmath
    w = mpmath.exp(-z * z) * mpmath.erfc(-1j * z)
    dw = -2 * z * w + 2j / mpmath.sqrt(mpmath.pi)
    return float(w.real), float(dw.real), float(-dw.imag), float((w + z * dw).real)


def mpmath_jacobian_at(om, theta, wave, px, dps=60):
    """dM_p/dtheta_i [len(theta), len(px)] with x, a and the line constants formed at ``dps`` digits from the doubles
    the oracle lowers (lambda_0, Gamma, f, z, N = 10^logN, b, v) and H, H_x, H_a, E from w = exp(-z^2) erfc(-iz)
    (``_mp_terms``): independent of the tiers of both the oracle and the kernels.  The LSF, if any, is applied as
    in ``oracle_jacobian_at``.  60 digits: E at |x| = 1e6 cancels about 24 of them."""
    import mpmath
    theta = np.asarray(theta, dtype=np.float64)
    wave = np.asarray(wave, dtype=np.float64)
    src, k = _stencil(om, wave.size, px)
    need = np.unique(src)
    pos = np.searchsorted(need, src)
    L, n = om.n_lines, need.size
    H, Hx, Ha, E = (np.empty((L, n)) for _ in range(4))
    S, A, b, v = (np.empty(L) for _ in range(4))
    with mpmath.workdps(dps):
        mp = mpmath.mpf
        cf, ck, kon = mp(2.99792458e18), mp(C_KMS), mp(4.48898479507e3)
        for l in range(L):
            lam0 = mp(float(om.atomic_lambda0[l]))
            bl, vl = mp(float(theta[om.b_indices[l]])), mp(float(theta[om.v_indices[l]]))
            N = mp(float(10 ** theta[om.N_indices[l]]))
            zt = mp(float(om.z_factors[l])) * (1 + vl / ck) - 1
            b_f = bl / lam0 * mp(10) ** 13
            nu0 = cf / lam0
            Al, Bl = cf * (1 + zt) / b_f, nu0 / b_f
            al = mp(float(om.atomic_gamma[l])) / (4 * mpmath.pi * b_f)
            for q, p in enumerate(need):
                H[l, q], Hx[l, q], Ha[l, q], E[l, q] = _mp_terms(mpmath.mpc(Al / mp(float(wave[p])) - Bl, al))
            S[l] = float(N * mp(float(om.atomic_f[l])) * kon / (nu0 * bl))
            A[l], b[l], v[l] = float(Al), float(bl), float(vl)
    u = 1.0 / wave[need]
    F = np.exp(-np.sum(S[:, None] * H, axis=0))
    dtau = np.zeros((theta.size, n))
    np.add.at(dtau, om.N_indices, LN10 * S[:, None] * H)
    np.add.at(dtau, om.b_indices, -(S / b)[:, None] * E)
    np.add.at(dtau, om.v_indices, (S * A / (C_KMS + v))[:, None] * Hx * u[None, :])
    return ((-F * dtau)[:, pos] * k).sum(axis=2)


def wing_b_mask(om, theta, wave, px, d_min=64.0):
    """[len(theta), len(px)] True on the b column of component c at pixel p when every line of c has |z|^2 >= d_min
    and a <= 1 at every source pixel of p.  There E = (2a/sqrt(pi)) (-q_2 rho^2 + ...) has one sign for every line
    and every tap, so |J| itself is a scale with nothing cancelled, and a far-wing b derivative can be held to a
    bound relative to its own size rather than to Jhat (which carries H, ~x^2 times larger than E)."""
    theta = np.asarray(theta, dtype=np.float64)
    wave = np.asarray(wave, dtype=np.float64)
    src, _k = _stencil(om, wave.size, px)
    x, a = spu.line_x_a(om, theta, wave)
    wing = (x[:, src] ** 2 + (a ** 2)[:, None, None] >= d_min).all(axis=2) & (a <= 1.0)[:, None]   # [L, n]
    out = np.zeros((theta.size, len(px)), dtype=bool)
    for c in range(om.total_components):
        lines = np.flatnonzero(om.N_indices == c)
        out[om.b_indices[lines[0]]] = wing[lines].all(axis=0)
    return out


def hi_pair_at(a_target):
    """Two HI components over Lyman alpha-delta at z = 2.5 (the stream probes' Voigt-tier system) with the first
    line's damping a = ``a_target``, on 3000 px over +-300 Doppler widths of that line: (systems, theta rows, lb, ub,
    wave, b0).  a scales as 1 / b, so b0 = a(b = 1) / a_target."""
    from oracle import voigt_oracle as vo
    systems = [(2.5, "HI", [1215.67, 1025.72, 972.54, 949.74], 2)]
    cfg = vo.OracleConfig()
    cfg.add_system(*systems[0])
    lam = 1215.67 * 3.5
    _x, a = spu.line_x_a(vo.lower(cfg, FWHM=None), np.array([14.0, 13.5, 1.0, 25.0, 0.0, 40.0]), np.array([lam]))
    b0 = float(a[0] / a_target)
    th = np.array([14.0, 13.5, b0, 25.0, 0.0, 40.0])
    lb = np.array([12.0, 12.0, b0 * 0.5, 5.0, -50.0, -20.0])
    ub = np.array([16.0, 16.0, b0 * 2.0, 60.0, 50.0, 90.0])
    dw = lam * b0 / 299792.458
    thetas = np.array([th, th * [1, 1, 1.01, 1, 1, 1] + [0.3, 0, 0, 0, 0.2 * b0 / 30, 0]])
    return systems, thetas, lb, ub, np.linspace(lam - 300 * dw, lam + 300 * dw, 3000), b0


# ------------------------------------------------------------------------------------------------------ survey probe
def survey_from_fisher(v, g, F):
    """(M [..], J [.., ndim], F) from the survey probe's lnlike, gradient and Gauss-Newton matrix."""
    M = spu.flux_from_lnprob(v)
    return M, g / (2.0 - M)[..., None], F


def probe_survey(model, wave, thetas, px, lb, ub, max_bytes=2e9):
    """Survey probe through ``SightlineBatch.lnlike_and_fisher`` (the SL instantiations of every derivative
    kernel): (M [Ws, n], J [Ws, ndim, n], F [Ws, n, ndim, ndim]) at pixels ``px`` for theta rows ``thetas`` [Ws,
    ndim].  The launch covers every sightline and needs about 2 * 3C * P doubles per row, so the pixels go in groups
    of at most ``max_bytes`` of workspace."""
    from rbvfit_b200.likelihood import SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
    compiled = model.compile() if isinstance(model, GpuVoigtModel) else model
    thetas = np.atleast_2d(np.asarray(thetas, dtype=np.float64))
    Ws, nd = thetas.shape
    wave = np.asarray(wave, dtype=np.float64)
    px = np.asarray(px, dtype=np.int64)
    per_row = 8.0 * (2 * nd + 4) * (wave.size + 1024) * Ws        # ndim >= 3C columns of JF and JM, F, r, g
    step = max(1, int(max_bytes // per_row))
    M, J, Fm = np.empty((Ws, px.size)), np.empty((Ws, nd, px.size)), np.empty((Ws, px.size, nd, nd))
    for j0 in range(0, px.size, step):
        sel = px[j0:j0 + step]
        batch = SightlineBatch(spu.probe_sightlines(compiled, wave, sel), lb, ub)
        try:
            v, g, F = batch.lnlike_and_fisher(np.ascontiguousarray(np.broadcast_to(thetas, (sel.size, Ws, nd))))
        finally:
            batch.close()
        m, jj, ff = survey_from_fisher(v, g, F)                   # [n, Ws], [n, Ws, nd], [n, Ws, nd, nd]
        M[:, j0:j0 + step] = m.T
        J[:, :, j0:j0 + step] = np.transpose(jj, (1, 2, 0))
        Fm[:, j0:j0 + step] = np.swapaxes(ff, 0, 1)
    return M, J, Fm


def probe_fisher_numpy(om, thetas, wave, px):
    """The survey probe's (lnlike [n, Ws], gradient [n, Ws, ndim], Gauss-Newton matrix [n, Ws, ndim, ndim]) restated
    on the oracle (voigt_fisher_oracle.lnlike_fisher with weight 1 at p_j only): the CPU self-check of the
    recovery."""
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_oracle as vo
    thetas = np.atleast_2d(np.asarray(thetas, dtype=np.float64))
    wave = np.asarray(wave, dtype=np.float64)
    n, Ws, nd = len(px), thetas.shape[0], thetas.shape[1]
    v, g, F = np.empty((n, Ws)), np.empty((n, Ws, nd)), np.empty((n, Ws, nd, nd))
    for j, s in enumerate(spu.probe_sightlines(None, wave, px)):
        comp = vo.compile_instruments({"S": dict(model=om, wave=wave, flux=s["flux"], error=s["error"])})
        comp["S"]["inv_sigma2"] = np.where(s["weight_mask"], comp["S"]["inv_sigma2"], 0.0)
        comp["S"]["log_inv_sigma2"] = np.where(s["weight_mask"], comp["S"]["log_inv_sigma2"], 0.0)
        for r, th in enumerate(thetas):
            v[j, r], g[j, r], F[j, r] = vf.lnlike_fisher(comp, th)
    return v, g, F
