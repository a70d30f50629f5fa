"""Per-pixel probes of the derivative kernels (tests/deriv_probe_util.py) on the device: at every place the gradient
and Jacobian / Fisher kernels handle explicitly -- 256-pixel blocks, 1024-pixel tiles, 32-pixel Gram chunks, the
P == 1 adjoint, every LSF width up to 8193 taps and K > P, unsorted grids, the Voigt tiers along real spectra,
32-line chunks of the line passes, lines in component order across chunks, the 48 KB Gram shared-memory switch,
joint fits with unequal instruments and zero columns -- each case checks
  (a) GpuLikelihood.model_jacobian against the oracle at the probe pixels: |dJ_ip| <= JAC_TOL Jhat_ip + x allowance,
  (b) lnlike_and_grad against voigt_grad_oracle.lnlike_grad: |dg_i| <= GRAD_TOL Ghat_i (G_i without cancellation),
  (c) lnlike_and_fisher against voigt_fisher_oracle.lnlike_fisher: |dF_ij| <= FISHER_TOL sqrt(F_ii F_jj),
and the survey cases run the SL instantiations through single-pixel sightlines (deriv_probe_util.probe_survey).
Maxima per group are printed at the end of the module."""
import numpy as np
import pytest

import deriv_probe_util as dpu
import stream_probe_util as spu
from deriv_probe_util import hi_pair_at
from test_gpu_stream_probes import _asym_taps, _joint_instruments, _lya_forest, _mgii, _models, _rows

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
JAC_TOL = 1e-10         # Jacobian against the oracle, per pixel, in units of Jhat (beyond the x allowance)
GRAD_TOL = 1e-9         # gradient against the oracle, in units of Ghat_i (deriv_probe_util.grad_scale_nc)
WING_TOL = 1e-9         # far-wing b columns against the oracle, in units of |J| (deriv_probe_util.wing_b_mask)
FISHER_TOL = 1e-9       # Gauss-Newton matrix against the oracle, in units of sqrt(F_ii F_jj)
FLUX_TOL = 1e-10        # survey M (the derivative path's forward pass) against the oracle
TILE_TOL = 1e-11        # survey M against the tile kernel's flux mode
SL_ULPS = 8             # survey J (recovered) against the joint-path J: |dJ| <= SL_ULPS eps |J|
SUBNORMAL = 1e-290      # floor of (a): F = exp(-tau) is subnormal for tau > 708 and J = F dtau/dtheta with it
MAXIMA = {}


@pytest.fixture(scope="module", autouse=True)
def _report_maxima():
    yield
    for key in sorted(MAXIMA):
        print(f"derivative probe maximum {key}: {MAXIMA[key]:.3e}")


def _note(key, value):
    MAXIMA[key] = max(MAXIMA.get(key, 0.0), float(value))


def _ratio(err, scale):
    """max err / scale where scale > 0; where scale == 0, err must be 0 (returned as inf otherwise)."""
    pos = scale > 0
    if np.any(err[~pos] != 0):
        return np.inf
    return float(np.max(err[pos] / scale[pos])) if pos.any() else 0.0


def _data(model, om, wave, theta, seed, sigma=0.02):
    from oracle import voigt_oracle as vo
    rng = np.random.default_rng(seed)
    flux = vo.model_flux(om, theta, wave) + sigma * rng.standard_normal(wave.size)
    return dict(model=model, wave=wave, flux=flux, error=np.full(wave.size, sigma))


def _check_jacobian(group, like, k, om, wave, thetas, px):
    """(a) at pixels ``px`` of instrument k; returns the device Jacobian rows [n, ndim, len(px)].  The x allowance
    (deriv_probe_util.x_allowance) applies everywhere: in saturated pixels the oracle's flux factor, whose x comes
    from another lowering than its columns', moves by |dtau/dx| eps c / b relative, and tau_x reaches hundreds
    there."""
    Jd = np.swapaxes(like.model_jacobian(thetas, k), 1, 2)                # [n, ndim, P]
    ncol = 3 * om.total_components
    assert np.all(Jd[:, ncol:] == 0.0)
    out = Jd[:, :, px]
    for th, Jr in zip(thetas, out):
        J, Jhat = dpu.oracle_jacobian_at(om, th, wave, px, with_scale=True)
        X = dpu.x_allowance(om, th, wave, px)
        err = np.abs(Jr - J)
        _note(f"{group} Jacobian / Jhat", _ratio(err, Jhat))
        _note(f"{group} Jacobian: x allowance / (JAC_TOL Jhat)", _ratio(X, JAC_TOL * Jhat))
        r = _ratio(err, JAC_TOL * Jhat + X + SUBNORMAL)
        _note(f"{group} Jacobian / bound", r)
        assert r <= 1.0, (group, r)
        # far from every line of a component its b column is E-dominated, ~x^2 below Jhat: held to its own size
        wing = dpu.wing_b_mask(om, th, wave, px)
        if wing.any():
            rw = _ratio(err[wing], WING_TOL * np.abs(J[wing]) + X[wing] + SUBNORMAL)
            _note(f"{group} far-wing b column / bound", rw)
            _note(f"{group} far-wing b column / |J|", _ratio(err[wing], np.abs(J[wing])))
            assert rw <= 1.0, (group, "far-wing b", rw)
    return out


def _check_rows(group, like, comp, thetas, grad=True, fisher=True, row_allow=None):
    """(b) and (c) over the whole fit; ``row_allow(th) -> (gradient allowance [ndim], Fisher allowance [ndim,
    ndim])`` adds the x-conditioning of small-b cases."""
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_grad_oracle as vg
    if grad:
        _v, g = like.lnlike_and_grad(thetas)
    if fisher:
        _v2, _g2, F = like.lnlike_and_fisher(thetas)
    for r, th in enumerate(thetas):
        ag, aF = row_allow(th) if row_allow is not None else (0.0, 0.0)
        if grad:
            gr, G = vg.lnlike_grad(comp, th), vg.grad_scale(comp, th)
            Gh = sum(dpu.grad_scale_nc(dd, th) for dd in comp.values())
            err = np.abs(g[r] - gr)
            _note(f"{group} gradient / G", _ratio(err, G))
            _note(f"{group} gradient / Ghat", _ratio(err, Gh))
            rr = _ratio(err, GRAD_TOL * Gh + ag)
            _note(f"{group} gradient / bound", rr)
            assert rr <= 1.0, (group, rr)
        if fisher:
            _ll, _gf, Fo = vf.lnlike_fisher(comp, th)
            d = np.sqrt(np.outer(np.diag(Fo), np.diag(Fo)))
            err = np.abs(F[r] - Fo)
            _note(f"{group} Fisher / sqrt(FiiFjj)", _ratio(err, d))
            rr = _ratio(err, FISHER_TOL * d + aF)
            _note(f"{group} Fisher / bound", rr)
            assert rr <= 1.0, (group, rr)


def _row_allowance(om, d):
    """x-conditioning of (b) and (c) from the per-pixel allowance over the whole spectrum: sum_p |r_p| X_ip and
    sum_p w_p (|J_ip| X_jp + X_ip |J_jp|)."""
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_oracle as vo
    allpx = np.arange(d["wave"].size)

    def allow(th):
        X = dpu.x_allowance(om, th, d["wave"], allpx)
        J = np.abs(vf.model_jacobian(d, th))
        w = d["inv_sigma2"]
        r = np.abs(d["flux"] - vo.model_flux(om, th, d["wave"])) * w
        return X @ r, (J * w) @ X.T + (X * w) @ J.T
    return allow


def _check_survey(group, model, om, wave, thetas, lb, ub, px, J_joint, flux_tol=FLUX_TOL):
    """Survey probe: M against the oracle and the tile kernel's flux mode, the recovered J against the joint path's,
    F against J_i J_j."""
    M, J, F = dpu.probe_survey(model, wave, thetas, px, lb, ub)
    ref = np.array([spu.oracle_flux_at(om, th, wave, px) for th in thetas])
    d = np.max(np.abs(M - ref))
    _note(f"{group} survey M vs oracle", d)
    _note(f"{group} survey M vs oracle / bound", d / flux_tol)
    assert d <= flux_tol, (group, d)
    tile = model.compile().model_flux(thetas, wave)[:, px]
    d = np.max(np.abs(M - tile))
    _note(f"{group} survey M vs tile flux", d)
    assert d <= TILE_TOL, (group, d)
    err = np.abs(J - J_joint)
    r = _ratio(err, EPS * np.abs(J_joint))
    _note(f"{group} survey J vs joint J (ulps of |J|)", r)
    assert r <= SL_ULPS, (group, r)
    outer = np.einsum("wip,wjp->wpij", J_joint, J_joint)
    r = _ratio(np.abs(F - outer), EPS * np.abs(outer))
    _note(f"{group} survey F vs J_i J_j (ulps)", r)
    assert r <= 2, (group, r)


def _single(group, model, om, wave, thetas, lb, ub, px=None, grad=True, fisher=True, survey=False, xcond=False,
            flux_tol=FLUX_TOL, seed=0, jac=True):
    from oracle import voigt_oracle as vo
    from rbvfit_b200.likelihood import GpuLikelihood
    wave = np.asarray(wave, dtype=np.float64)
    thetas = np.atleast_2d(thetas)
    if px is None:
        px = spu.probe_pixels(wave.size, spu.n_taps(om), om, thetas[0], wave, n_random=16, seed=wave.size + seed)
    d = _data(model, om, wave, thetas[0], seed)
    like = GpuLikelihood({"S": d}, lb, ub)
    try:
        Jd = _check_jacobian(group, like, 0, om, wave, thetas, px) if jac else None
        comp = vo.compile_instruments({"S": dict(d, model=om)})
        allow = _row_allowance(om, comp["S"]) if xcond else None
        _check_rows(group, like, comp, thetas, grad=grad, fisher=fisher, row_allow=allow)
    finally:
        like.close()
    if survey:
        _check_survey(group, model, om, wave, thetas, lb, ub, px, Jd, flux_tol=flux_tol)


# --------------------------------------------------------------------------------- blocks, tiles and Gram chunks
@pytest.mark.parametrize("P", [1, 2, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 1055, 2049, 4100])
def test_block_tile_and_gram_chunk_edges(P):
    """256-pixel blocks, 1024-pixel tiles, 32-pixel Gram chunks (partial last chunk) and the P == 1 adjoint; MgII
    with 4 components, asymmetric 7-tap LSF, survey probe included."""
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems, FWHM=None, taps=_asym_taps(7))
    wave = np.linspace(3755.0, 3795.0, P) if P > 1 else np.array([3769.5])
    _single("edges", model, om, wave, _rows(th, lb, ub, 2, P), lb, ub, survey=True, seed=P)


# --------------------------------------------------------------------------------- LSF widths
@pytest.mark.parametrize("K", [1, 3, 7, 23, 25, 65, 321])
def test_lsf_widths(K):
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems, FWHM=None, taps=None if K == 1 else _asym_taps(K))
    _single("lsf", model, om, np.linspace(3740.0, 3810.0, 3000), _rows(th, lb, ub, 2, K), lb, ub, survey=True,
            seed=K)


def test_lsf_wider_than_the_spectrum():
    """K = 321 > P = 40: every output pixel clamps on both edges (cum_lo and cum_hi of the adjoint)."""
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems, FWHM=None, taps=_asym_taps(321))
    _single("lsf", model, om, np.linspace(3772.0, 3782.0, 40), _rows(th, lb, ub, 3, 321), lb, ub,
            px=np.arange(40), survey=True)


def test_lsf_of_8193_taps():
    """The widest LSF (K - 1 = 8192) on a 20 000-pixel spectrum; one theta row, probes thinned to keep oracle time
    down."""
    systems, th, lb, ub = _mgii(4)
    K = 8193
    model, om = _models(systems, FWHM=None, taps=_asym_taps(K))
    wave = np.linspace(3700.0, 3860.0, 20000)
    px = spu.probe_pixels(wave.size, K, om, th, wave, n_random=16, seed=8193)
    px = np.unique(np.concatenate([px[::64], px[:8], px[-8:]]))
    _single("lsf 8193", model, om, wave, th[None, :], lb, ub, px=px)


# --------------------------------------------------------------------------------- unsorted grids
@pytest.mark.parametrize("order", ["descending", "permuted"])
def test_unsorted_grids(order):
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems)
    wave = np.linspace(3740.0, 3810.0, 3000)
    wave = wave[::-1].copy() if order == "descending" else np.random.default_rng(3).permutation(wave)
    _single("grids", model, om, wave, _rows(th, lb, ub, 2, 6), lb, ub)


# --------------------------------------------------------------------------------- Voigt tiers
@pytest.mark.parametrize("a_target", [0.04, 0.06, 0.5, 0.99, 1.01, 2.0])
def test_voigt_tiers_on_real_spectra(a_target):
    """Damping a of the first line across kAFast = 0.05 (table / Weideman) and kABig = 1 (rho-series / complex
    asymptotic tier and weideman_grad in the core), on 3000 px over +-300 Doppler widths, probes at |z|^2 = 64, 576
    and 4e4.  Such a needs b <= 0.15 km/s: every bound adds the x allowance (deriv_probe_util)."""
    systems, thetas, lb, ub, wave, b0 = hi_pair_at(a_target)
    model, om = _models(systems)
    _single("voigt tiers", model, om, wave, thetas, lb, ub, survey=True, xcond=True,
            flux_tol=FLUX_TOL + 8 * EPS * 299792.458 / (0.5 * b0))


def test_dla_next_to_weak_lines():
    """A damped Lyman alpha line (saturated pixels: F underflows, J = 0 there) with weak CIV in its wings."""
    systems = [(2.5, "HI", [1215.67], 1), (1.748, "CIV", [1548.2, 1550.77], 3)]
    model, om = _models(systems)
    th = np.array([21.0, 12.8, 13.0, 12.6, 20.0, 15.0, 30.0, 10.0, 0.0, -60.0, 20.0, 80.0])
    thetas = np.array([th, th + np.array([-0.5] + [0.2] * 11)])
    wave = np.linspace(4200.0, 4310.0, 6000)
    _single("dla", model, om, wave, thetas, th - 3.0, th + 3.0, survey=True)
    from oracle import voigt_oracle as vo
    assert np.any(vo.model_flux(om, th, wave, convolve=False) == 0.0)      # the saturated pixels exist


# --------------------------------------------------------------------------------- line and component counts
@pytest.mark.parametrize("L", [31, 32, 33, 64, 65, 127, 128, 129, 300])
def test_line_counts(L):
    """32-line chunks of grad_line_kernel / fisher_col_kernel and 128-line blocks of grad_prep_kernel (Lyman alpha
    forest: L lines, L components)."""
    systems, th, lb, ub = _lya_forest(L)
    model, om = _models(systems)
    thetas = _rows(th, lb, ub, 2 if L < 300 else 1, L,
                   scale=np.concatenate([np.full(L, 0.02), np.full(L, 0.5), np.full(L, 1.0)]))
    wave = np.linspace(3400.0, 6100.0, 9000 if L < 128 else 4000)
    # L = 300 components is past the Jacobian / Fisher path's component limit: the gradient alone.  The damped lines
    # (logN 19) saturate cores whose Jacobian carries an x allowance up to 19 JAC_TOL Jhat; the gradient there differs
    # from the oracle by up to 1.4e-9 G_i, identically through the adjoint and the Fisher path (to 1e-15), so the
    # rows take the x allowance too
    _single("lines", model, om, wave, thetas, lb, ub, fisher=L <= 129, jac=L <= 129, xcond=L <= 129)


def _tied(C=8):
    """One HI system of C components over five Lyman lines: the lowering is transition-major, so component c's lines
    are c, c + C, ... and order[] runs them across 32-line chunks."""
    systems = [(2.5, "HI", [1215.67, 1025.72, 972.54, 949.74, 937.80], C)]
    rng = np.random.default_rng(C)
    th = np.concatenate([rng.uniform(13.0, 15.0, C), rng.uniform(1.5, 4.0, C), np.linspace(-150.0, 150.0, C)])
    return systems, th, th - np.r_[np.full(C, 1.0), np.full(C, 1.0), np.full(C, 20.0)], \
        th + np.r_[np.full(C, 1.0), np.full(C, 10.0), np.full(C, 20.0)]


def test_tied_transitions_straddle_line_chunks():
    """b = 1.5-4 km/s: the series coefficients q_p(a^2) of the wing tiers differ between lines by a^2 ~ 1e-5, enough
    for a coefficient taken from the wrong line of a chunk to show (at b ~ 25 km/s a^2 ~ 1e-7 and it hides below
    the bounds)."""
    systems, th, lb, ub = _tied(8)
    model, om = _models(systems)
    assert om.n_lines == 40
    _single("tied", model, om, np.linspace(3250.0, 4300.0, 6000), _rows(th, lb, ub, 2, 8), lb, ub, survey=True)


def test_c2_components_out_of_line_order():
    """C2's systems (12 components, 33 lines, several ions and transitions per system) on a 6000-pixel grid."""
    from rbvfit_b200 import workloads as wl
    w = wl.get_workload("C2")
    model, om = _models(w["systems"])
    assert om.n_lines > 32 and np.any(np.diff(om.N_indices) < 0)
    _single("tied", model, om, np.linspace(3300.0, 5700.0, 6000), _rows(w["theta_true"], w["lb"], w["ub"], 2, 2),
            w["lb"], w["ub"])


@pytest.mark.parametrize("C", [63, 64, 100])
def test_gram_shared_memory_threshold(C):
    """(3C + 2) 32 8 B crosses 48 KB between C = 63 and C = 64: the Gram kernel's opt-in dynamic shared memory; the
    Jacobian and (c) on a short spectrum."""
    systems, th, lb, ub = _mgii(C)
    model, om = _models(systems)
    _single("gram smem", model, om, np.linspace(3755.0, 3795.0, 300), _rows(th, lb, ub, 1, C), lb, ub, grad=False)


# --------------------------------------------------------------------------------- joint fits
def _joint_check(group, inst, thetas, lb, ub, masks=None):
    """(a) per instrument, (b) and (c) over the joint fit.  ``inst``: {name: (model, om, wave)}."""
    from oracle import voigt_oracle as vo
    from rbvfit_b200.likelihood import GpuLikelihood
    data = {}
    for j, (name, (model, om, wave)) in enumerate(inst.items()):
        data[name] = _data(model, om, wave, thetas[0], 100 + j)
        if masks is not None:
            data[name]["weight_mask"] = masks[name]
    like = GpuLikelihood(data, lb, ub)
    try:
        for k, (name, (model, om, wave)) in enumerate(inst.items()):
            px = spu.probe_pixels(wave.size, spu.n_taps(om), om, thetas[0], wave, n_random=8, seed=k)
            _check_jacobian(group, like, k, om, wave, thetas, px)
        comp = vo.compile_instruments({n: dict(data[n], model=inst[n][1]) for n in inst})
        for n in inst:
            if masks is not None:
                comp[n]["inv_sigma2"] = np.where(masks[n], comp[n]["inv_sigma2"], 0.0)
                comp[n]["log_inv_sigma2"] = np.where(masks[n], comp[n]["log_inv_sigma2"], 0.0)
        _check_rows(group, like, comp, thetas)
    finally:
        like.close()


def test_joint_instruments_with_different_L_P_K():
    inst, th, lb, ub = _joint_instruments()
    _joint_check("joint", inst, _rows(th, lb, ub, 2, 91), lb, ub)


def test_joint_instrument_with_fewer_components():
    """Instrument D models only the first two of the four HI components: its columns 6..11 of the Jacobian are
    zero, and it reads theta with its own layout (logN 0-1, b 2-3, v 4-5) as the oracle lowers it."""
    inst, th, lb, ub = _joint_instruments()
    model, om = _models([(z, "HI", [1215.67, 1025.72], 1) for z in (2.30, 2.45)], taps=_asym_taps(9))
    inst["D"] = (model, om, np.linspace(3350.0, 4050.0, 2500))
    assert om.total_components == 2
    _joint_check("joint fewer components", inst, _rows(th, lb, ub, 2, 92), lb, ub)


def test_joint_sixteen_instruments():
    """The 16-instrument maximum: P from 300 to 2550 px, K cycling through 1, 3, 7, 23 and 65."""
    zs = [2.30, 2.45, 2.60, 2.75]
    lyman = [1215.67, 1025.72, 972.54]
    inst = {}
    Ks = [1, 3, 7, 23, 65]
    for i in range(16):
        K = Ks[i % 5]
        model, om = _models([(z, "HI", lyman[:1 + i % 3], 1) for z in zs], FWHM=None,
                            taps=None if K == 1 else _asym_taps(K))
        inst[f"I{i}"] = (model, om, np.linspace(3300.0 + 40 * i, 4500.0 - 20 * i, 300 + 150 * i))
    _i, th, lb, ub = _joint_instruments()
    _joint_check("joint 16", inst, _rows(th, lb, ub, 2, 93), lb, ub)


def test_joint_ndim_beyond_3C():
    """ndim > 3C: the extra theta entries have zero Jacobian rows, gradient entries and Fisher rows / columns."""
    inst, th, lb, ub = _joint_instruments()
    extra = np.array([0.7, -1.3])
    thx, lbx, ubx = np.r_[th, extra], np.r_[lb, extra - 5], np.r_[ub, extra + 5]
    rows = np.hstack([_rows(th, lb, ub, 2, 94), np.tile(extra, (2, 1))])
    _joint_check("joint ndim > 3C", inst, rows, lbx, ubx)
    from rbvfit_b200.likelihood import GpuLikelihood
    data = {n: _data(m, om, w, thx, 7) for n, (m, om, w) in inst.items()}
    like = GpuLikelihood(data, lbx, ubx)
    try:
        _v, g, F = like.lnlike_and_fisher(rows)
        _v, g2 = like.lnlike_and_grad(rows)
    finally:
        like.close()
    assert np.all(g[:, 12:] == 0.0) and np.all(g2[:, 12:] == 0.0)
    assert np.all(F[:, 12:, :] == 0.0) and np.all(F[:, :, 12:] == 0.0)


def test_piecewise_lsf_weight_mask():
    """The piecewise-LSF problem (one instrument per LSF block, each with a weight_mask): the Jacobian of every
    instrument at its probes, (b) and (c) with the masks."""
    from test_gradient_oracle import piecewise_compiled
    from rbvfit_b200.likelihood import GpuLikelihood
    w, entries, comp, theta = piecewise_compiled()
    like = GpuLikelihood(entries, w["lb"], w["ub"])
    thetas = np.array([theta, theta + np.r_[0.02, -0.02, 0.5, -0.5, 1.0, -1.0]])
    try:
        for k, (n, d) in enumerate(comp.items()):
            om, wave = d["model"], d["wave"]
            px = spu.probe_pixels(wave.size, spu.n_taps(om), om, theta, wave, n_random=8, seed=k)
            _check_jacobian("piecewise", like, k, om, wave, thetas, px)
        _check_rows("piecewise", like, comp, thetas)
    finally:
        like.close()
