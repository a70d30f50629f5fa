"""CPU self-check of the derivative probes (tests/deriv_probe_util.py): the sparse Jacobian oracle equals the full one,
the oracle Jacobian agrees with a 60-digit mpmath evaluation at every Voigt tier switch and in the far wings, and the
survey probe's recovery identities hold on the oracle.  No GPU needed: a failure here is a bug of the harness or of the oracle, not
of a kernel."""
import numpy as np
import pytest

import deriv_probe_util as dpu
import stream_probe_util as spu
from deriv_probe_util import hi_pair_at
from test_gpu_stream_probes import _asym_taps

MPMATH_TOL = 2e-12      # oracle Jacobian against mpmath, in units of Jhat, beyond the x-conditioning allowance
MAXIMA = {}


@pytest.fixture(scope="module", autouse=True)
def _report_maxima():
    yield
    for key in sorted(MAXIMA):
        print(f"harness maximum {key}: {MAXIMA[key]:.3e}")


def _note(key, value):
    MAXIMA[key] = max(MAXIMA.get(key, 0.0), float(value))


def _oracle_model(systems, taps=None):
    from oracle import voigt_oracle as vo
    cfg = vo.OracleConfig()
    for (z, ion, trans, comps) in systems:
        cfg.add_system(z, ion, trans, comps)
    return vo.lower(cfg, FWHM=None, custom_taps=taps)


MGII = [(0.348, "MgII", [2796.3, 2803.5], 2)]
TH = np.array([[14.2, 14.5, 40.0, 30.0, -25.0, 35.0], [13.6, 12.9, 8.0, 55.0, 10.0, -40.0]])


@pytest.mark.parametrize("P", [5, 2050, 3000])
@pytest.mark.parametrize("K", [1, 7, 23, 65])
def test_sparse_jacobian_equals_full_oracle(K, P):
    from oracle import voigt_fisher_oracle as vf
    om = _oracle_model(MGII, None if K == 1 else _asym_taps(K))
    wave = np.linspace(3755.0, 3795.0, P)
    px = spu.probe_pixels(P, K, om, TH[0], wave, n_random=16, seed=K + P)
    for th in TH:
        th = np.concatenate([th, [0.3]])                                 # ndim > 3C: a zero row
        full = vf.model_jacobian(dict(model=om, wave=wave), th)[:, px]
        J, Jhat = dpu.oracle_jacobian_at(om, th, wave, px, with_scale=True)
        assert np.all(J[6:] == 0.0) and np.all(Jhat[6:] == 0.0)
        assert np.all(Jhat[:6] > 0.0)
        assert np.all(np.abs(J) <= Jhat * (1 + 1e-14))                   # the scale bounds what it scales
        d = np.max(np.abs(J - full)[:6] / Jhat[:6])
        _note("sparse vs full oracle Jacobian / Jhat", d)
        assert d <= (1e-15 if K <= 23 else 2e-15), d     # np.convolve adds the K products in another order


A_TIERS = [0.04, 0.06, 0.5, 0.99, 1.01, 2.0]


@pytest.mark.parametrize("a_target", A_TIERS)
def test_oracle_jacobian_vs_mpmath_at_tier_switches(a_target):
    """At the pixels nearest |z|^2 = 36, 64, 576 and 4e4 on both sides of every line and at every line centre:
    |J_oracle - J_mpmath| <= MPMATH_TOL Jhat + x_allowance."""
    systems, thetas, _lb, _ub, wave, _b0 = hi_pair_at(a_target)
    om = _oracle_model(systems)
    _x, a = spu.line_x_a(om, thetas[0], wave[:1])
    assert abs(a[0] / a_target - 1) < 1e-6
    px = spu.probe_pixels(wave.size, 1, om, thetas[0], wave, n_random=0, targets=(36.0, 64.0, 576.0, 4e4))
    for th in thetas:
        J, Jhat = dpu.oracle_jacobian_at(om, th, wave, px, with_scale=True)
        ref = dpu.mpmath_jacobian_at(om, th, wave, px)
        X = dpu.x_allowance(om, th, wave, px)
        err = np.abs(J - ref)
        bound = MPMATH_TOL * Jhat + X + np.finfo(float).tiny   # the floor: one rounding of a subnormal F
        assert np.all(err[Jhat == 0] == 0.0)                   # saturated pixels: F underflows in both, J = 0
        nz = Jhat > 0
        _note("oracle vs mpmath Jacobian / Jhat", np.max(err[nz] / Jhat[nz]))
        _note("oracle vs mpmath Jacobian / Jhat where the x allowance is below 1e-13 Jhat",
              np.max(np.where(X < 1e-13 * Jhat, err, 0.0)[nz] / Jhat[nz]))
        _note("oracle vs mpmath Jacobian / (MPMATH_TOL Jhat + x allowance)", np.max(err / bound))
        assert np.all(err <= bound), (a_target, np.max(err / bound))


def test_oracle_far_wing_b_column_vs_mpmath():
    """The b column far from every line, where E = H + x H_x + a H_a is ~x^-2 times smaller than H and Jhat: the
    oracle's differentiated series against mpmath relative to |J| itself (deriv_probe_util.wing_b_mask), |z|^2 from
    ~70 to ~3e6 -- the reference for the device's far tiers."""
    om = _oracle_model(MGII)
    th = TH[0].copy()
    th[2:4] = [5.0, 12.0]
    wave = np.linspace(3760.0, 4100.0, 2000)                 # from just redward of MgII 2803 (z = 0.348) outward
    px = np.arange(0, 2000, 50)
    mask = dpu.wing_b_mask(om, th, wave, px)
    assert mask[2].sum() >= 30 and mask[3].sum() >= 30
    J = dpu.oracle_jacobian_at(om, th, wave, px)
    ref = dpu.mpmath_jacobian_at(om, th, wave, px)
    d = np.max(np.abs(J - ref)[mask] / np.abs(ref[mask]))
    _note("oracle vs mpmath far-wing b column / |J|", d)
    # measured 2.1e-12: x carries eps c / b = 1.3e-11 at b = 5 km/s, and |d ln E / dx| ~ 4 / |x| <= 0.5 out here
    assert d <= 1e-11, d


def test_survey_probe_recovery_on_the_oracle():
    """v = -(2 - M)^2 / 2, g = (2 - M) J, F = J J^T of one unmasked pixel: the recovery returns the oracle's flux and
    Jacobian to <= 1e-15 (Jhat-relative for J)."""
    om = _oracle_model(MGII, _asym_taps(7))
    wave = np.linspace(3755.0, 3795.0, 300)
    px = np.array([0, 1, 3, 150, 151, 296, 299])
    v, g, F = dpu.probe_fisher_numpy(om, TH, wave, px)
    M, J, Fr = dpu.survey_from_fisher(v, g, F)                   # [n, Ws], [n, Ws, nd], [n, Ws, nd, nd]
    for r, th in enumerate(TH):
        assert np.max(np.abs(M[:, r] - spu.oracle_flux_at(om, th, wave, px))) <= 1e-15
        Jo, Jhat = dpu.oracle_jacobian_at(om, th, wave, px, with_scale=True)
        assert np.max(np.abs(J[:, r].T - Jo) / Jhat) <= 1e-15
        outer = np.einsum("in,jn->nij", Jo, Jo)
        sc = np.einsum("in,jn->nij", Jhat, Jhat)
        assert np.max(np.abs(Fr[:, r] - outer) / sc) <= 1e-15
