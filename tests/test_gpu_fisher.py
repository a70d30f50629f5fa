"""GPU: the model Jacobian and Gauss-Newton matrix (rbv_model_jacobian_batch, rbv_lnlike_fisher_batch) against the
Jacobian / Fisher oracle and the gradient path, special rows, determinism, and the device Levenberg-Marquardt fit
(fit_quick(method="lm")) against the same driver run on the oracle."""
import os
import sys

import numpy as np
import pytest

from golden_util import CASES, Golden

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_gradient import _in_bounds, _like  # noqa: E402
from test_gradient_oracle import piecewise_compiled  # noqa: E402

pytestmark = pytest.mark.gpu

JAC_TOL = 1e-8          # |device - oracle| <= JAC_TOL * max_p |oracle column|
FISHER_TOL = 1e-8       # |device - oracle| <= FISHER_TOL * sqrt(F_ii F_jj)
VALUE_RTOL = 1e-12
GRAD_TOL = 1e-10        # |fisher-path gradient - gradient path| <= GRAD_TOL * G_i


def _check(like, comp, thetas):
    """Every device output on these rows against the oracle and the gradient path; returns the worst errors."""
    from oracle import voigt_fisher_oracle as vf
    from oracle import voigt_grad_oracle as vg
    thetas = np.atleast_2d(thetas)
    v, g, F = like.lnlike_and_fisher(thetas)
    v_ref, g_ref = like.lnlike_and_grad(thetas)
    assert np.array_equal(v, v_ref)                                  # same forward kernels, same finalize
    worst = dict(jac=0.0, fisher=0.0, grad=0.0, value=0.0)
    for th, vi, gi, Fi, gri in zip(thetas, v, g, F, g_ref):
        assert np.array_equal(Fi, Fi.T)
        ev = np.linalg.eigvalsh(Fi)
        assert ev.min() >= -1e-12 * ev.max()
        ll, _g, F_or = vf.lnlike_fisher(comp, th)
        worst["value"] = max(worst["value"], abs(vi - ll) / abs(ll))
        d = np.sqrt(np.outer(np.diag(F_or), np.diag(F_or)))
        ok = d > 0
        assert np.all(Fi[~ok] == 0.0)
        worst["fisher"] = max(worst["fisher"], float(np.max(np.abs(Fi - F_or)[ok] / d[ok])))
        G = vg.grad_scale(comp, th)
        nz = G > 0
        assert np.all(gi[~nz] == 0.0)
        worst["grad"] = max(worst["grad"], float(np.max(np.abs(gi - gri)[nz] / G[nz])))
        for k, (name, dd) in enumerate(comp.items()):
            J = like.model_jacobian(th, k).T                                  # [ndim, P]
            J_or = vf.model_jacobian(dd, th)
            ncol = 3 * dd["model"].total_components
            assert np.all(J[ncol:] == 0.0)
            scale = np.max(np.abs(J_or[:ncol]), axis=1)
            worst["jac"] = max(worst["jac"], float(np.max(np.max(np.abs(J[:ncol] - J_or[:ncol]), axis=1) / scale)))
    return worst


def _assert_worst(worst, value_rtol=VALUE_RTOL):
    assert worst["jac"] <= JAC_TOL
    assert worst["fisher"] <= FISHER_TOL
    assert worst["grad"] <= GRAD_TOL
    assert worst["value"] <= value_rtol


@pytest.mark.parametrize("case", [c for c in CASES if c != "C1_fast"])
def test_fisher_vs_oracle_golden(case):
    g = Golden(case)
    rows = _in_bounds(g, g.flux_rows)
    if not rows:
        pytest.skip("no in-bounds fixture row")
    like = _like(g)
    worst = _check(like, g.oracle_compiled(), g.thetas[rows])
    print(case, worst)
    _assert_worst(worst)
    like.close()


def test_fisher_vs_oracle_c5a():
    g = Golden("C5a")
    rows = _in_bounds(g, range(len(g.thetas)))[:2]
    assert len(rows) == 2
    like = _like(g)
    worst = _check(like, g.oracle_compiled(), g.thetas[rows])
    print("C5a", worst)
    _assert_worst(worst)
    like.close()


def test_fisher_piecewise_lsf():
    from rbvfit_b200.likelihood import GpuLikelihood
    w, entries, comp, theta = piecewise_compiled()
    like = GpuLikelihood(entries, w["lb"], w["ub"])
    worst = _check(like, comp, theta)
    print("piecewise", worst)
    _assert_worst(worst)
    like.close()


def _c1_on_grid(P, K):
    """C1's lines on a P-pixel grid with a K-tap COS-like LSF: (GpuLikelihood, oracle instruments, theta)."""
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.likelihood import GpuLikelihood
    from rbvfit_b200.model import GpuVoigtModel
    w = wl.get_workload("C1")
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    for (z, ion, trans, comps) in w["systems"]:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        ocfg.add_system(z, ion, trans, comps)
    taps = vo.cos_like_lsf(K)
    wave = np.linspace(3770.0, 3780.0, P) if P > 1 else np.array([3774.6])
    om = vo.lower(ocfg, custom_taps=taps)
    rng = np.random.default_rng(P)
    flux = vo.model_flux(om, w["theta_true"], wave) + 0.02 * rng.standard_normal(P)
    err = np.full(P, 0.02)
    model = GpuVoigtModel(cfg, FWHM=None, lsf_taps=taps)
    like = GpuLikelihood({"COS": dict(model=model, wave=wave, flux=flux, error=err)}, w["lb"], w["ub"])
    comp = vo.compile_instruments({"COS": dict(model=om, wave=wave, flux=flux, error=err)})
    return like, comp, w["theta_true"] + np.array([0.05, -0.03, 2.0, -1.5, 3.0, -4.0])


@pytest.mark.parametrize("P,K", [(40, 321), (1000, 321), (3000, 61), (1, 5)])
def test_fisher_edge_geometry(P, K):
    like, comp, theta = _c1_on_grid(P, K)
    worst = _check(like, comp, theta)
    print(P, K, worst)
    # value against the oracle: measured 5.8e-12 at (1000, 321) and 1.3e-11 at (3000, 61) on a B200 -- the forward
    # model's own error, weighted by w = 1 / 0.02^2; _check has already found the value bit-identical to the gradient
    # path's
    _assert_worst(worst, value_rtol=3e-11)
    like.close()


def test_determinism_across_batch_order_and_chunks():
    from rbvfit_b200 import workloads as wl
    g = Golden("C1")
    like = _like(g)
    ens = wl.make_ensemble(wl.get_workload("C1"), 700)
    v1, g1, F1 = like.lnlike_and_fisher(ens)
    perm = np.random.default_rng(1).permutation(len(ens))
    v2, g2, F2 = like.lnlike_and_fisher(ens[perm])
    assert np.array_equal(v2, v1[perm]) and np.array_equal(g2, g1[perm]) and np.array_equal(F2, F1[perm])
    for i in (0, 3, 699):
        vi, gi, Fi = like.lnlike_and_fisher(ens[i])
        assert np.array_equal(np.array(vi), v1[i]) and np.array_equal(gi, g1[i]) and np.array_equal(Fi, F1[i])
    J1 = like.model_jacobian(ens, 0)
    like.engine.fisher_chunk_bytes = 1                                     # one row per launch
    v3, g3, F3 = like.lnlike_and_fisher(ens)
    assert np.array_equal(v3, v1) and np.array_equal(g3, g1) and np.array_equal(F3, F1)
    assert np.array_equal(like.model_jacobian(ens[:50], 0), J1[:50])
    like.close()


def test_special_rows():
    from rbvfit_b200._lib import RbvError
    from rbvfit_b200.engine import Engine
    from rbvfit_b200.likelihood import GpuLikelihood
    from test_gpu_parity import _gpu_models
    g = Golden("C1")
    like = _like(g)
    th = g.thetas[0].copy()
    C = len(th) // 3
    nan_row, bad_b, out = th.copy(), th.copy(), th.copy()
    nan_row[1] = np.nan
    bad_b[C] = -1.0
    out[0] = g.ub[0] + 1.0
    v, gr, F = like.lnlike_and_fisher(np.stack([nan_row, bad_b, out]))
    assert np.all(np.isnan(v[:2])) and np.all(np.isnan(gr[:2, :3 * C]).any(axis=1))
    assert np.all(np.isnan(F[:2, :3 * C, :3 * C]).any(axis=(1, 2)))
    assert np.isfinite(v[2]) and np.all(np.isfinite(gr[2])) and np.all(np.isfinite(F[2]))
    assert abs(v[2] - like.lnlike(out)) <= VALUE_RTOL * abs(v[2])          # no prior: evaluated like any row
    assert np.all(np.isnan(like.model_jacobian(bad_b, 0)[:, :3 * C]))
    # flux-only instrument: the Jacobian works, the Fisher call (it needs data) is refused
    eng = Engine()
    n = g.instruments[0]
    compiled = _gpu_models(g)[n].compile(verbose=False).data
    eng.add_instrument(compiled, g.inst(n, "wave"), taps=compiled.kernel, normalize_taps=compiled.kernel_normalize)
    eng.set_bounds(g.lb, g.ub)
    J = eng.model_jacobian(0, th[None, :])
    assert np.array_equal(J, like.engine.model_jacobian(0, th[None, :]))
    with pytest.raises(RbvError):
        eng.lnlike_fisher_host(th[None, :])
    eng.close()
    like.close()
    gf = Golden("C1_fast")
    models = _gpu_models(gf)
    nf = gf.instruments[0]
    fast = GpuLikelihood({nf: dict(model=models[nf], wave=gf.inst(nf, "wave"), flux=gf.inst(nf, "flux"),
                                   error=gf.inst(nf, "error"))}, gf.lb, gf.ub)
    with pytest.raises(RbvError):
        fast.lnlike_and_fisher(gf.thetas[0])
    with pytest.raises(RbvError):
        fast.model_jacobian(gf.thetas[0], 0)
    fast.close()


def _fitter(g):
    from test_gpu_parity import _gpu_models
    from rbvfit_b200.vfit_mcmc import vfit
    models = _gpu_models(g)
    inst = {n: dict(model=models[n], wave=g.inst(n, "wave"), flux=g.inst(n, "flux"), error=g.inst(n, "error"))
            for n in g.instruments}
    theta0 = np.clip(g.thetas[_in_bounds(g, range(len(g.thetas)))[0]], g.lb, g.ub)
    return vfit(inst, theta0, g.lb, g.ub, no_of_Chain=8, no_of_steps=2), theta0


@pytest.mark.parametrize("case", ["C1", "C2", "C3", "C4"])
def test_device_lm_vs_oracle_lm(case):
    from oracle import voigt_fisher_oracle as vf
    from rbvfit_b200.lm import levenberg_marquardt
    g = Golden(case)
    fitter, theta0 = _fitter(g)
    calls = []
    orig = fitter._like.lnlike_and_fisher

    def spy(theta):
        calls.append(np.atleast_2d(theta).shape[0])
        return orig(theta)

    n0 = fitter._like.engine.launch_count
    orig(theta0)
    per_call = fitter._like.engine.launch_count - n0
    fitter._like.lnlike_and_fisher = spy
    n0 = fitter._like.engine.launch_count
    best, err = fitter.fit_quick(verbose=False, method="lm")
    assert set(calls) == {1} and per_call in (6, 7)
    assert fitter._like.engine.launch_count - n0 == per_call * len(calls)   # one Fisher sequence per point
    fitter._like.lnlike_and_fisher = orig
    comp = g.oracle_compiled()
    ref = levenberg_marquardt(lambda x: vf.lnlike_fisher(comp, x), theta0, g.lb.astype(float), g.ub.astype(float))
    chi2_dev = fitter._chi2_batch(best)[0]
    chi2_ref = fitter._chi2_batch(ref.x)[0]
    cov, cref = fitter.theta_best_covariance, ref.cov
    d = np.sqrt(np.outer(np.diag(cref), np.diag(cref)))
    ok = np.isfinite(d)
    assert np.array_equal(ok, np.isfinite(cov))
    cov_err = float(np.max(np.abs(cov - cref)[ok] / d[ok]))
    assert np.array_equal(err[np.isfinite(err)], np.sqrt(np.diag(cov))[np.isfinite(err)])
    fitter2, _ = _fitter(g)
    _b, _e = fitter2.fit_quick(verbose=False, gradient="device")
    chi2_lbfgsb = fitter2._chi2_batch(_b)[0]
    print(case, "chi2 device LM", chi2_dev, "oracle LM", chi2_ref, "L-BFGS-B (device gradient)", chi2_lbfgsb,
          "| LM points", len(calls), "oracle LM points", ref.n_evals, "| max cov err", cov_err)
    assert abs(chi2_dev - chi2_ref) <= 1e-9 * chi2_ref
    assert cov_err <= 1e-6
    assert chi2_dev <= chi2_lbfgsb * (1 + 1e-9)
    np.testing.assert_array_equal(fitter.covariance(best), cov)


def test_lm_method_arguments():
    fitter, _ = _fitter(Golden("C1"))
    with pytest.raises(ValueError):
        fitter.fit_quick(verbose=False, method="lm", gradient="device")
    with pytest.raises(ValueError):
        fitter.fit_quick(verbose=False, method="newton")


def test_lm_coverage_c1():
    """64 noise realisations of C1 at theta_true, fitted with fit_quick(method="lm"): the mean Mahalanobis distance
    (theta_hat - theta_true)^T Cov^-1 (theta_hat - theta_true) is the chi^2_6 mean, 6, within 3.5 standard errors
    (sd of chi^2_6 is sqrt(12); / 8 for 64 fits).  The noise is workloads.SIGMA / 100: at SIGMA itself C1's two
    saturated, blended MgII components make the likelihood far from Gaussian (the fits are genuine minima tens of
    local sigmas from theta_true; DESIGN.md section 15), and no curvature-based covariance covers them."""
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    from rbvfit_b200.vfit_mcmc import vfit
    w = wl.get_workload("C1")
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    for (z, ion, trans, comps) in w["systems"]:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        ocfg.add_system(z, ion, trans, comps)
    (name, spec), = w["instruments"].items()
    wave, t = spec["wave"], w["theta_true"]
    clean = vo.model_flux(vo.lower(ocfg, FWHM=spec["FWHM"]), t, wave)
    sigma = wl.SIGMA / 100
    err = np.full(wave.size, sigma)
    rng = np.random.default_rng(20261)
    d2 = []
    for _ in range(64):
        flux = clean + sigma * rng.standard_normal(wave.size)
        model = GpuVoigtModel(cfg, FWHM=spec["FWHM"])
        fitter = vfit({name: dict(model=model, wave=wave, flux=flux, error=err)}, t, w["lb"], w["ub"],
                      no_of_Chain=8, no_of_steps=2)
        best, _e = fitter.fit_quick(verbose=False, method="lm")
        cov = fitter.theta_best_covariance
        assert np.all(np.isfinite(cov))
        dx = best - t
        d2.append(float(dx @ np.linalg.solve(cov, dx)))
        fitter._like.close()
    m = float(np.mean(d2))
    print("C1 coverage at SIGMA / 100: mean (theta_hat - theta_true)^T Cov^-1 (theta_hat - theta_true) =", m)
    assert 4.5 <= m <= 7.5
