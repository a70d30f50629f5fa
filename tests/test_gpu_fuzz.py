"""GPU parity on randomly drawn problems (fixed seeds): random systems / ions / component counts, redshifts,
wavelength windows and pixel counts, LSFs, column densities up to the damped regime, Doppler widths from 3 to 80 km/s
-- lnprob and model flux against the CPU oracle at the north-star tolerances."""
import numpy as np
import pytest

from fuzz_util import draw_problem as _draw

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", range(24))
def test_random_problem_matches_oracle(seed):
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration
    from rbvfit_b200.likelihood import GpuLikelihood
    from rbvfit_b200.model import GpuVoigtModel
    systems, wave, fwhm, taps, theta, thetas, lb, ub, rng = _draw(1000 + seed)
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    for (z, ion, trans, comps) in systems:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        ocfg.add_system(z, ion, trans, comps)
    model = GpuVoigtModel(cfg, FWHM=fwhm, lsf_taps=taps)
    om = vo.lower(ocfg, FWHM=fwhm, custom_taps=taps)
    truth = vo.model_flux(om, theta, wave)
    flux = truth + 0.03 * rng.standard_normal(wave.size)
    error = np.full(wave.size, 0.03)
    like = GpuLikelihood({"S": dict(model=model, wave=wave, flux=flux, error=error)}, lb, ub)
    comp = vo.compile_instruments({"S": dict(model=om, wave=wave, flux=flux, error=error)})
    got, ref = like.lnprob(thetas), vo.lnprob_batch(comp, thetas, lb, ub)
    assert np.array_equal(np.isneginf(got), np.isneginf(ref)) and np.isneginf(ref).sum() >= 1
    fin = np.isfinite(ref)
    assert np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin])) <= 1e-9
    gf = model.compile().model_flux(thetas[:3], wave)
    rf = np.array([vo.model_flux(om, t, wave) for t in thetas[:3]])
    assert np.max(np.abs(gf - rf)) <= 1e-10
    like.close()


@pytest.mark.parametrize("seed", range(24))
def test_random_problem_derivatives_match_oracle(seed):
    """The same problems through the derivative kernels: the Jacobian at stream_probe_util.probe_pixels per pixel,
    the gradient and the Gauss-Newton matrix per row (tests/test_gpu_deriv_probes.py's bounds).  Row 4 lies outside
    the box; the derivative calls take no prior, so it is evaluated like any row."""
    import stream_probe_util as spu
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration
    from rbvfit_b200.likelihood import GpuLikelihood
    from rbvfit_b200.model import GpuVoigtModel
    from test_gpu_deriv_probes import _check_jacobian, _check_rows, _row_allowance
    systems, wave, fwhm, taps, theta, thetas, lb, ub, rng = _draw(1000 + seed)
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    for (z, ion, trans, comps) in systems:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        ocfg.add_system(z, ion, trans, comps)
    model = GpuVoigtModel(cfg, FWHM=fwhm, lsf_taps=taps)
    om = vo.lower(ocfg, FWHM=fwhm, custom_taps=taps)
    flux = vo.model_flux(om, theta, wave) + 0.03 * rng.standard_normal(wave.size)
    error = np.full(wave.size, 0.03)
    rows = thetas[[0, 1, 4]]
    like = GpuLikelihood({"S": dict(model=model, wave=wave, flux=flux, error=error)}, lb, ub)
    try:
        px = spu.probe_pixels(wave.size, spu.n_taps(om), om, rows[0], wave, n_random=16, seed=seed)
        _check_jacobian("fuzz", like, 0, om, wave, rows, px)
        comp = vo.compile_instruments({"S": dict(model=om, wave=wave, flux=flux, error=error)})
        # b down to 3 km/s and damped HI: the x-conditioning allowance of the rows applies (tests/deriv_probe_util.py)
        _check_rows("fuzz", like, comp, rows, row_allow=_row_allowance(om, comp["S"]))
    finally:
        like.close()
