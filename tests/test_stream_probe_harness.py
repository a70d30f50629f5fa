"""CPU self-check of the per-pixel probe (tests/stream_probe_util.py): the masks, data and flux recovery of the probe
return the oracle's model flux from a numpy lnlike to <= 1e-15, and the sparse oracle evaluation equals the full one.
No GPU needed: a failure here is a bug of the harness, not of a kernel."""
import numpy as np
import pytest

import stream_probe_util as spu


def _model(K, P, lo=3755.0, hi=3795.0):
    from oracle import voigt_oracle as vo
    cfg = vo.OracleConfig()
    cfg.add_system(0.348, "MgII", [2796.3, 2803.5], 2)
    if K == 1:
        om = vo.lower(cfg, FWHM=None)
    elif K == 23:
        om = vo.lower(cfg, FWHM="6.5")
    else:
        x = np.arange(-(K // 2), K // 2 + 1)
        taps = np.exp(-0.5 * (x / max(K / 6.0, 0.8)) ** 2) * (1 + 0.3 * (x > 0))
        om = vo.lower(cfg, FWHM=None, custom_taps=taps / taps.sum())
    assert spu.n_taps(om) == K
    return om, np.linspace(lo, hi, P)


TH = np.array([[14.2, 14.5, 40.0, 30.0, -25.0, 35.0], [13.6, 12.9, 8.0, 55.0, 10.0, -40.0]])


@pytest.mark.parametrize("K,P", [(1, 2100), (7, 3000), (23, 2050), (23, 5), (65, 2500), (41, 30)])
def test_probe_recovers_oracle_flux(K, P):
    from oracle import voigt_oracle as vo
    om, wave = _model(K, P)
    px = spu.probe_pixels(P, K, om, TH[0], wave, n_random=8, seed=K)
    full = np.array([vo.model_flux(om, th, wave)[px] for th in TH])
    sparse = np.array([spu.oracle_flux_at(om, th, wave, px) for th in TH])
    assert np.max(np.abs(sparse - full)) <= 1e-15
    lnp = spu.probe_lnprob_numpy(om, TH, wave, px)
    assert np.all(lnp <= -0.5) and np.all(lnp >= -2.0)
    assert np.max(np.abs(spu.flux_from_lnprob(lnp.T) - full)) <= 1e-15


def test_probe_pixel_selection():
    from oracle import voigt_oracle as vo
    K, P = 23, 5000
    om, wave = _model(K, P)
    px = spu.probe_pixels(P, K, om, TH[0], wave, n_random=0)
    assert np.array_equal(px, np.unique(px)) and px[0] == 0 and px[-1] == P - 1
    s = set(px.tolist())
    for m in (1024, 2048, 3072, 4096):
        assert set(range(m - K - 1, m + K + 2)) <= s
    assert set(range(K + 2)) <= s and set(range(P - K - 2, P)) <= s
    assert {255, 256, 257, 1791, 1792, 1793, 2047, 2048} <= s
    x, a = spu.line_x_a(om, TH[0], wave)
    # the line lowering is the oracle's: tau from x and a equals the oracle's tau
    from scipy.special import wofz
    N = 10 ** TH[0][om.N_indices]
    const = 4.48898479507e3 / (2.99792458e18 / om.atomic_lambda0 * TH[0][om.b_indices])
    tau = np.sum((N * om.atomic_f * const)[:, None] * wofz(x + 1j * a[:, None]).real, axis=0)
    assert np.allclose(tau, vo.model_flux(om, TH[0], wave, return_tau=True), rtol=1e-13, atol=0)
    for xl in x:
        assert int(np.argmin(np.abs(xl))) in s
    assert spu.boundary_windows(1024, K).size == 0
    bw = spu.boundary_windows(3000, 5)
    assert bw.tolist() == list(range(1024 - 7, 1024 + 7)) + list(range(2048 - 7, 2048 + 7))
