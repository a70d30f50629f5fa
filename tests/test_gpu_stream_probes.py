"""Per-pixel probes of the lnprob kernels (tests/stream_probe_util.py): the streaming kernel's model flux, recovered
pixel by pixel from sightline-mode lnprob launches, against the CPU oracle (|dM| <= 1e-10, the flux contract) and
against the tile kernel's flux mode (<= 1e-11), at range boundaries, short last ranges, row starts, every LSF width
the kernel takes, both boundary-record modes, the far-field remainder, the Voigt tiers, the exp switch and unsorted
grids; the tile kernel's chi^2 path gets the same probes with RBVFIT_B200_STREAM=0.  Every case asserts which kernel
ran.  Also here: joint fits, batch invariants and the samplers, all on the streaming kernel."""
import numpy as np
import pytest

import stream_probe_util as spu

pytestmark = pytest.mark.gpu

FLUX_TOL = 1e-10        # model flux against the oracle
TILE_TOL = 1e-11        # streaming kernel's chi^2 flux against the tile kernel's flux mode
KERNEL_ENV = {"stream": "1", "tile": "0"}
MAXIMA = {}             # largest |dM| per (group, kernel, reference), printed at the end of the module


@pytest.fixture(scope="module", autouse=True)
def _report_maxima():
    yield
    for key in sorted(MAXIMA):
        print(f"probe maximum {key}: {MAXIMA[key]:.3e}")


def _note(key, value):
    MAXIMA[key] = max(MAXIMA.get(key, 0.0), float(value))


def _models(systems, FWHM="6.5", taps=None, voigt_method="wofz"):
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration
    from rbvfit_b200.model import GpuVoigtModel
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    for (z, ion, trans, comps) in systems:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        ocfg.add_system(z, ion, trans, comps)
    return (GpuVoigtModel(cfg, FWHM=FWHM, lsf_taps=taps, voigt_method=voigt_method),
            vo.lower(ocfg, FWHM=FWHM, custom_taps=taps, voigt_method=voigt_method))


def _asym_taps(K):
    """Asymmetric LSF (fuzz_util.draw_problem's custom kernel): a tap-order bug cannot hide behind symmetry."""
    x = np.arange(-(K // 2), K // 2 + 1)
    taps = np.exp(-0.5 * (x / max(K / 5.0, 0.8)) ** 2) * (1 + 0.3 * (x > 0))
    return taps / taps.sum()


def _mgii(C):
    """MgII doublet with C components (L = 2 C) at z = 0.348 and a theta box around a blended profile."""
    rng = np.random.default_rng(C)
    th = np.concatenate([rng.uniform(13.0, 14.2, C), rng.uniform(12.0, 45.0, C), np.linspace(-60.0, 60.0, C)])
    lb = th - np.concatenate([np.full(C, 2.0), np.full(C, 10.0), np.full(C, 50.0)])
    ub = th + np.concatenate([np.full(C, 2.0), np.full(C, 40.0), np.full(C, 50.0)])
    return [(0.348, "MgII", [2796.3, 2803.5], C)], th, lb, ub


def _rows(th, lb, ub, n, seed, scale=None):
    C = th.size // 3
    if scale is None:
        scale = np.concatenate([np.full(C, 0.05), np.full(C, 1.0), np.full(C, 2.0)])
    rng = np.random.default_rng(seed)
    return np.clip(th + scale * rng.standard_normal((n, th.size)), lb, ub)


def _probe(monkeypatch, group, kernel, model, om, wave, thetas, lb, ub, segs=None, px=None, far_field=None,
           oracle_tol=FLUX_TOL):
    """Probe ``px`` (default: spu.probe_pixels) for every row of ``thetas`` through ``kernel``; assert the kernel
    and both bounds."""
    monkeypatch.setenv("RBVFIT_B200_STREAM", KERNEL_ENV[kernel])
    if segs is None:
        monkeypatch.delenv("RBVFIT_B200_STREAM_SEGS", raising=False)
    else:
        monkeypatch.setenv("RBVFIT_B200_STREAM_SEGS", str(segs))
    wave = np.asarray(wave, dtype=np.float64)
    P, K = wave.size, spu.n_taps(om)
    if px is None:
        px = spu.probe_pixels(P, K, om, thetas[0], wave, seed=P + K)
    got, ran = spu.probe_model_flux(model, wave, thetas, px, lb, ub, far_field=far_field)
    assert ran == kernel
    ref = np.array([spu.oracle_flux_at(om, th, wave, px) for th in thetas])
    d_oracle = np.max(np.abs(got - ref))
    tile = model.compile().model_flux(thetas, wave)[:, px]
    d_tile = np.max(np.abs(got - tile))
    _note(f"{group} {kernel} vs oracle", d_oracle)
    _note(f"{group} {kernel} vs tile flux", d_tile)
    bad = np.unravel_index(np.argmax(np.abs(got - ref)), got.shape)
    assert d_oracle <= oracle_tol, (d_oracle, int(px[bad[1]]), bad[0])
    assert d_tile <= TILE_TOL, d_tile
    return got, px


# --------------------------------------------------------------------------------- ragged ends and short last ranges
RAGGED = [0, 1, 5, 11, 12, 21, 22, 23, 255, 256, 257]


@pytest.mark.parametrize("kernel,n", [("stream", 2), ("stream", 3), ("stream", 4), ("tile", 2)])
@pytest.mark.parametrize("C", [4, 2])          # L = 8 (boundary records on) and L = 4 (records off)
def test_ragged_ends_and_short_last_ranges(monkeypatch, kernel, n, C):
    systems, th, lb, ub = _mgii(C)
    model, om = _models(systems)
    for extra in RAGGED:
        P = 1024 * n + extra
        _probe(monkeypatch, "ragged", kernel, model, om, np.linspace(3755.0, 3795.0, P), _rows(th, lb, ub, 3, P),
               lb, ub, segs=1)


@pytest.mark.parametrize("kernel", ["stream", "tile"])
@pytest.mark.parametrize("P", [1, 7, 22, 23, 300])
def test_single_range_spectra(monkeypatch, kernel, P):
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems)
    wave = np.linspace(3762.0, 3786.0, P) if P > 1 else np.array([3769.5])
    _probe(monkeypatch, "ragged", kernel, model, om, wave, _rows(th, lb, ub, 3, P), lb, ub, segs=1)


# --------------------------------------------------------------------------------- LSF widths
LSF_K = [1, 3, 7, 9, 15, 17, 23, 25, 41, 63, 65]


@pytest.mark.parametrize("kernel,segs", [("stream", 1), ("stream", 3), ("tile", None)])
@pytest.mark.parametrize("K", LSF_K)
def test_lsf_widths(monkeypatch, kernel, segs, K):
    """K = 1 (no LSF), the fully unrolled 1-3 tap blocks (K <= 24) and the looped ones (K > 24, NB = 0), up to the
    widest LSF the streaming kernel takes (K - 1 = 64), asymmetric taps."""
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems, FWHM=None, taps=None if K == 1 else _asym_taps(K))
    _probe(monkeypatch, "lsf", kernel, model, om, np.linspace(3740.0, 3810.0, 7000), _rows(th, lb, ub, 3, K), lb, ub,
           segs=segs)


def test_lsf_too_wide_for_the_streaming_kernel_takes_the_tile_kernel(monkeypatch):
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems, FWHM=None, taps=_asym_taps(67))
    wave = np.linspace(3740.0, 3810.0, 3000)
    px = spu.probe_pixels(wave.size, 67, n_random=8)[::4]
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    got, ran = spu.probe_model_flux(model, wave, _rows(th, lb, ub, 2, 67), px, lb, ub)
    assert ran == "tile"
    ref = np.array([spu.oracle_flux_at(om, t, wave, px) for t in _rows(th, lb, ub, 2, 67)])
    assert np.max(np.abs(got - ref)) <= FLUX_TOL


# --------------------------------------------------------------------------------- schedules
@pytest.fixture(scope="module")
def long_problem():
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems)
    wave = np.linspace(3700.0, 3860.0, 40000)
    thetas = _rows(th, lb, ub, 3, 40)
    px = spu.probe_pixels(wave.size, 23, om, thetas[0], wave, n_random=16, seed=40)
    return model, om, wave, thetas, lb, ub, px


@pytest.mark.parametrize("segs", [None, 1, 2, 7])
def test_schedules_on_a_long_spectrum(monkeypatch, long_problem, segs):
    """40 000 px: the default schedule (ranges of a third of what is left) and uniform ranges of 1, 2 and 7
    segments.  The probes see every multiple of 1024, so every boundary of every schedule."""
    model, om, wave, thetas, lb, ub, px = long_problem
    _probe(monkeypatch, "schedule", "stream", model, om, wave, thetas, lb, ub, segs=segs, px=px)


def test_schedules_agree_on_lnprob(monkeypatch, long_problem):
    from rbvfit_b200.likelihood import GpuLikelihood
    model, om, wave, thetas, lb, ub, _px = long_problem
    rng = np.random.default_rng(41)
    flux = model.compile().model_flux(thetas[0], wave) + 0.05 * rng.standard_normal(wave.size)
    rows = _rows(thetas[0], lb, ub, 6, 42)
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    out = {}
    for segs in (None, 1, 2, 7):
        if segs is None:
            monkeypatch.delenv("RBVFIT_B200_STREAM_SEGS", raising=False)
        else:
            monkeypatch.setenv("RBVFIT_B200_STREAM_SEGS", str(segs))
        like = GpuLikelihood({"S": dict(model=model, wave=wave, flux=flux, error=np.full(wave.size, 0.05))}, lb, ub)
        out[segs] = like.lnprob(rows)
        assert like.engine.last_kernel == "stream"
        like.close()
    for segs in (1, 2, 7):
        rel = np.max(np.abs(out[segs] - out[None]) / np.abs(out[None]))
        _note("schedule lnprob rel. spread", rel)
        assert rel <= 1e-13, (segs, rel)


# --------------------------------------------------------------------------------- line count and far field
def _lya_forest(L):
    """L single-line HI systems over 3400-6100 A (L lines, L components), every seventh one damped."""
    zs = np.linspace(1.85, 3.95, L) if L > 1 else np.array([2.5])
    systems = [(float(z), "HI", [1215.67], 1) for z in zs]
    rng = np.random.default_rng(L)
    N = rng.uniform(12.5, 14.5, L)
    N[::7] = 19.0
    th = np.concatenate([N, rng.uniform(10.0, 40.0, L), rng.uniform(-50.0, 50.0, L)])
    lb = th - np.concatenate([np.full(L, 1.0), np.full(L, 8.0), np.full(L, 20.0)])
    ub = th + np.concatenate([np.full(L, 1.0), np.full(L, 20.0), np.full(L, 20.0)])
    return systems, th, lb, ub


@pytest.mark.parametrize("far_field", ["chebyshev", "direct"])
@pytest.mark.parametrize("L", [1, 7, 8, 32, 33, 40, 96])
def test_line_count_and_far_field(monkeypatch, L, far_field):
    """The boundary-record switch at L = 8 and the far-field (line, node) remainder above 32 lines."""
    systems, th, lb, ub = _lya_forest(L)
    model, om = _models(systems)
    assert om.n_lines == L
    thetas = _rows(th, lb, ub, 2, L, scale=np.concatenate([np.full(L, 0.02), np.full(L, 0.5), np.full(L, 1.0)]))
    _probe(monkeypatch, "lines", "stream", model, om, np.linspace(3400.0, 6100.0, 9000), thetas, lb, ub, segs=1,
           far_field=far_field)


# --------------------------------------------------------------------------------- Voigt tiers and the exp switch
def _hi_pair(b0):
    """HI Lyman alpha-delta at z = 2.5, two components: the first with Doppler parameter ``b0``."""
    systems = [(2.5, "HI", [1215.67, 1025.72, 972.54, 949.74], 2)]
    th = np.array([14.0, 13.5, b0, 25.0, 0.0, 40.0])
    lb = np.array([12.0, 12.0, b0 * 0.5, 5.0, -50.0, -20.0])
    ub = np.array([16.0, 16.0, b0 * 2.0, 60.0, 50.0, 90.0])
    return systems, th, lb, ub


@pytest.mark.parametrize("kernel", ["stream", "tile"])
@pytest.mark.parametrize("a_target", [0.08, 0.5, 2.0])
def test_voigt_tiers_small_b(monkeypatch, kernel, a_target):
    """Damping parameter a > 0.05 (small b) up to a >= 1 (the general algorithm), on a grid fine enough to resolve
    the line core: 3000 px over +-300 Doppler widths of the first component's Lyman alpha line.  x = (nu - nu0) / b_nu
    is a difference of two numbers c / b times larger than x's unit, so any two evaluations of it (oracle, kernel)
    differ by a few eps c / b: the oracle bound widens by 8 eps c / b (|dM/dx| <= 1); the two kernels share that
    arithmetic and are held to 1e-11."""
    systems, th, lb, ub = _hi_pair(1.0)
    model, om = _models(systems)
    lam = 1215.67 * 3.5
    x, a = spu.line_x_a(om, th, np.array([lam]))
    b0 = float(a[0] / a_target)                      # a scales as 1 / b
    systems, th, lb, ub = _hi_pair(b0)
    model, om = _models(systems)
    x, a = spu.line_x_a(om, th, np.array([lam]))
    assert abs(a[0] / a_target - 1) < 1e-6
    dw = lam * b0 / 299792.458
    thetas = np.array([th, th * [1, 1, 1.01, 1, 1, 1] + [0.3, 0, 0, 0, 0.2 * b0 / 30, 0]])
    _probe(monkeypatch, "voigt tiers", kernel, model, om, np.linspace(lam - 300 * dw, lam + 300 * dw, 3000), thetas,
           lb, ub, segs=1, oracle_tol=FLUX_TOL + 8 * np.finfo(float).eps * 299792.458 / (0.5 * b0))


@pytest.mark.parametrize("kernel", ["stream", "tile"])
def test_dla_next_to_weak_lines(monkeypatch, kernel):
    """A damped Lyman alpha line (saturated rows: flux underflows to 0) with weak CIV lines in its wings."""
    systems = [(2.5, "HI", [1215.67], 1), (1.748, "CIV", [1548.2, 1550.77], 3)]
    model, om = _models(systems)
    th = np.array([21.0, 12.8, 13.0, 12.6, 20.0, 15.0, 30.0, 10.0, 0.0, -60.0, 20.0, 80.0])
    lb, ub = th - 3.0, th + 3.0
    thetas = np.array([th, th + np.array([-0.5] + [0.2] * 11), th + np.array([0.3] + [-0.2] * 11)])
    _probe(monkeypatch, "dla", kernel, model, om, np.linspace(4200.0, 4310.0, 6000), thetas, lb, ub, segs=1)


@pytest.mark.parametrize("kernel", ["stream", "tile"])
def test_exp_switch_straddled(monkeypatch, kernel):
    """Rows whose largest optical depth lies just below and just above 2^-6 (where the kernels switch between the
    short exp of optically thin rows and the full one), and one well above."""
    from oracle import voigt_oracle as vo
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems)
    wave = np.linspace(3740.0, 3810.0, 5000)
    C = 4
    base = th.copy()
    base[:C] = 12.0
    tau0 = vo.model_flux(om, base, wave, return_tau=True).max()
    thetas = []
    for target in (2.0 ** -6 * 0.999, 2.0 ** -6 * 1.001, 2.0 ** -6 * 1.05, 0.2):
        t = base.copy()
        t[:C] += np.log10(target / tau0)                   # tau is linear in 10^N: the largest tau is the target
        thetas.append(t)
    thetas = np.array(thetas)
    for t, target in zip(thetas, (2.0 ** -6 * 0.999, 2.0 ** -6 * 1.001, 2.0 ** -6 * 1.05, 0.2)):
        assert abs(vo.model_flux(om, t, wave, return_tau=True).max() / target - 1) < 1e-9
    lb, ub = np.minimum(lb, thetas.min(0)), np.maximum(ub, thetas.max(0))
    _probe(monkeypatch, "exp switch", kernel, model, om, wave, thetas, lb, ub, segs=1)


@pytest.mark.parametrize("kernel", ["stream", "tile"])
def test_fast_voigt_method(monkeypatch, kernel):
    """voigt_method='fast' (the streaming kernel's tau_fast path; oracle H_tepper_garcia)."""
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems, voigt_method="fast")
    _probe(monkeypatch, "fast", kernel, model, om, np.linspace(3740.0, 3810.0, 5000), _rows(th, lb, ub, 3, 5), lb, ub,
           segs=1)


# --------------------------------------------------------------------------------- unsorted grids
@pytest.mark.parametrize("order", ["descending", "permuted"])
@pytest.mark.parametrize("segs", [None, 1])
def test_unsorted_grids(monkeypatch, order, segs):
    """The streaming kernel takes the range of 1/lambda of each super-chunk from a min/max table."""
    systems, th, lb, ub = _mgii(4)
    model, om = _models(systems)
    wave = np.linspace(3740.0, 3810.0, 5000)
    wave = wave[::-1].copy() if order == "descending" else np.random.default_rng(3).permutation(wave)
    _probe(monkeypatch, "grids", "stream", model, om, wave, _rows(th, lb, ub, 3, 6), lb, ub, segs=segs)


# --------------------------------------------------------------------------------- golden tie-in
def test_c5a_probes_vs_reference_flux(monkeypatch):
    """C5a (100 000 px, L = 33, default schedule, boundary records on): the streaming kernel's probed flux for the
    fixture's flux rows against the live reference's own model flux.  The fixture keeps 19 780 pixels; probed here
    are a seeded subset of those within K + 1 of a multiple of 1024 and a seeded sample of the rest."""
    from golden_util import Golden
    from test_gpu_parity import _gpu_models
    g = Golden("C5a")
    n = g.instruments[0]
    model = _gpu_models(g)[n]
    wave, fpx, ref = g.inst(n, "wave"), g.inst(n, "flux_px"), g.inst(n, "ref_flux")
    K = model.compile().data.kernel.size
    near = np.isin(fpx, spu.boundary_windows(wave.size, K))
    rng = np.random.default_rng(5)
    pick = np.sort(np.concatenate([rng.choice(np.flatnonzero(near), 320, replace=False),
                                   rng.choice(np.flatnonzero(~near), 64, replace=False)]))
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    monkeypatch.delenv("RBVFIT_B200_STREAM_SEGS", raising=False)
    got, ran = spu.probe_model_flux(model, wave, g.thetas[g.flux_rows], fpx[pick], g.lb, g.ub)
    assert ran == "stream"
    d = np.max(np.abs(got - ref[:, pick]))
    _note("C5a stream vs reference", d)
    assert d <= FLUX_TOL, d


# --------------------------------------------------------------------------------- joint fits
def _joint_instruments():
    """Three instruments of one fit with different P, K and L (same four HI components): (3000 px, K = 3, L = 4),
    (9000 px, K = 65, L = 36), (5000 px, no LSF, L = 8)."""
    zs = [2.30, 2.45, 2.60, 2.75]
    lyman = [1215.67, 1025.72, 972.54, 949.74, 937.80, 930.75, 926.23, 923.15, 920.96]
    spec = {"A": (1, np.linspace(4000.0, 4570.0, 3000), None, _asym_taps(3)),
            "B": (9, np.linspace(3000.0, 3700.0, 9000), None, _asym_taps(65)),
            "C": (2, np.linspace(3350.0, 4600.0, 5000), None, None)}
    out = {}
    for name, (nt, wave, fwhm, taps) in spec.items():
        model, om = _models([(z, "HI", lyman[:nt], 1) for z in zs], FWHM=fwhm, taps=taps)
        out[name] = (model, om, wave)
    assert [out[k][1].n_lines for k in "ABC"] == [4, 36, 8]
    th = np.array([14.6, 13.4, 15.2, 13.9, 22.0, 35.0, 18.0, 28.0, 5.0, -20.0, 12.0, 0.0])
    lb = th - np.concatenate([np.full(4, 1.5), np.full(4, 12.0), np.full(4, 40.0)])
    ub = th + np.concatenate([np.full(4, 1.5), np.full(4, 30.0), np.full(4, 40.0)])
    return out, th, lb, ub


@pytest.mark.parametrize("segs", [None, 1])
def test_joint_fit_equals_sum_of_instruments(monkeypatch, segs):
    """Slot -> instrument mapping, line bases and a record stride set by the widest K: the joint lnprob is the sum of
    the single-instrument ones.  With the same schedule and the same boundary-record decision (B and C: records on
    alone and jointly) the sum is bit-identical; A alone has too few lines for records, so A + B + C agrees to
    rounding."""
    from rbvfit_b200.likelihood import GpuLikelihood
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    if segs is None:
        monkeypatch.delenv("RBVFIT_B200_STREAM_SEGS", raising=False)
    else:
        monkeypatch.setenv("RBVFIT_B200_STREAM_SEGS", str(segs))
    inst, th, lb, ub = _joint_instruments()
    rng = np.random.default_rng(61)
    data = {}
    for name, (model, om, wave) in inst.items():
        flux = model.compile().model_flux(th, wave) + 0.02 * rng.standard_normal(wave.size)
        data[name] = dict(model=model, wave=wave, flux=flux, error=np.full(wave.size, 0.02))
    rows = _rows(th, lb, ub, 8, 62)
    single = {}
    for name in data:
        like = GpuLikelihood({name: data[name]}, lb, ub)
        single[name] = like.lnprob(rows)
        assert like.engine.last_kernel == "stream"
        like.close()
    for names in ("ABC", "BC"):
        like = GpuLikelihood({k: data[k] for k in names}, lb, ub)
        got = like.lnprob(rows)
        assert like.engine.last_kernel == "stream"
        like.close()
        want = np.zeros(len(rows))
        for k in names:
            want = want + single[k]
        rel = np.max(np.abs(got - want) / np.abs(want))
        _note(f"joint {names} vs sum of instruments, rel.", rel)
        assert rel <= 1e-13, (names, rel)
        if names == "BC":
            assert np.array_equal(got, want)


@pytest.mark.parametrize("segs", [None, 1])
def test_joint_fit_boundary_windows_vs_oracle(monkeypatch, segs):
    """Only the pixels within K + 2 of each multiple of 1024 enter (weight_mask), data = oracle flux + 1, error 1:
    every residual is 1 + (M_oracle - M), so |d lnprob| <= 1e-10 per pixel is the flux contract itself."""
    from rbvfit_b200.likelihood import GpuLikelihood
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    if segs is None:
        monkeypatch.delenv("RBVFIT_B200_STREAM_SEGS", raising=False)
    else:
        monkeypatch.setenv("RBVFIT_B200_STREAM_SEGS", str(segs))
    inst, th, lb, ub = _joint_instruments()
    rows = _rows(th, lb, ub, 3, 63, scale=np.concatenate([np.full(4, 0.01), np.full(4, 0.1), np.full(4, 0.2)]))
    data, want, n_win = {}, np.zeros(len(rows)), 0
    for name, (model, om, wave) in inst.items():
        win = spu.boundary_windows(wave.size, spu.n_taps(om))
        mask = np.zeros(wave.size, dtype=bool)
        mask[win] = True
        flux = np.ones(wave.size)
        flux[win] = spu.oracle_flux_at(om, th, wave, win) + 1.0
        data[name] = dict(model=model, wave=wave, flux=flux, error=np.ones(wave.size), weight_mask=mask)
        for r, t in enumerate(rows):
            want[r] += -0.5 * np.sum((flux[win] - spu.oracle_flux_at(om, t, wave, win)) ** 2)
        n_win += win.size
    like = GpuLikelihood(data, lb, ub)
    got = like.lnprob(rows)
    assert like.engine.last_kernel == "stream"
    like.close()
    d = np.abs(got - want)
    _note("joint boundary windows |d lnprob| / N_window", np.max(d) / n_win)
    assert np.all(d <= 1e-10 * n_win + 1e-15 * np.abs(want)), (d, n_win)


def test_sightline_batch_weight_mask_shape_error():
    from rbvfit_b200.likelihood import SightlineBatch
    systems, th, lb, ub = _mgii(2)
    model, _om = _models(systems)
    wave = np.linspace(3755.0, 3795.0, 500)
    good = dict(model=model, wave=wave, flux=np.ones(500), error=np.ones(500))
    with pytest.raises(ValueError, match="sightline 1: weight_mask"):
        SightlineBatch([good, dict(good, weight_mask=np.ones(499, dtype=bool))], lb, ub)


# --------------------------------------------------------------------------------- invariants
@pytest.fixture(scope="module")
def invariant_problem():
    systems, th, lb, ub = _mgii(4)
    model, _om = _models(systems)
    wave = np.linspace(3700.0, 3860.0, 9000)
    rng = np.random.default_rng(71)
    flux = model.compile().model_flux(th, wave) + 0.05 * rng.standard_normal(wave.size)
    data = dict(model=model, wave=wave, flux=flux, error=np.full(wave.size, 0.05))
    return data, _rows(th, lb, ub, 700, 72), lb, ub


def test_stream_lnprob_is_bit_identical_across_batches(monkeypatch, invariant_problem):
    """A row's lnprob does not depend on the batch size, its position, the number of resident CTAs, or on whether it
    comes from a joint-fit context or a one-sightline survey context (the schedule depends on the spectrum only)."""
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    data, rows, lb, ub = invariant_problem
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    monkeypatch.delenv("RBVFIT_B200_STREAM_SEGS", raising=False)
    like = GpuLikelihood({"S": data}, lb, ub)
    ref = like.lnprob(rows)
    assert like.engine.last_kernel == "stream" and np.all(np.isfinite(ref))
    rng = np.random.default_rng(73)
    for W in (1, 5, 64, 700):
        for _ in range(2):
            idx = rng.choice(700, W, replace=False)
            got = like.lnprob(rows[idx])
            assert like.engine.last_kernel == "stream"
            assert np.array_equal(np.atleast_1d(got), ref[idx]), W
    like.close()
    monkeypatch.setenv("RBVFIT_B200_STREAM_CTAS", "1")
    like = GpuLikelihood({"S": data}, lb, ub)
    assert np.array_equal(like.lnprob(rows), ref)
    assert like.engine.last_kernel == "stream"
    like.close()
    monkeypatch.delenv("RBVFIT_B200_STREAM_CTAS")
    batch = SightlineBatch([data], lb, ub)
    assert np.array_equal(batch.lnprob(rows[None])[0], ref)
    assert batch.engine.last_kernel == "stream"
    batch.close()


# --------------------------------------------------------------------------------- samplers on the streaming kernel
@pytest.fixture()
def sampler_problem(monkeypatch):
    """8 lines, 3000 px in uniform 1-segment ranges: three ranges and boundary records, so the stretch move runs
    finalize_stream_kernel with the fused accept."""
    from rbvfit_b200.likelihood import GpuLikelihood
    monkeypatch.setenv("RBVFIT_B200_STREAM", "1")
    monkeypatch.setenv("RBVFIT_B200_STREAM_SEGS", "1")
    systems, th, lb, ub = _mgii(4)
    model, _om = _models(systems)
    wave = np.linspace(3755.0, 3795.0, 3000)
    rng = np.random.default_rng(81)
    flux = model.compile().model_flux(th, wave) + 0.05 * rng.standard_normal(wave.size)
    data = dict(model=model, wave=wave, flux=flux, error=np.full(wave.size, 0.05))
    like = GpuLikelihood({"S": data}, lb, ub)
    yield like, data, th, lb, ub
    like.close()


def test_stretch_sampler_on_the_streaming_kernel_matches_replay(sampler_problem):
    from oracle import stretch_replay as sr
    from rbvfit_b200.sampler import DeviceEnsembleSampler
    like, _data, th, lb, ub = sampler_problem
    rng = np.random.default_rng(82)
    for W in (16, 21):
        p0 = np.clip(th + 1e-3 * rng.standard_normal((W, th.size)), lb, ub)
        dev = DeviceEnsembleSampler(W, th.size, like, seed=77)
        dev.run_mcmc(p0, 40)
        assert like.engine.last_kernel == "stream"
        chain, lps, nacc = sr.run(like.lnprob, p0, like.lnprob(p0), 40, dev._seed)
        assert np.allclose(dev.get_chain(), chain, rtol=0, atol=1e-9)
        assert np.max(np.abs(dev.get_log_prob() - lps) / np.abs(lps)) <= 1e-9
        assert np.array_equal(np.rint(dev.acceptance_fraction * 40).astype(int), nacc)
        assert nacc.sum() > 0


def test_slice_sampler_on_the_streaming_kernel_matches_replay(sampler_problem):
    from oracle import slice_replay as sl
    from rbvfit_b200.slice_sampler import DeviceEnsembleSliceSampler
    like, _data, th, lb, ub = sampler_problem
    rng = np.random.default_rng(83)
    W, nsteps = 24, 20                     # zeus: at least 2 ndim walkers
    p0 = np.clip(th + 1e-3 * rng.standard_normal((W, th.size)), lb, ub)
    dev = DeviceEnsembleSliceSampler(W, th.size, like, seed=77, depth=1)
    dev.run_mcmc(p0, nsteps)
    assert like.engine.last_kernel == "stream"
    ref = sl.run(like.lnprob, p0, like.lnprob(p0), nsteps, dev._seed)
    assert np.allclose(dev.get_chain(), ref["chain"], rtol=0, atol=1e-9)
    assert np.max(np.abs(dev.get_log_prob() - ref["lnp_chain"]) / np.abs(ref["lnp_chain"])) <= 1e-9
    assert (dev.nexp, dev.ncon) == (ref["nexp"], ref["ncon"])
    assert dev.ncall == W + ref["ncall"] and dev.mu == ref["mu"]


def test_sightline_slice_sampler_on_the_streaming_kernel_matches_replays(sampler_problem):
    from oracle import slice_replay_sightlines as sl
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.slice_sampler import SightlineEnsembleSliceSampler
    _like, data, th, lb, ub = sampler_problem
    rng = np.random.default_rng(84)
    sight = [data] + [dict(data, flux=data["flux"] + 0.05 * rng.standard_normal(data["flux"].size)) for _ in range(2)]
    batch = SightlineBatch(sight, lb, ub)
    singles = [GpuLikelihood({"S": s}, lb, ub) for s in sight]
    S, W, nsteps = len(sight), 24, 15
    p0 = np.clip(th + 1e-3 * rng.standard_normal((S, W, th.size)), lb, ub)
    smp = SightlineEnsembleSliceSampler(W, th.size, batch, seed=77, depth=1)
    smp.run_mcmc(p0, nsteps)
    assert batch.engine.last_kernel == "stream"
    chain, lps = smp.get_chain(), smp.get_log_prob()
    for e in range(S):
        like = singles[e]
        ref = sl.run(like.lnprob, p0[e], like.lnprob(p0[e]), nsteps, smp._seed, walker_offset=e * W)
        assert like.engine.last_kernel == "stream"
        assert np.allclose(chain[:, e], ref["chain"], rtol=0, atol=1e-9), e
        assert np.max(np.abs(lps[:, e] - ref["lnp_chain"]) / np.abs(ref["lnp_chain"])) <= 1e-9, e
        assert (smp.nexp[e], smp.ncon[e], smp.ncall[e]) == (ref["nexp"], ref["ncon"], W + ref["ncall"]), e
        assert smp.mu[e] == ref["mu"], e
    for like in singles:
        like.close()
    batch.close()
