"""GPU: survey-mode Fisher matrix (rbv_lnlike_fisher_batch_sightlines) and the device Levenberg-Marquardt loop over
sightlines (rbv_lm_run_sightlines, SightlineBatch.fit_quick) against one-sightline contexts, the scalar replay
oracle/lm_replay.py and the host driver."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FISHER_TOL = 1e-8       # |device - oracle| <= FISHER_TOL * sqrt(F_ii F_jj)  (DESIGN.md section 15)


def _sightlines(indices, FWHM="6.5", extra=0, workload=None):
    """C5b sightlines (or copies of ``workload`` with their own noise): (SightlineBatch, [GpuLikelihood], lb, ub,
    theta_true, [oracle instruments])."""
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
    sight, singles, comps = [], [], []
    for s in indices:
        if workload is None:
            w = wl.c5b_sightline(s)
        else:
            w = dict(workload, seed=workload["seed"] + 1000 * s)
        cfg, ocfg = FitConfiguration(), vo.OracleConfig()
        for (z, ion, trans, c) in w["systems"]:
            cfg.add_system(z=z, ion=ion, transitions=trans, components=c)
            ocfg.add_system(z, ion, trans, c)
        om = vo.lower(ocfg, FWHM=FWHM)
        m = GpuVoigtModel(cfg, FWHM=FWHM)
        sp = next(iter(wl.make_spectra(w, lambda n, th, wave: vo.model_flux(om, th, wave)).values()))
        sight.append(dict(model=m, **sp))
        comps.append(vo.compile_instruments({"S": dict(model=om, **sp)}))
        lb = np.concatenate([w["lb"], np.zeros(extra)])
        ub = np.concatenate([w["ub"], np.ones(extra)])
        singles.append(GpuLikelihood({"S": dict(model=m, **sp)}, lb, ub))
    theta_true = np.concatenate([w["theta_true"], np.full(extra, 0.5)])
    batch = SightlineBatch(sight, lb, ub)
    batch.test_inputs = sight
    return batch, singles, lb, ub, theta_true, comps


def _starts(theta_true, lb, ub, S, seed):
    rng = np.random.default_rng(seed)
    C = (theta_true.size - theta_true.size % 3) // 3
    scale = np.concatenate([np.full(C, 0.1), np.full(C, 3.0), np.full(C, 4.0), np.zeros(theta_true.size - 3 * C)])
    return np.clip(theta_true + scale * rng.standard_normal((S, theta_true.size)), lb, ub)


def _close(batch, singles):
    batch.close()
    for s in singles:
        s.close()


def _fisher_rows_equal(batch, singles, theta):
    v, g, F = batch.lnlike_and_fisher(theta)
    for s, like in enumerate(singles):
        v1, g1, F1 = like.lnlike_and_fisher(theta[s])
        assert np.array_equal(v[s], v1) and np.array_equal(g[s], g1) and np.array_equal(F[s], F1), s
    return v, g, F


def test_sightline_fisher_bit_identical_to_single():
    from oracle import voigt_fisher_oracle as vf
    S, Ws = 24, 3
    batch, singles, lb, ub, t, comps = _sightlines(range(S))
    theta = np.stack([_starts(t, lb, ub, Ws, 10 + s) for s in range(S)])
    v, g, F = _fisher_rows_equal(batch, singles, theta)
    perm = np.random.default_rng(3).permutation(Ws)
    v2, g2, F2 = batch.lnlike_and_fisher(theta[:, perm])
    assert np.array_equal(v2, v[:, perm]) and np.array_equal(g2, g[:, perm]) and np.array_equal(F2, F[:, perm])
    batch.engine.fisher_chunk_bytes = 1                    # one walker of every sightline per launch
    v3, g3, F3 = batch.lnlike_and_fisher(theta)
    assert np.array_equal(v3, v) and np.array_equal(g3, g) and np.array_equal(F3, F)
    worst = 0.0
    for s in (0, 7, 23):
        _ll, _g, F_or = vf.lnlike_fisher(comps[s], theta[s, 1])
        d = np.sqrt(np.outer(np.diag(F_or), np.diag(F_or)))
        worst = max(worst, float(np.max(np.abs(F[s, 1] - F_or) / d)))
    print("sightline Fisher against the oracle:", worst)
    assert worst <= FISHER_TOL
    _close(batch, singles)


def test_sightline_fisher_many_sightlines_and_no_lsf():
    S = 40                                                  # beyond the 16-instrument kernel-parameter tables
    batch, singles, lb, ub, t, _ = _sightlines(range(S))
    _fisher_rows_equal(batch, singles, _starts(t, lb, ub, S, 5)[:, None, :])
    _close(batch, singles)
    batch, singles, lb, ub, t, _ = _sightlines(range(4), FWHM=None)
    n0 = batch.engine.launch_count
    _fisher_rows_equal(batch, singles, np.stack([_starts(t, lb, ub, 2, s) for s in range(4)]))
    assert batch.engine.launch_count - n0 == 6             # prep, flux, resid, columns, Gram, finalize: no LSF pass
    _close(batch, singles)


def _replay_all(singles, x0, lb, ub, **kw):
    from oracle import lm_replay
    return [lm_replay.run(like.lnlike_and_fisher, x0[s], lb, ub, **kw) for s, like in enumerate(singles)]


def _assert_replayed(res, reps):
    for s, r in enumerate(reps):
        assert np.array_equal(res.x[s], r.x), s
        assert res.chi2[s] == r.chi2 and res.n_evals[s] == r.n_evals and res.status[s] == r.status, s
        assert np.array_equal(np.isnan(res.cov[s]), np.isnan(r.cov)), s
        ok = np.isfinite(r.cov)
        assert np.max(np.abs(res.cov[s] - r.cov)[ok], initial=0.0) <= 1e-12 * np.max(np.abs(r.cov)[ok], initial=1.0)


def test_device_lm_equals_replay():
    from rbvfit_b200 import lm
    S = 10
    batch, singles, lb, ub, t, _ = _sightlines(range(S))
    x0 = _starts(t, lb, ub, S, 21)
    x0[2, 0] = ub[0]                                       # a start on a bound
    x0[5, 3] = lb[3]
    n0 = batch.engine.launch_count
    res = batch.fit_quick(x0)
    launches = batch.engine.launch_count - n0
    print("statuses", res.status, "n_evals", res.n_evals, "launches", launches)
    assert np.all(res.status > 0)
    assert launches == 1 + res.n_evals.max() * 8           # init + per iteration 7 Fisher launches and the update
    _assert_replayed(res, _replay_all(singles, x0, lb, ub))
    assert np.array_equal(res.errors, np.sqrt(np.diagonal(res.cov, axis1=1, axis2=2)), equal_nan=True)
    with pytest.warns(UserWarning, match=f"{S} of {S} sightlines"):
        short = batch.fit_quick(x0, max_evals=3)
    assert np.all(short.status == lm.STATUS_MAX_EVALS) and np.all(short.n_evals == 3)
    _assert_replayed(short, _replay_all(singles, x0, lb, ub, max_evals=3))
    _close(batch, singles)


def test_device_lm_unconstrained_parameter():
    """ndim = 3C + 1: the extra column of J is exactly 0, so F_ii = 0, the parameter never moves and its covariance
    row and column are NaN."""
    S = 8
    batch, singles, lb, ub, t, _ = _sightlines(range(S), extra=1)
    x0 = _starts(t, lb, ub, S, 4)
    res = batch.fit_quick(x0)
    assert np.all(res.status > 0)
    assert np.array_equal(res.x[:, -1], x0[:, -1])
    assert np.all(np.isnan(res.cov[:, -1, :])) and np.all(np.isnan(res.cov[:, :, -1]))
    assert np.all(np.isfinite(res.cov[:, :-1, :-1]))
    _assert_replayed(res, _replay_all(singles, x0, lb, ub))
    _close(batch, singles)


def test_device_lm_vs_host_fit_quick():
    from rbvfit_b200.vfit_mcmc import vfit
    S = 4
    batch, singles, lb, ub, t, _ = _sightlines(range(S))
    x0 = _starts(t, lb, ub, S, 8)
    res = batch.fit_quick(x0)
    worst = dict(chi2=0.0, x=0.0, cov=0.0)
    for s in range(S):
        fitter = vfit({"S": batch.test_inputs[s]}, x0[s], lb, ub, no_of_Chain=8, no_of_steps=2)
        best, _err = fitter.fit_quick(verbose=False, method="lm")
        cov = fitter.theta_best_covariance
        chi2 = -2.0 * singles[s].lnlike(best)
        sig = np.sqrt(np.diag(cov))
        ok = np.isfinite(sig)
        assert np.array_equal(ok, np.isfinite(res.errors[s])) and np.array_equal(res.x[s][~ok], best[~ok])
        worst["chi2"] = max(worst["chi2"], abs(res.chi2[s] - chi2) / abs(chi2))
        worst["x"] = max(worst["x"], float(np.max(np.abs(res.x[s] - best)[ok] / sig[ok])))
        dd = np.sqrt(np.outer(sig, sig))
        both = np.isfinite(dd)
        worst["cov"] = max(worst["cov"], float(np.max(np.abs(res.cov[s] - cov)[both] / dd[both])))
        fitter._like.close()
    print("device LM against vfit.fit_quick(method='lm'):", worst)
    assert worst["chi2"] <= 1e-10 and worst["x"] <= 1e-4
    assert worst["cov"] <= 1e-6     # the two x differ in their last digits; DESIGN.md section 16 records the value
    _close(batch, singles)


def test_device_lm_independent_of_block_and_order():
    S = 8
    batch, singles, lb, ub, t, _ = _sightlines(range(S))
    x0 = _starts(t, lb, ub, S, 30)
    full = batch.engine.lm_sightlines(x0, 0, S)
    a = batch.engine.lm_sightlines(x0[:3], 0, 3)
    b = batch.engine.lm_sightlines(x0[3:], 3, S - 3)
    for i in range(6):
        assert np.array_equal(np.concatenate([a[i], b[i]]), full[i], equal_nan=i in (0, 1, 2))
    _close(batch, singles)
    perm = np.random.default_rng(2).permutation(S)
    pbatch, psingles, *_ = _sightlines(perm)
    p = pbatch.engine.lm_sightlines(x0[perm], 0, S)
    for i in range(6):
        assert np.array_equal(p[i], full[i][perm], equal_nan=i in (0, 1, 2))
    _close(pbatch, psingles)


def test_device_lm_c2_structure():
    """Four sightlines of C2's structure (12 components, 36 parameters, 20 000 pixels)."""
    from rbvfit_b200 import workloads as wl
    w = wl.get_workload("C2")
    batch, singles, lb, ub, t, _ = _sightlines(range(4), workload=w)
    rng = np.random.default_rng(7)
    C = 12
    x0 = np.clip(t + np.concatenate([np.full(C, 0.02), np.full(C, 0.5), np.full(C, 0.5)]) *
                 rng.standard_normal((4, 3 * C)), lb, ub)
    res = batch.fit_quick(x0)
    print("C2 structure: status", res.status, "n_evals", res.n_evals)
    assert np.all(res.status > 0)
    _assert_replayed(res, _replay_all(singles, x0, lb, ub))
    _close(batch, singles)


def test_device_lm_coverage_c1():
    """test_lm_coverage_c1 as one 64-sightline batch: the mean Mahalanobis distance of the fits from theta_true is 6
    within 3.5 standard errors."""
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.likelihood import SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
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
    model = GpuVoigtModel(cfg, FWHM=spec["FWHM"])
    sight = [dict(model=model, wave=wave, flux=clean + sigma * rng.standard_normal(wave.size), error=err)
             for _ in range(64)]
    batch = SightlineBatch(sight, w["lb"], w["ub"])
    res = batch.fit_quick(t)
    assert np.all(res.status > 0) and np.all(np.isfinite(res.cov))
    dx = res.x - t
    d2 = np.array([dx[s] @ np.linalg.solve(res.cov[s], dx[s]) for s in range(64)])
    print("C1 coverage, one 64-sightline batch: mean Mahalanobis distance", d2.mean())
    assert 4.5 <= d2.mean() <= 7.5
    batch.close()


def test_errors():
    import torch
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200._lib import RbvError
    from rbvfit_b200.engine import Engine
    from rbvfit_b200.model import GpuVoigtModel

    def engine(P=(2048, 2048), components=2, method="wofz", flux=True, bounds=True, ndim=None):
        cfg = FitConfiguration()
        cfg.add_system(z=0.35, ion="MgII", transitions=[2796.3, 2803.5], components=components)
        data = GpuVoigtModel(cfg, FWHM="6.5", voigt_method=method).compile(verbose=False).data
        eng = Engine()
        n = 3 * components if ndim is None else ndim
        if ndim is not None:         # rbv_set_bounds refuses ndim < 3C once the instruments are there
            eng.set_bounds(np.full(n, -1e3), np.full(n, 1e3))
        for p in P:
            wave = np.linspace(3760.0, 3800.0, p)
            kw = dict(flux=np.ones(p), inv_sigma2=np.full(p, 400.0), log_inv_sigma2=np.full(p, np.log(400.0))) \
                if flux else {}
            eng.add_instrument(data, wave, taps=data.kernel, normalize_taps=data.kernel_normalize, **kw)
        if bounds and ndim is None:
            eng.set_bounds(np.full(n, -1e3), np.full(n, 1e3))
        return eng, np.tile(np.concatenate([np.full(components, 14.0), np.full(components, 30.0),
                                            np.linspace(-20, 20, components)])[:ndim], (len(P), 1))

    def code(fn):
        with pytest.raises(RbvError) as e:
            fn()
        return int(str(e.value).split("status ")[1].split(")")[0])

    eng, th = engine(P=(2048, 1024))
    assert code(lambda: eng.lnlike_fisher_sightlines_host(th, 1)) == 1          # mismatched geometry
    assert code(lambda: eng.lm_sightlines(th, 0, 2)) == 1
    eng.close()
    eng, th = engine()
    thd = torch.as_tensor(np.concatenate([th, th]), device=eng.tdev)
    assert code(lambda: eng.lnlike_fisher_sightlines_device(thd, 1)) == 1        # n_walkers != S * wps
    assert code(lambda: eng.lm_sightlines(th[:1], 2, 1)) == 1                     # bad [first, first + n)
    assert code(lambda: eng.lm_sightlines(th, -1, 2)) == 1
    ws = torch.empty(8, dtype=torch.uint8, device=eng.tdev)
    out = torch.empty(64, dtype=torch.float64, device=eng.tdev)
    th2 = torch.as_tensor(th, device=eng.tdev)
    assert eng.lib.rbv_lnlike_fisher_batch_sightlines(eng._h, th2.data_ptr(), 2, 1, out.data_ptr(), out.data_ptr(),
                                                      out.data_ptr(), ws.data_ptr(), 8, eng._stream()) == 3
    eng.close()
    eng, th = engine(method="fast")
    assert code(lambda: eng.lm_sightlines(th, 0, 2)) == 1                        # voigt_method='fast'
    eng.close()
    eng, th = engine(ndim=5)
    assert code(lambda: eng.lnlike_fisher_sightlines_host(th, 1)) == 1           # ndim < 3C
    eng.close()
    eng, th = engine(components=320, P=(64, 64))
    assert code(lambda: eng.lm_sightlines(th, 0, 2)) == 1                        # too many components for the Gram pass
    eng.close()
    eng, th = engine(flux=False)
    assert code(lambda: eng.lm_sightlines(th, 0, 2)) == 4                        # flux-only sightline
    eng.close()
    eng, th = engine(bounds=False)
    eng.ndim = 6
    assert code(lambda: eng.lnlike_fisher_sightlines_host(th, 1)) == 4           # bounds not set
    eng.close()
