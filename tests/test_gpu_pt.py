"""GPU: parallel tempering on the device (rbv_pt_run, DeviceParallelTemperingSampler) -- bit-for-bit against the
stretch-move sampler and the numpy replay, the evidence against brute-force quadrature, model selection,
label-switching, and vfit(sampler='pt')."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ONE_COMP = ([13.0], [30.0], [0.0])       # unsaturated MgII doublet component


def _models(w, comps=None):
    from rbvfit_b200 import FitConfiguration, lsf
    from rbvfit_b200.model import GpuVoigtModel
    cfg = FitConfiguration()
    for (z, ion, trans, c) in w["systems"]:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=c if comps is None else comps)
    return {name: GpuVoigtModel(cfg, FWHM=inst["FWHM"],
                                lsf_taps=lsf.cos_like_taps(321) if inst.get("lsf") == "cos_like" else None)
            for name, inst in w["instruments"].items()}


def _fitter(w, spectra, theta0, lb, ub, comps=None, nwalkers=32, nsteps=60, seed=5, sampler="emcee", betas=None):
    from rbvfit_b200.vfit_mcmc import vfit
    data = {n: dict(model=m, **spectra[n]) for n, m in _models(w, comps).items()}
    return vfit(data, theta0, lb, ub, no_of_Chain=nwalkers, no_of_steps=nsteps, seed=seed, sampler=sampler,
                betas=betas)


def _workload(name):
    """A workload and its spectra (GPU model at theta_true + seeded noise)."""
    from rbvfit_b200 import workloads as wl
    w = wl.get_workload(name)
    compiled = {n: m.compile() for n, m in _models(w).items()}
    return w, wl.make_spectra(w, lambda n, th, wave: compiled[n].model_flux(th, wave))


def _c1(nwalkers=32, seed=5, **kw):
    w, spectra = _workload("C1")
    theta0 = np.clip(w["theta_true"] + np.array([0.05, -0.05, 2, -2, 3, -3.0]), w["lb"], w["ub"])
    return w, _fitter(w, spectra, theta0, w["lb"], w["ub"], nwalkers=nwalkers, seed=seed, **kw)


def _start(w, T, W, seed, scale=1e-3):
    rng = np.random.default_rng(seed)
    return np.clip(w["theta_true"] + np.asarray(scale) * rng.standard_normal((T, W, len(w["lb"]))), w["lb"], w["ub"])


def _replay(like, smp, p0, nsteps, n_record=1, adapt=False, first_step=0, bh=None):
    from oracle import pt_replay as pr
    T, W, nd = p0.shape
    lp = like.lnprob(p0.reshape(-1, nd)).reshape(T, W)
    return pr.run(like.lnprob, p0, lp, smp._betas0, nsteps, smp._seed, first_step=first_step, n_record=n_record,
                  adapt=adapt, lag=smp.adaptation_lag, tau=smp.adaptation_time, beta_history_device=bh)


def test_one_temperature_is_the_stretch_sampler():
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler
    from rbvfit_b200.sampler import DeviceEnsembleSampler
    w, fitter = _c1()
    like = fitter._like
    p0 = _start(w, 1, 20, 3)[0]
    for use_graph, n in ((True, 60), (False, 25)):
        ref = DeviceEnsembleSampler(20, 6, like, seed=5, use_graph=use_graph)
        ref.run_mcmc(p0, n)
        pt = DeviceParallelTemperingSampler(20, 6, like, betas=[1.0], seed=5, use_graph=use_graph)
        pt.run_mcmc(p0, n)
        assert np.array_equal(pt.get_chain(), ref.get_chain())
        assert np.array_equal(pt.get_log_like()[:, 0], ref.get_log_prob())
        assert np.array_equal(pt.acceptance_fraction[0], ref.acceptance_fraction)
        assert pt.tswap_acceptance_fraction.shape == (0,)


@pytest.mark.parametrize("use_graph,n_record,adapt", [(True, 1, False), (False, 4, False), (True, 4, True)])
def test_four_temperatures_match_the_replay(use_graph, n_record, adapt):
    """T = 4 on C1 against oracle/pt_replay.py driven by the GPU lnprob: coordinates, the lnprob chain, swap and
    accept counts bit for bit (graph + chain sink / plain loop + device arrays; n_record 1 / T; adaptation, whose
    ladder the replay predicts to a few ulp and then takes from the device)."""
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler
    w, fitter = _c1()
    like = fitter._like
    T, W, n = 4, 20, 40
    betas = [1.0, 0.4, 0.1, 0.0]
    p0 = _start(w, T, W, 4, scale=[0.05, 0.05, 2, 2, 3, 3])
    smp = DeviceParallelTemperingSampler(W, 6, like, betas=betas, seed=11, use_graph=use_graph,
                                         adaptation_time=5.0)
    smp.run_mcmc(p0, n, adapt=adapt, n_record=n_record)
    bh = smp.beta_history if adapt else None
    r = _replay(like, smp, p0, n, n_record=n_record, adapt=adapt, bh=bh)
    for t in range(n_record):
        assert np.array_equal(smp.get_chain(temp=t), r["chain"][:, t]), t
    assert np.array_equal(smp.get_log_like(), r["lnp_chain"])
    assert np.array_equal(np.rint(smp.acceptance_fraction * n).astype(int), r["n_accepted"])
    assert np.array_equal(np.rint(smp.tswap_acceptance_fraction * n * W).astype(int), r["n_swaps"])
    assert r["n_swaps"].min() > 0
    if adapt:
        assert not np.array_equal(smp.beta_history[-1], betas)
        np.testing.assert_array_max_ulp(r["beta_pred"], smp.beta_history, maxulp=8)
        np.testing.assert_array_max_ulp(r["betas"], smp.betas, maxulp=8)
    else:
        assert np.array_equal(smp.beta_history, np.tile(betas, (n, 1))) and np.array_equal(smp.betas, betas)


def test_engine_device_arrays_with_graph_and_continuation():
    """Engine.pt_run with device chains under the CUDA graph equals the sampler's sink run; run(30) + run(None, 25)
    equals run(55)."""
    import torch
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler
    w, fitter = _c1()
    like = fitter._like
    eng = like.engine
    T, W = 3, 16
    betas = [1.0, 0.3, 0.0]
    p0 = _start(w, T, W, 6, scale=[0.05, 0.05, 2, 2, 3, 3])
    one = DeviceParallelTemperingSampler(W, 6, like, betas=betas, seed=3)
    one.run_mcmc(p0, 55, n_record=2)
    two = DeviceParallelTemperingSampler(W, 6, like, betas=betas, seed=3)
    two.run_mcmc(p0, 30, n_record=2)
    two.run_mcmc(None, 25, n_record=2)
    assert np.array_equal(one.get_chain(temp=1), two.get_chain(temp=1))
    assert np.array_equal(one.get_log_like(), two.get_log_like())
    assert np.array_equal(one.tswap_acceptance_fraction, two.tswap_acceptance_fraction)
    dev = eng.tdev
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        c = torch.as_tensor(p0, device=dev)
        lp = eng.lnprob_device(c.view(T * W, 6)).view(T, W).contiguous()
        b = torch.as_tensor(betas, dtype=torch.float64, device=dev)
        chain = torch.empty((55, 2, W, 6), dtype=torch.float64, device=dev)
        lps = torch.empty((55, T, W), dtype=torch.float64, device=dev)
        nacc = torch.zeros((T, W), dtype=torch.int32, device=dev)
        nsw = torch.zeros(T - 1, dtype=torch.int64, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        eng.pt_run(c, lp, b, 55, 2.0, one._seed, 0, chain, lps, None, nacc, nsw, flag, use_graph=True, n_record=2)
        st.synchronize()
    assert np.array_equal(chain.cpu().numpy(), one._all()[0])
    assert np.array_equal(lps.cpu().numpy(), one.get_log_like())
    with pytest.raises(Exception):       # betas[0] != 1 is refused by the library
        eng.pt_run(c, lp, torch.tensor([0.9, 0.3, 0.0], dtype=torch.float64, device=dev), 4, 2.0, 1, 0, None, None,
                   None, nacc, nsw, flag)
    with pytest.raises(Exception):       # n_record > T
        eng.pt_run(c, lp, b, 4, 2.0, 1, 0, None, None, None, nacc, nsw, flag, n_record=4)


def test_two_instruments_run_and_give_finite_evidence():
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler
    w, spectra = _workload("C3")
    fitter = _fitter(w, spectra, w["theta_true"], w["lb"], w["ub"])
    smp = DeviceParallelTemperingSampler(24, 6, fitter._like, betas=[1.0, 0.3, 0.05, 0.0], seed=2)
    smp.run_mcmc(_start(w, 4, 24, 7), 60)
    lnz, dlnz = smp.log_evidence_estimate(discard=20)
    assert np.isfinite(lnz) and np.isfinite(dlnz) and np.all(np.isfinite(smp.get_log_like()))


def _one_comp_problem(truth=ONE_COMP, P=512, seed=31):
    """A one-component MgII doublet spectrum (GPU model + seeded noise) and its workload dict."""
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    n, b, v = truth
    lb, ub = wl.default_bounds(n, b, v)
    w = dict(systems=[(0.348, "MgII", [2796.3, 2803.5], 1)],
             instruments={"COS": dict(wave=np.linspace(3760.0, 3790.0, P), FWHM="6.5", lsf=None)},
             theta_true=np.array(n + b + v), lb=lb, ub=ub)
    cfg = FitConfiguration()
    cfg.add_system(z=0.348, ion="MgII", transitions=[2796.3, 2803.5], components=1)
    wave = w["instruments"]["COS"]["wave"]
    model = GpuVoigtModel(cfg, FWHM="6.5").compile()
    flux = model.model_flux(w["theta_true"], wave) + wl.SIGMA * np.random.default_rng(seed).standard_normal(P)
    return w, {"COS": dict(wave=wave, flux=flux, error=np.full(P, wl.SIGMA))}


def _pt_evidence(fitter, betas, n=3000, burn=1000, seed=1):
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler
    best, _err = fitter.fit_quick(verbose=False, method="lm")
    fitter.theta = best
    p0 = fitter._initialize_walkers(best)
    smp = DeviceParallelTemperingSampler(fitter.nwalkers, fitter.ndim, fitter._like, betas=betas, seed=seed)
    smp.run_mcmc(p0, n)
    return smp, smp.log_evidence_estimate(discard=burn)


def test_evidence_matches_quadrature():
    """One unsaturated component (3 parameters, P = 512), ratio-1.5 ladder to beta = 0: lnZ within 0.3 nats of the
    midpoint rule over a 96^3 grid spanning +-8 sigma of the LM covariance (one device lnprob batch)."""
    from scipy.special import logsumexp
    w, spectra = _one_comp_problem()
    fitter = _fitter(w, spectra, w["theta_true"], w["lb"], w["ub"], comps=1)
    betas = np.append(1.5 ** -np.arange(0.0, 35.0), 0.0)
    smp, (lnz, dlnz) = _pt_evidence(fitter, betas)
    best = fitter.theta_best
    sig = np.sqrt(np.diag(fitter.theta_best_covariance))
    assert np.all(np.isfinite(sig))
    n = 96
    axes = [best[k] + sig[k] * (-8.0 + 16.0 * (np.arange(n) + 0.5) / n) for k in range(3)]
    grid = np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1).reshape(-1, 3)
    lnl = fitter._like.lnprob(grid)
    cell = np.prod(16.0 * sig / n)
    quad = logsumexp(lnl) + np.log(cell / np.prod(w["ub"] - w["lb"]))
    print(f"\nPT lnZ {lnz:.4f} +- {dlnz:.4f}, quadrature {quad:.4f}, difference {lnz - quad:+.4f}; "
          f"swap acceptance {np.round(smp.tswap_acceptance_fraction, 2)}")
    assert abs(lnz - quad) < 0.3


def test_model_selection():
    """C1's spectrum (two components): lnZ(2) - lnZ(1) > 10.  A spectrum drawn from one component:
    lnZ(1) >= lnZ(2) - 3 dlnZ."""
    from rbvfit_b200 import workloads as wl
    from rbvfit_b200.pt_sampler import default_betas
    w, spectra = _workload("C1")
    lb1, ub1 = wl.default_bounds([14.6], [40.0], [0.0])
    one = _fitter(w, spectra, np.array([14.6, 40.0, 0.0]), lb1, ub1, comps=1, nwalkers=40)
    two = _fitter(w, spectra, np.clip(w["theta_true"] + [0.05, -0.05, 2, -2, 3, -3.0], w["lb"], w["ub"]),
                  w["lb"], w["ub"], nwalkers=40)
    _s, (z1, d1) = _pt_evidence(one, default_betas(3), n=2000, burn=700)
    _s, (z2, d2) = _pt_evidence(two, default_betas(6), n=2000, burn=700)
    print(f"\nC1: lnZ(1) = {z1:.2f} +- {d1:.2f}, lnZ(2) = {z2:.2f} +- {d2:.2f}")
    assert z2 - z1 > 10
    w1, spectra1 = _one_comp_problem(truth=([13.4], [25.0], [0.0]), seed=41)
    one = _fitter(w1, spectra1, w1["theta_true"], w1["lb"], w1["ub"], comps=1, nwalkers=40)
    lb2, ub2 = wl.default_bounds([13.4, 13.0], [25.0, 25.0], [-10.0, 10.0])
    two = _fitter(w1, spectra1, np.array([13.3, 12.6, 25.0, 25.0, -2.0, 8.0]), lb2, ub2, comps=2, nwalkers=40)
    _s, (y1, e1) = _pt_evidence(one, default_betas(3), n=2000, burn=700)
    _s, (y2, e2) = _pt_evidence(two, default_betas(6), n=2000, burn=700)
    print(f"one-component spectrum: lnZ(1) = {y1:.2f} +- {e1:.2f}, lnZ(2) = {y2:.2f} +- {e2:.2f}")
    assert y1 >= y2 - 3 * max(e1, e2)


def test_label_switching():
    """Two components of one ion with identical bounds: an exactly label-symmetric posterior.  The cold PT chain
    visits both labellings (fraction in [0.2, 0.8]); the stretch sampler from the same start is reported."""
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler, default_betas
    from rbvfit_b200.sampler import DeviceEnsembleSampler
    w, spectra = _workload("C1")
    lb = np.array([12.2, 12.2, 2.0, 2.0, -75.0, -75.0])
    ub = np.array([16.5, 16.5, 80.0, 80.0, 85.0, 85.0])
    n, burn, W = 3000, 1000, 40
    fitter = _fitter(w, spectra, w["theta_true"], lb, ub, nwalkers=W)
    best, _e = fitter.fit_quick(verbose=False, method="lm")
    p0 = fitter._initialize_walkers(best)
    smp = DeviceParallelTemperingSampler(W, 6, fitter._like, betas=default_betas(6), seed=4)
    smp.run_mcmc(p0, n)
    cold = smp.get_chain(discard=burn)
    frac = float(np.mean(cold[..., 4] < cold[..., 5]))
    ref = DeviceEnsembleSampler(W, 6, fitter._like, seed=4)
    ref.run_mcmc(p0, n)
    c = ref.get_chain(discard=burn)
    frac_stretch = float(np.mean(c[..., 4] < c[..., 5]))
    print(f"\nlabelling v1 < v2: PT {frac:.3f}, stretch from the same start {frac_stretch:.3f}; "
          f"start {np.mean(p0[:, 4] < p0[:, 5]):.2f}")
    assert 0.2 <= frac <= 0.8


def test_vfit_pt_contract():
    w, fitter = _c1(nwalkers=24, sampler="pt", betas=[1.0, 0.5, 0.2, 0.05, 0.0])
    fitter.no_of_steps = 200
    fitter.runmcmc(optimize=True, verbose=True, progress=False)
    s = fitter.sampler
    assert fitter.mcmc_flag and fitter.pt_sampler.ntemps == 5
    assert s.get_chain().shape == (200, 24, 6) and s.get_chain(discard=100, flat=True).shape == (100 * 24, 6)
    assert s.get_log_prob().shape == (200, 24) and s.acceptance_fraction.shape == (24,)
    assert fitter.samples.shape == (100 * 24, 6) and fitter.best_theta.shape == (6,)
    assert s.get_autocorr_time(quiet=True).shape == (6,)
    assert fitter.get_samples(burn_in=0.5).shape == (100 * 24, 6)
    lo, hi = np.percentile(fitter.samples, [0.5, 99.5], axis=0)
    assert np.all(lo < w["theta_true"]) and np.all(w["theta_true"] < hi)
    lnz, dlnz = fitter.log_evidence()
    assert np.isfinite(lnz) and np.isfinite(dlnz)
    with pytest.raises(ValueError):
        _c1(sampler="nope")
