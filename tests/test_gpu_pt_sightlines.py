"""GPU: survey-mode parallel tempering (rbv_pt_run_sightlines, SightlineParallelTemperingSampler) -- one tempered
ladder per sightline of a SightlineBatch in one device loop, with the thermodynamic-integration moments accumulated on
the device.  Bit for bit against the joint sampler, the survey stretch move and the numpy replay; independence,
continuation, the evidence from the moments, model selection across a survey, and the launch count."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BETAS4 = [1.0, 0.4, 0.1, 0.0]


def _sightlines(indices, singles_for=None, repeat=1):
    """C5b sightlines (C1's structure, each at its own redshift) as a SightlineBatch (the list ``repeat`` times over)
    plus one single-sightline GpuLikelihood for each index in ``singles_for`` (default: all)."""
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
    sight, singles = [], []
    keep = set(indices if singles_for is None else singles_for)
    for s in indices:
        w = wl.c5b_sightline(s)
        cfg = FitConfiguration()
        for (z, ion, trans, comps) in w["systems"]:
            cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        m = GpuVoigtModel(cfg, FWHM="6.5")
        c = m.compile()
        sp = wl.make_spectra(w, lambda n, th, wave: c.model_flux(th, wave))["COS"]
        sight.append(dict(model=m, **sp))
        if s in keep:
            singles.append(GpuLikelihood({"COS": dict(model=m, **sp)}, w["lb"], w["ub"]))
    w0 = wl.c5b_sightline(indices[0])
    return w0, SightlineBatch(sight * repeat, w0["lb"], w0["ub"]), singles


@pytest.fixture(scope="module")
def c5b():
    return _sightlines(list(range(5)))


SCALE = np.array([0.05, 0.05, 2.0, 2.0, 3.0, 3.0])


def _start(w0, shape, seed, scale=SCALE):
    rng = np.random.default_rng(seed)
    nd = len(w0["theta_true"])
    return np.clip(w0["theta_true"] + scale * rng.standard_normal(tuple(shape) + (nd,)), w0["lb"], w0["ub"])


@pytest.mark.parametrize("use_graph,n_record,adapt", [(True, 1, False), (False, 2, False), (True, 1, True)])
def test_one_sightline_is_the_joint_sampler(use_graph, n_record, adapt):
    """S = 1: chain, lnprob chain, acceptances, swaps and ladder equal DeviceParallelTemperingSampler on that
    sightline's GpuLikelihood bit for bit (graph + chain sink / plain loop / adaptation)."""
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler, SightlineParallelTemperingSampler
    w0, batch, singles = _sightlines([0])
    T, W, n, nd = 4, 16, 40, batch.ndim
    p0 = _start(w0, (1, T, W), 4)
    ref = DeviceParallelTemperingSampler(W, nd, singles[0], betas=BETAS4, seed=11, use_graph=use_graph,
                                         adaptation_time=5.0)
    ref.run_mcmc(p0[0], n, adapt=adapt, n_record=n_record)
    smp = SightlineParallelTemperingSampler(W, nd, batch, betas=BETAS4, seed=11, use_graph=use_graph,
                                            record_log_like=True, adaptation_time=5.0)
    smp.run_mcmc(p0, n, adapt=adapt, n_record=n_record)
    for t in range(n_record):
        assert np.array_equal(smp.get_chain(temp=t, sightline=0), ref.get_chain(temp=t)), t
    assert np.array_equal(smp.get_log_like(sightline=0), ref.get_log_like())
    assert np.array_equal(smp.acceptance_fraction[0], ref.acceptance_fraction)
    assert np.array_equal(smp.tswap_acceptance_fraction[0], ref.tswap_acceptance_fraction)
    assert np.array_equal(smp.beta_history[:, 0], ref.beta_history) and np.array_equal(smp.betas[0], ref.betas)
    assert ref.tswap_acceptance_fraction.min() > 0
    if adapt:
        assert smp.evidence_steps == 0 and not np.array_equal(smp.betas[0], BETAS4)
    else:
        assert smp.evidence_steps == n
        lnz, dlnz = smp.log_evidence_estimate()
        assert abs(lnz[0] - ref.log_evidence_estimate()[0]) < 1e-8
    v = smp.sightline(0)
    assert np.array_equal(v.cold().get_chain(), ref.cold().get_chain())
    assert np.array_equal(v.cold().get_log_prob(), ref.cold().get_log_prob())
    batch.close()
    singles[0].close()


def test_one_temperature_is_the_survey_stretch_move(c5b):
    """T = 1 reproduces SightlineEnsembleSampler (rbv_stretch_run_sightlines) bit for bit, sink and plain loop."""
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    from rbvfit_b200.sampler import SightlineEnsembleSampler
    w0, batch, _singles = c5b
    S, W, n, nd = batch.n_sightlines, 16, 30, batch.ndim
    p0 = _start(w0, (S, W), 3, scale=1e-3)
    ref = SightlineEnsembleSampler(W, nd, batch, seed=5)
    ref.run_mcmc(p0, n)
    for use_graph in (True, False):
        smp = SightlineParallelTemperingSampler(W, nd, batch, betas=[1.0], seed=5, use_graph=use_graph,
                                                record_log_like=True)
        smp.run_mcmc(p0, n)
        assert np.array_equal(smp.get_chain(), ref.get_chain()), use_graph
        assert np.array_equal(smp.get_log_like()[:, :, 0], ref.get_log_prob()), use_graph
        assert np.array_equal(smp.acceptance_fraction[:, 0], ref.acceptance_fraction), use_graph
        assert smp.tswap_acceptance_fraction.shape == (S, 0)


def _rel(a, b):
    return float(np.max(np.abs(a - b) / np.abs(b)))


@pytest.mark.parametrize("W", [16, 13])
def test_every_sightline_matches_its_replay(c5b, W):
    """S = 5, T = 4: every sightline equals oracle/pt_replay_sightlines.py with walker_offset = s T W driven by its
    own single-sightline likelihood -- chain, lnprob chain, counters and the device moments; with adaptation the
    ladder within 8 ulp of the replay's prediction.  The survey's half-steps evaluate S times the rows of the
    replay's, which can select another lnprob kernel: the lnprob chain is compared bit for bit where it agrees
    bitwise with the replay's and to the slice-sightline test's tolerance otherwise (the moments likewise), and the
    test prints which held."""
    from oracle import pt_replay_sightlines as prs
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    w0, batch, singles = c5b
    S, T, n, nd = batch.n_sightlines, 4, 40, batch.ndim
    p0 = _start(w0, (S, T, W), 7 + W)
    held = []
    for adapt in (False, True):
        smp = SightlineParallelTemperingSampler(W, nd, batch, betas=BETAS4, seed=21, record_log_like=True,
                                                adaptation_time=5.0)
        smp.run_mcmc(p0, n, adapt=adapt, n_record=2)
        for s in range(S):
            like = singles[s]
            lp = like.lnprob(p0[s].reshape(-1, nd)).reshape(T, W)
            r = prs.run(like.lnprob, p0[s], lp, BETAS4, n, smp._seed, n_record=2, adapt=adapt, tau=5.0,
                       walker_offset=s * T * W, beta_history_device=smp.beta_history[:, s] if adapt else None)
            chain = np.stack([smp.get_chain(temp=t, sightline=s) for t in range(2)], axis=1)
            ll = smp.get_log_like(sightline=s)
            bitwise = np.array_equal(ll, r["lnp_chain"])
            held.append((bitwise, np.array_equal(chain, r["chain"]), _rel(ll, r["lnp_chain"])))
            assert np.allclose(chain, r["chain"], rtol=0, atol=1e-9), (adapt, s)
            assert _rel(ll, r["lnp_chain"]) <= 1e-9, (adapt, s)
            if not adapt:
                if bitwise:
                    assert np.array_equal(smp.ti_moments[s], r["ti"]), s
                else:
                    assert np.allclose(smp.ti_moments[s], r["ti"], rtol=1e-9, atol=0), s
            assert np.array_equal(np.rint(smp.acceptance_fraction[s] * n).astype(int), r["n_accepted"]), (adapt, s)
            assert np.array_equal(np.rint(smp.tswap_acceptance_fraction[s] * n * W).astype(int), r["n_swaps"])
            if adapt:
                np.testing.assert_array_max_ulp(r["beta_pred"], smp.beta_history[:, s], maxulp=8)
                np.testing.assert_array_max_ulp(r["betas"], smp.betas[s], maxulp=8)
            else:
                assert np.array_equal(smp.beta_history[:, s], np.tile(BETAS4, (n, 1)))
    print(f"\nW = {W}: lnprob chain bitwise on {sum(h[0] for h in held)} of {len(held)} (sightline, run) pairs, "
          f"chain bitwise on {sum(h[1] for h in held)}; largest relative lnprob difference "
          f"{max(h[2] for h in held):.2e}; survey kernel {batch.engine.last_kernel}, one sightline "
          f"{singles[0].engine.last_kernel}")


def test_sightlines_are_independent(c5b):
    """Perturbing sightline 3's start leaves every other sightline's chain, lnprob chain and moments bit-identical."""
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    w0, batch, _singles = c5b
    S, T, W, n, nd = batch.n_sightlines, 4, 16, 30, batch.ndim
    p0 = _start(w0, (S, T, W), 8)
    runs = []
    for p in (p0, np.where(np.arange(S)[:, None, None, None] == 3, _start(w0, (S, T, W), 9), p0)):
        smp = SightlineParallelTemperingSampler(W, nd, batch, betas=BETAS4, seed=2, record_log_like=True)
        smp.run_mcmc(p, n)
        runs.append(smp)
    a, b = runs
    keep = [0, 1, 2, 4]
    assert np.array_equal(a.get_chain()[:, keep], b.get_chain()[:, keep])
    assert np.array_equal(a.get_log_like()[:, keep], b.get_log_like()[:, keep])
    assert np.array_equal(a.ti_moments[keep], b.ti_moments[keep])
    assert not np.array_equal(a.get_chain()[:, 3], b.get_chain()[:, 3])
    assert not np.array_equal(a.ti_moments[3], b.ti_moments[3])


def test_continuation(c5b):
    """run(30) + run(None, 25) equals run(55): chains, lnprob chains, counters, and the moments bitwise."""
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    w0, batch, _singles = c5b
    S, T, W, nd = batch.n_sightlines, 3, 16, batch.ndim
    p0 = _start(w0, (S, T, W), 6)
    kw = dict(betas=[1.0, 0.3, 0.0], seed=3, record_log_like=True)
    one = SightlineParallelTemperingSampler(W, nd, batch, **kw)
    one.run_mcmc(p0, 55, n_record=2)
    two = SightlineParallelTemperingSampler(W, nd, batch, **kw)
    two.run_mcmc(p0, 30, n_record=2)
    two.run_mcmc(None, 25, n_record=2)
    assert np.array_equal(one.get_chain(temp=1), two.get_chain(temp=1))
    assert np.array_equal(one.get_log_like(), two.get_log_like())
    assert np.array_equal(one.tswap_acceptance_fraction, two.tswap_acceptance_fraction)
    assert np.array_equal(one.ti_moments, two.ti_moments) and two.evidence_steps == 55
    lnz1, _ = one.log_evidence_estimate()
    lnz2, _ = two.log_evidence_estimate()
    assert np.array_equal(lnz1, lnz2)
    assert one.get_last_sample()[0].shape == (S, T, W, nd)


def test_moments_give_the_chain_evidence(c5b):
    """The default ladder: lnZ from the device moments is within 1e-8 nats of log_evidence on the recorded lnprob
    chain, for every sightline."""
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler, default_betas, log_evidence
    w0, batch, _singles = c5b
    S, W, nd = batch.n_sightlines, 16, batch.ndim
    betas = default_betas(nd)
    smp = SightlineParallelTemperingSampler(W, nd, batch, betas=betas, seed=4, record_log_like=True)
    smp.run_mcmc(_start(w0, (S, W), 5, scale=1e-3), 200)
    lnz, dlnz = smp.log_evidence_estimate()
    worst = 0.0
    for s in range(S):
        ref = log_evidence(betas, smp.get_log_like(sightline=s))
        worst = max(worst, abs(lnz[s] - ref[0]), abs(dlnz[s] - ref[1]))
    print(f"\nT = {len(betas)}: max |lnZ(moments) - lnZ(chain)| = {worst:.3e} nats")
    assert worst <= 1e-8


def _mgii_survey(indices, two_comp):
    """Sightlines at C5b's redshifts whose spectra were drawn from two components (C5b's truth) or from one
    ([13.4], [25], [0]); returns (sightline dicts for a 1-component and a 2-component batch, their bounds)."""
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    one, two = [], []
    truth1 = np.array([13.4, 25.0, 0.0])
    for s, gen2 in zip(indices, two_comp):
        w = wl.c5b_sightline(s)
        z = w["systems"][0][0]
        models = {}
        for C_ in (1, 2):
            cfg = FitConfiguration()
            cfg.add_system(z=z, ion="MgII", transitions=[2796.3, 2803.5], components=C_)
            models[C_] = GpuVoigtModel(cfg, FWHM="6.5")
        wave = w["instruments"]["COS"]["wave"]
        truth = w["theta_true"] if gen2 else truth1
        flux = models[2 if gen2 else 1].compile().model_flux(truth, wave)
        flux = flux + wl.SIGMA * np.random.default_rng(w["seed"]).standard_normal(wave.size)
        sp = dict(wave=wave, flux=flux, error=np.full(wave.size, wl.SIGMA))
        one.append(dict(model=models[1], **sp))
        two.append(dict(model=models[2], **sp))
    w0 = wl.c5b_sightline(indices[0])
    return one, two, wl.default_bounds([14.6], [40.0], [0.0]), (w0["lb"], w0["ub"])


def _survey_evidence(batch, theta0, lb, ub, seed, W=40, burn=700, n=1300):
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler, default_betas
    fit = batch.fit_quick(theta0)
    rng = np.random.default_rng(seed)
    p0 = np.clip(fit.x[:, None, :] + 1e-4 * rng.standard_normal((batch.n_sightlines, W, batch.ndim)),
                 lb + 1e-10, ub - 1e-10)
    smp = SightlineParallelTemperingSampler(W, batch.ndim, batch, betas=default_betas(batch.ndim), seed=seed,
                                            record_chain=False)
    smp.run_mcmc(p0, burn, accumulate=False)
    smp.run_mcmc(None, n)
    return smp.log_evidence_estimate()


def test_model_selection_across_a_survey():
    """8 sightlines, 4 drawn from two MgII components and 4 from one: lnZ(2) - lnZ(1) > 10 on every two-component
    sightline, lnZ(1) >= lnZ(2) - 3 dlnZ on every one-component sightline (test_model_selection's criteria)."""
    from rbvfit_b200.likelihood import SightlineBatch
    gen2 = [True, False] * 4
    one, two, (lb1, ub1), (lb2, ub2) = _mgii_survey(list(range(20, 28)), gen2)
    b1, b2 = SightlineBatch(one, lb1, ub1), SightlineBatch(two, lb2, ub2)
    th1 = np.array([[14.6, 40.0, 0.0] if g else [13.4, 25.0, 0.0] for g in gen2])
    th2 = np.array([[14.25, 14.45, 42.0, 28.0, -22.0, 32.0] if g else [13.3, 12.6, 25.0, 25.0, -2.0, 8.0]
                    for g in gen2])
    z1, d1 = _survey_evidence(b1, th1, lb1, ub1, seed=1)
    z2, d2 = _survey_evidence(b2, th2, lb2, ub2, seed=2)
    for s, g in enumerate(gen2):
        print(f"\nsightline {s} ({2 if g else 1} components): lnZ(1) = {z1[s]:.2f} +- {d1[s]:.2f}, "
              f"lnZ(2) = {z2[s]:.2f} +- {d2[s]:.2f}", end="")
    print()
    for s, g in enumerate(gen2):
        if g:
            assert z2[s] - z1[s] > 10, s
        else:
            assert z1[s] >= z2[s] - 3 * max(d1[s], d2[s]), s
    b1.close()
    b2.close()


def test_nonfinite_moments_name_their_sightline(c5b):
    """A walker of sightline 2 starts far outside the bounds and accumulation runs from step 0: its moments are not
    finite, lnZ is NaN for sightline 2 only, and one warning names it."""
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    w0, batch, _singles = c5b
    S, W, nd = batch.n_sightlines, 16, batch.ndim
    p0 = _start(w0, (S, W), 12, scale=1e-3)
    p0[2, 0, 0] = w0["ub"][0] + 100.0 * (w0["ub"][0] - w0["lb"][0])
    smp = SightlineParallelTemperingSampler(W, nd, batch, betas=BETAS4, seed=6, record_chain=False)
    smp.run_mcmc(p0, 20, skip_initial_state_check=True)
    with pytest.warns(RuntimeWarning, match=r"sightlines \[2\]"):
        lnz, dlnz = smp.log_evidence_estimate()
    assert np.isnan(lnz[2]) and np.isnan(dlnz[2])
    assert np.all(np.isfinite(np.delete(lnz, 2))) and np.all(np.isfinite(np.delete(dlnz, 2)))


def test_scale_sightline_zero_is_its_single_run():
    """S = 256 (C5b's first 16 sightlines 16 times over), T = 23, W = 32 (94 208 rows per half-step, past 65 535):
    the run completes and sightline 0 equals DeviceParallelTemperingSampler on that sightline alone."""
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler, SightlineParallelTemperingSampler, \
        default_betas
    w0, batch, singles = _sightlines(list(range(16)), singles_for=[0], repeat=16)
    S, W, n, nd = 256, 32, 8, batch.ndim
    betas = default_betas(nd)
    assert len(betas) == 23 and S * len(betas) * W // 2 == 94208
    p0 = _start(w0, (S, W), 13, scale=1e-3)
    smp = SightlineParallelTemperingSampler(W, nd, batch, betas=betas, seed=17, record_log_like=True)
    smp.run_mcmc(p0, n)
    ref = DeviceParallelTemperingSampler(W, nd, singles[0], betas=betas, seed=17)
    ref.run_mcmc(p0[0], n)
    kernels = (batch.engine.last_kernel, singles[0].engine.last_kernel)
    ll, ref_ll = smp.get_log_like(sightline=0), ref.get_log_like()
    same_chain = np.array_equal(smp.get_chain(sightline=0), ref.get_chain())
    print(f"\nS = 256 sightline 0 vs one sightline: chain bitwise {same_chain}, lnprob chain bitwise "
          f"{np.array_equal(ll, ref_ll)} (largest relative difference {_rel(ll, ref_ll):.2e}); lnprob kernels "
          f"{kernels}")
    # where the two evaluate lnprob bit for bit (the same kernel) the runs are identical; else the tolerance of
    # the replay comparison
    if np.array_equal(ll, ref_ll):
        assert np.array_equal(smp.get_chain(sightline=0), ref.get_chain())
    assert np.allclose(smp.get_chain(sightline=0), ref.get_chain(), rtol=0, atol=1e-9)
    assert _rel(ll, ref_ll) <= 1e-9
    assert np.array_equal(smp.tswap_acceptance_fraction[0], ref.tswap_acceptance_fraction)
    assert np.all(np.isfinite(smp.log_evidence_estimate()[0]))
    batch.close()
    singles[0].close()


def test_launches_per_step_do_not_depend_on_sightlines_or_temperatures(c5b):
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    w0, batch5, _singles = c5b
    _w, batch1, singles1 = _sightlines([0], singles_for=[])
    per_step = {}
    for name, batch in (("S=1", batch1), ("S=5", batch5)):
        for betas in ([1.0, 0.0], [1.0, 0.6, 0.3, 0.1, 0.03, 0.0]):
            for use_graph in (True, False):
                S, T = batch.n_sightlines, len(betas)
                smp = SightlineParallelTemperingSampler(16, batch.ndim, batch, betas=betas, seed=1,
                                                        use_graph=use_graph, record_chain=False)
                smp.run_mcmc(_start(w0, (S, 16), 2, scale=1e-3), 4)
                before = batch.engine.launch_count
                smp.run_mcmc(None, 10)
                per_step[name, T, use_graph] = (batch.engine.launch_count - before) / 10
    print(f"\nlaunches per step: {per_step}")
    assert len(set(per_step.values())) == 1
    batch1.close()


def test_errors(c5b):
    import torch
    from rbvfit_b200._lib import RbvChainSink, RbvError, RbvPtControl, load
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler
    w0, batch, singles = c5b
    S, T, W, nd = batch.n_sightlines, 4, 12, batch.ndim
    p0 = _start(w0, (S, W), 8, scale=1e-3)
    smp = SightlineParallelTemperingSampler(W, nd, batch, betas=BETAS4, seed=1)
    with pytest.raises(ValueError):
        smp.run_mcmc(p0[:2], 3)                                                   # wrong start shape
    with pytest.raises(ValueError):
        smp.run_mcmc(p0[:, None].repeat(3, axis=1), 3)                            # [S, 3, W, nd] with T = 4
    with pytest.raises(ValueError, match="adapt"):
        smp.run_mcmc(p0, 3, adapt=True, accumulate=True)
    with pytest.raises(TypeError):
        SightlineParallelTemperingSampler(W, nd, singles[0])
    bad = p0.copy()
    bad[1, 0, 0] = np.nan
    with pytest.raises(ValueError):
        smp.run_mcmc(bad, 3)
    smp.run_mcmc(p0, 3, adapt=True)                                               # burn-in, then a changed ladder
    assert smp.evidence_steps == 0
    eng, dev = batch.engine, batch.engine.tdev
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        c = torch.as_tensor(np.broadcast_to(p0[:, None], (S, T, W, nd)).copy(), device=dev)
        lp = eng.lnprob_sightlines_device(c.view(-1, nd), T * W).view(S, T, W).contiguous()
        b = torch.as_tensor(np.tile(BETAS4, (S, 1)), device=dev)
        nacc = torch.zeros((S, T, W), dtype=torch.int32, device=dev)
        nsw = torch.zeros((S, T - 1), dtype=torch.int64, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        ti = torch.zeros((S, T, 3), dtype=torch.float64, device=dev)
        b[3, 2] = 0.5                                                             # not decreasing on sightline 3
        with pytest.raises(RbvError, match="sightline 3"):
            eng.pt_run_sightlines(c, lp, b, 4, 2.0, 1, 0, None, None, None, None, nacc, nsw, flag)
        b[3, 2] = 0.1
        with pytest.raises(RbvError, match="adapt"):
            eng.pt_run_sightlines(c, lp, b, 4, 2.0, 1, 0, None, None, None, ti, nacc, nsw, flag, adapt=True)
        for n_record in (0, T + 1):
            with pytest.raises(RbvError, match="n_record"):
                eng.pt_run_sightlines(c, lp, b, 4, 2.0, 1, 0, None, None, None, None, nacc, nsw, flag,
                                      n_record=n_record)
        with pytest.raises(ValueError):
            eng.pt_run_sightlines(c[:, :2], lp, b, 4, 2.0, 1, 0, None, None, None, None, nacc, nsw, flag)
        # a sink needs the graph
        lib = load()
        ring = torch.empty(2 * 4 * S * W * nd, dtype=torch.float64, device=dev)
        pin = torch.empty(2 * 4 * S * W * nd, dtype=torch.float64, pin_memory=True)
        host = np.empty((8, S, 1, W, nd))
        sink = RbvChainSink(host.ctypes.data, None, ring.data_ptr(), pin.data_ptr(), 4)
        ctl = RbvPtControl(2.0, 0, 1e4, 100.0, 0, 1)
        nbytes = C.c_size_t(0)
        assert lib.rbv_pt_workspace_bytes_sightlines(eng._h, T, W, C.byref(nbytes)) == 0
        ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=dev)

        def call(use_graph, n_ws):
            return lib.rbv_pt_run_sightlines(eng._h, c.data_ptr(), lp.data_ptr(), b.data_ptr(), T, W, 8,
                                             C.byref(ctl), 1, 0, None, None, C.byref(sink), None, None,
                                             nacc.data_ptr(), nsw.data_ptr(), flag.data_ptr(), ws.data_ptr(), n_ws,
                                             use_graph, st.cuda_stream)
        assert call(0, int(nbytes.value)) == 1 and b"use_graph" in lib.rbv_last_error()    # RBV_EINVAL
        assert call(1, int(nbytes.value) - 256) == 3                                        # RBV_ENOMEM
        assert call(1, int(nbytes.value)) == 0                # chain rows only in the ring (no lnprob host array)
        st.synchronize()
        assert np.all(np.isfinite(host))
