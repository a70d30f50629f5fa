"""Survey-mode ensemble slice sampler (rbv_slice_run_sightlines, SightlineEnsembleSliceSampler): one zeus ensemble per
sightline of a SightlineBatch, all advancing in lockstep on the device."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _sightlines(indices):
    """C5b sightlines (C1's structure, each at its own redshift) as a SightlineBatch plus one single-sightline
    GpuLikelihood per sightline."""
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
    sight, singles = [], []
    for s in indices:
        w = wl.c5b_sightline(s)
        cfg = FitConfiguration()
        for (z, ion, trans, comps) in w["systems"]:
            cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        m = GpuVoigtModel(cfg, FWHM="6.5")
        c = m.compile()
        sp = wl.make_spectra(w, lambda n, th, wave: c.model_flux(th, wave))["COS"]
        sight.append(dict(model=m, **sp))
        singles.append(GpuLikelihood({"COS": dict(model=m, **sp)}, w["lb"], w["ub"]))
    w0 = wl.c5b_sightline(indices[0])
    return w0, SightlineBatch(sight, w0["lb"], w0["ub"]), singles


@pytest.fixture(scope="module")
def c5b():
    return _sightlines(list(range(5)))


def _start(w0, S, W, seed):
    rng = np.random.default_rng(seed)
    nd = len(w0["theta_true"])
    return np.clip(w0["theta_true"] + 1e-3 * rng.standard_normal((S, W, nd)), w0["lb"], w0["ub"])


def _counters(s):
    return (s.mu.tolist(), s.tune.tolist(), s.ncall.tolist(), s.nexp.tolist(), s.ncon.tolist())


def test_slice_sightlines_match_per_sightline_replays(c5b):
    """Every sightline's chain, mu trajectory and counters equal the numpy replay of ITS ensemble driven by its own
    single-sightline likelihood (random streams offset by e W); a half-step launches as many batches as its slowest
    sightline needs."""
    from oracle import slice_replay_sightlines as sl
    from rbvfit_b200.slice_sampler import SightlineEnsembleSliceSampler
    w0, batch, singles = c5b
    S, nd = batch.n_sightlines, batch.ndim
    for W, nsteps in ((12, 40), (16, 30)):
        p0 = _start(w0, S, W, 12 + W)
        smp = SightlineEnsembleSliceSampler(W, nd, batch, seed=77, depth=1)
        smp.run_mcmc(p0, nsteps)
        chain, lps = smp.get_chain(), smp.get_log_prob()
        assert chain.shape == (nsteps, S, W, nd) and lps.shape == (nsteps, S, W)
        per_half = []
        for e in range(S):
            like = singles[e]
            ref = sl.run(like.lnprob, p0[e], like.lnprob(p0[e]), nsteps, smp._seed, walker_offset=e * W)
            assert np.allclose(chain[:, e], ref["chain"], rtol=0, atol=1e-9), e
            assert np.max(np.abs(lps[:, e] - ref["lnp_chain"]) / np.abs(ref["lnp_chain"])) <= 1e-9, e
            assert (smp.nexp[e], smp.ncon[e], smp.ncall[e]) == (ref["nexp"], ref["ncon"], W + ref["ncall"]), e
            assert smp.mu[e] == ref["mu"] and smp.tune[e] == ref["tune"], e
            assert np.array_equal(smp.mus[:, e], ref["mus"]), e
            assert ref["batches_per_half"].sum() == ref["nbatches"]
            per_half.append(ref["batches_per_half"])
        assert smp.nbatches == 1 + int(np.max(per_half, axis=0).sum())


def test_slice_sightlines_drivers_and_depth(c5b):
    """Depth 2 in graph mode and depths 1 and 2 host-polled give the chains, lnprob chains, mu and counters of depth 1
    in graph mode bit for bit; depth 2 needs fewer launches, the polled loop exactly one masked launch per half-step
    more."""
    from rbvfit_b200.slice_sampler import SightlineEnsembleSliceSampler
    w0, batch, singles = c5b
    S, nd, W, nsteps = batch.n_sightlines, batch.ndim, 14, 25
    p0 = _start(w0, S, W, 4)
    runs = {}
    for graph in (True, False):
        for depth in (1, 2):
            s = SightlineEnsembleSliceSampler(W, nd, batch, seed=9, depth=depth, use_graph=graph)
            s.run_mcmc(p0, nsteps)
            runs[graph, depth] = s
    ref = runs[True, 1]
    for key, s in runs.items():
        assert np.array_equal(s.get_chain(), ref.get_chain()), key
        assert np.array_equal(s.get_log_prob(), ref.get_log_prob()), key
        assert np.array_equal(s.mus, ref.mus) and _counters(s) == _counters(ref), key
    assert runs[True, 2].nbatches < runs[True, 1].nbatches
    assert runs[False, 2].nbatches < runs[False, 1].nbatches
    for depth in (1, 2):
        assert runs[False, depth].nbatches == runs[True, depth].nbatches + 2 * nsteps


def test_slice_sightline_zero_equals_single_ensemble_and_sightlines_are_independent(c5b):
    """Sightline 0 reproduces DeviceEnsembleSliceSampler on that sightline alone; the first three sightlines of the
    batch equal a three-sightline batch of the same spectra; a sightline that is much harder to sample changes the
    number of launches but not the other sightlines' chains."""
    from rbvfit_b200.slice_sampler import DeviceEnsembleSliceSampler, SightlineEnsembleSliceSampler
    w0, batch, singles = c5b
    S, nd, W, nsteps = batch.n_sightlines, batch.ndim, 16, 30
    p0 = _start(w0, S, W, 21)
    smp = SightlineEnsembleSliceSampler(W, nd, batch, seed=31)
    smp.run_mcmc(p0, nsteps)
    chain = smp.get_chain()
    one = DeviceEnsembleSliceSampler(W, nd, singles[0], seed=31)
    one.run_mcmc(p0[0], nsteps)
    assert np.allclose(one.get_chain(), chain[:, 0], rtol=0, atol=1e-9)
    assert np.array_equal(np.asarray(one.mus), smp.mus[:, 0])
    assert (one.mu, one.tune, one.ncall, one.nexp, one.ncon) == (smp.mu[0], smp.tune[0], smp.ncall[0], smp.nexp[0],
                                                                 smp.ncon[0])
    _, batch3, _ = _sightlines([0, 1, 2])
    three = SightlineEnsembleSliceSampler(W, nd, batch3, seed=31)
    three.run_mcmc(p0[:3], nsteps)
    assert np.allclose(three.get_chain(), chain[:, :3], rtol=0, atol=1e-9)
    assert _counters(three) == tuple(v[:3] for v in _counters(smp))
    assert np.array_equal(three.mus, smp.mus[:, :3])
    # sightline 4 starts spread over the whole prior box
    hard0 = p0.copy()
    rng = np.random.default_rng(5)
    hard0[4] = w0["lb"] + (w0["ub"] - w0["lb"]) * rng.uniform(0.05, 0.95, size=(W, nd))
    hard = SightlineEnsembleSliceSampler(W, nd, batch, seed=31)
    hard.run_mcmc(hard0, nsteps)
    assert hard.nbatches != smp.nbatches
    assert np.allclose(hard.get_chain()[:, :4], chain[:, :4], rtol=0, atol=1e-9)
    assert _counters(hard)[2:] != _counters(smp)[2:]
    assert tuple(v[:4] for v in _counters(hard)) == tuple(v[:4] for v in _counters(smp))
    batch3.close()


def test_slice_sightlines_bookkeeping_and_continuation(c5b):
    """The recorded lnprob of every stored position equals the batch likelihood recomputed for it, walkers stay in
    the prior box and move every step, run(30) + run(None, 20) equals run(50) bit for bit, another seed gives another
    chain, and the per-sightline view has zeus's accessors."""
    from rbvfit_b200.slice_sampler import SightlineEnsembleSliceSampler
    w0, batch, singles = c5b
    S, nd, W = batch.n_sightlines, batch.ndim, 12
    p0 = _start(w0, S, W, 3)
    a = SightlineEnsembleSliceSampler(W, nd, batch, seed=5)
    a.run_mcmc(p0, 50)
    chain, lps = a.get_chain(), a.get_log_prob()
    for step in (0, 17, 49):
        got = batch.lnprob(chain[step])
        assert np.max(np.abs(got - lps[step]) / np.abs(got)) <= 1e-12
    assert np.all(chain >= w0["lb"]) and np.all(chain <= w0["ub"]) and np.all(np.isfinite(lps))
    assert np.all(np.any(chain[1:] != chain[:-1], axis=3)) and a.acceptance_fraction.shape == (S, W)
    assert a.acceptance_fraction.min() > 0.95 and np.all(a.efficiency > 0.05)
    b = SightlineEnsembleSliceSampler(W, nd, batch, seed=5)
    b.run_mcmc(p0, 30)
    b.run_mcmc(None, 20)
    assert np.array_equal(b.get_chain(), chain) and np.array_equal(b.get_log_prob(), lps)
    assert np.array_equal(b.mus, a.mus) and _counters(b) == _counters(a)
    c = SightlineEnsembleSliceSampler(W, nd, batch, seed=6)
    c.run_mcmc(p0, 10)
    assert not np.array_equal(c.get_chain(), chain[:10])
    # zeus's conventions: arr[discard::thin]; flat per sightline
    assert np.array_equal(a.get_chain(discard=10, thin=3), chain[10::3])
    assert a.get_chain(flat=True, discard=10).shape == (S, 40 * W, nd)
    assert a.get_log_prob(flat=True, sightline=1).shape == (50 * W,)
    assert a.get_last_sample()[0].shape == (S, W, nd) and a.mus.shape == (50, S)
    v = a.sightline(2)
    assert np.array_equal(v.get_chain(), chain[:, 2]) and v.chain.shape == (50, W, nd)
    assert v.get_chain(flat=True, discard=5).shape == (45 * W, nd) and v.get_log_prob().shape == (50, W)
    assert v.acceptance_fraction.shape == (W,) and v.efficiency == a.efficiency[2] and v.mu == a.mu[2]
    assert np.array_equal(v.mus, a.mus[:, 2]) and (v.ncall, v.nexp, v.ncon) == (a.ncall[2], a.nexp[2], a.ncon[2])
    assert v.get_autocorr_time(quiet=True).shape == (nd,) and v.get_last_sample()[1].shape == (W,)
    with pytest.raises(IndexError):
        a.sightline(S)


def test_slice_sightlines_posterior_brackets_truth():
    """24 walkers x 250 steps per sightline: the 0.5-99.5 % interval of every parameter's post-burn-in samples
    brackets the truth of that sightline, and the autocorrelation time is finite."""
    from rbvfit_b200 import workloads as wl
    from rbvfit_b200.slice_sampler import SightlineEnsembleSliceSampler
    w0, batch, singles = _sightlines([10, 11, 12])
    S, nd, W = batch.n_sightlines, batch.ndim, 24
    p0 = _start(w0, S, W, 17)
    smp = SightlineEnsembleSliceSampler(W, nd, batch, seed=13)
    smp.run_mcmc(p0, 250)
    samples = smp.get_chain(flat=True, discard=100)
    assert samples.shape == (S, 150 * W, nd)
    for e, idx in enumerate((10, 11, 12)):
        truth = wl.c5b_sightline(idx)["theta_true"]
        lo, hi = np.percentile(samples[e], [0.5, 99.5], axis=0)
        assert np.all(lo < truth) and np.all(truth < hi), (e, lo, hi, truth)
        tau = smp.sightline(e).get_autocorr_time(quiet=True)
        assert tau.shape == (nd,) and np.all(np.isfinite(tau))
    batch.close()
    for like in singles:
        like.close()


def test_slice_sightlines_errors(c5b):
    import torch
    from rbvfit_b200._lib import RbvError, RbvSliceTuning, check, load
    from rbvfit_b200.slice_sampler import SightlineEnsembleSliceSampler
    w0, batch, singles = c5b
    S, nd, W = batch.n_sightlines, batch.ndim, 12
    p0 = _start(w0, S, W, 8)
    with pytest.raises(ValueError):
        SightlineEnsembleSliceSampler(W, nd, batch).run_mcmc(p0[:2], 3)          # wrong start shape
    with pytest.raises(ValueError):
        SightlineEnsembleSliceSampler(13, nd, batch)                            # odd
    with pytest.raises(ValueError):
        SightlineEnsembleSliceSampler(10, nd, batch)                            # fewer than 2 ndim
    with pytest.raises(TypeError):
        SightlineEnsembleSliceSampler(W, nd, singles[0])
    bad = p0.copy()
    bad[3, 0, 0] = w0["ub"][0] + 1.0
    with pytest.raises(ValueError):
        SightlineEnsembleSliceSampler(W, nd, batch, seed=1).run_mcmc(bad, 3)
    for graph in (True, False):
        with pytest.raises(RbvError, match=r"status 4.*maxiter"):
            SightlineEnsembleSliceSampler(W, nd, batch, seed=1, maxiter=1, use_graph=graph).run_mcmc(p0, 2)
    # the C entry point: workspace too small -> RBV_ENOMEM, non-positive mu -> RBV_EINVAL
    lib, eng = load(), batch.engine
    nbytes = C.c_size_t(0)
    check(lib.rbv_slice_workspace_bytes_sightlines(eng._h, W, C.byref(nbytes)))
    dev = eng.tdev
    coords = torch.as_tensor(p0, device=dev)
    lnp = torch.as_tensor(batch.lnprob(p0), device=dev)
    mu = torch.ones(S, dtype=torch.float64, device=dev)
    tg = torch.zeros((S, 2), dtype=torch.int32, device=dev)
    tot = torch.zeros((S, 3), dtype=torch.int64, device=dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=dev)
    tuning = RbvSliceTuning(tolerance=0.05, patience=5, maxsteps=10000, maxiter=10000, depth=2)
    st = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()

    def call(mu_t, n_ws):
        return lib.rbv_slice_run_sightlines(eng._h, coords.data_ptr(), lnp.data_ptr(), W, 2, C.byref(tuning),
                                            mu_t.data_ptr(), tg.data_ptr(), tot.data_ptr(), 3, 0, None, None, None,
                                            flag.data_ptr(), ws.data_ptr(), n_ws, 1, st.cuda_stream)
    assert call(mu, int(nbytes.value) - 256) == 3                               # RBV_ENOMEM
    mu[2] = 0.0
    torch.cuda.synchronize()
    assert call(mu, int(nbytes.value)) == 1                                     # RBV_EINVAL
    assert b"mu" in lib.rbv_last_error()
    mu[2] = 1.0
    torch.cuda.synchronize()
    assert call(mu, int(nbytes.value)) == 0 and int(tot[:, 2].min()) > 0 and tuning.n_batches >= 4
