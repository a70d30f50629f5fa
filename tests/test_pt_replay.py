"""CPU: the numpy restatement of the device's parallel tempering (oracle/pt_replay.py) against the stretch-move
replay, against analytic posteriors and evidences, and the host logic of DeviceParallelTemperingSampler."""
from math import erf, log, sqrt

import numpy as np
import pytest

from oracle import pt_replay as pr
from oracle import stretch_replay as sr
from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler, default_betas, log_evidence

BOX = 5.0


def _gauss(d):
    """Unit Gaussian likelihood (normalised) inside the box [-5, 5]^d, -inf outside."""
    def f(x):
        x = np.atleast_2d(x)
        out = -0.5 * np.sum(x * x, axis=1) - 0.5 * d * np.log(2 * np.pi)
        out[np.any(np.abs(x) > BOX, axis=1)] = -np.inf
        return out
    return f


def _start(f, T, W, d, seed, lo=-1.0, hi=1.0):
    c = np.random.default_rng(seed).uniform(lo, hi, size=(T, W, d))
    return c, f(c.reshape(-1, d)).reshape(T, W)


def _ratio_ladder(r, beta_min):
    n = int(np.ceil(np.log(1.0 / beta_min) / np.log(r)))
    return np.append(r ** -np.arange(n + 1.0), 0.0)


@pytest.mark.parametrize("W,first_step", [(16, 0), (13, 1000)])
def test_one_temperature_is_the_stretch_replay(W, first_step):
    d = 3
    f = _gauss(d)
    c, lp = _start(f, 1, W, d, 1)
    ch, lps, na = sr.run(f, c[0], lp[0], 30, seed=99, first_step=first_step)
    r = pr.run(f, c, lp, [1.0], 30, seed=99, first_step=first_step, block=7)
    assert np.array_equal(ch, r["chain"][:, 0])
    assert np.array_equal(lps, r["lnp_chain"][:, 0])
    assert np.array_equal(na, r["n_accepted"][0])


def test_vectorised_philox_is_stretch_replays():
    steps, walkers = np.array([0, 5, 2 ** 33 + 7]), np.array([0, 17, 0xFFFFFFFF])
    v = pr.philox_vec(0x123456789ABCDEF, steps, walkers, 6)
    for k in range(3):
        assert tuple(int(x[k]) for x in v) == sr._rand(0x123456789ABCDEF, steps[k], walkers[k], 6)


def test_continuation_and_blocks():
    d, T, W = 2, 4, 10
    f = _gauss(d)
    c, lp = _start(f, T, W, d, 2)
    betas = _ratio_ladder(2.0, 0.1)[:T]
    full = pr.run(f, c, lp, betas, 20, seed=5, n_record=T)
    a = pr.run(f, c, lp, betas, 8, seed=5, n_record=T, block=3)
    b = pr.run(f, a["coords"], a["lnp"], betas, 12, seed=5, first_step=8, n_record=T)
    assert np.array_equal(full["chain"], np.concatenate([a["chain"], b["chain"]]))
    assert np.array_equal(full["n_swaps"], a["n_swaps"] + b["n_swaps"])


def test_walker_outside_the_bounds_moves_at_every_temperature():
    """A walker that starts at -inf accepts any finite proposal, at beta = 0 too (beta (new - old) would be NaN)."""
    d, W = 2, 8
    f = _gauss(d)
    c, lp = _start(f, 2, W, d, 3)
    c[:, 0] = 7.0                     # outside the box
    lp = f(c.reshape(-1, d)).reshape(2, W)
    r = pr.run(f, c, lp, [1.0, 0.0], 60, seed=11, n_record=2)
    assert np.all(np.isfinite(r["lnp_chain"][-1]))


@pytest.mark.parametrize("d", [3, 6])
def test_gaussian_moments_and_evidence(d):
    """Cold-chain moments; lnZ at a ratio-1.5 ladder within 0.1 nats of the exact value (erf); at the default
    ladder the reported dlnZ covers the true error."""
    f = _gauss(d)
    exact = d * log(erf(BOX / sqrt(2.0)) / (2.0 * BOX))
    W, n, burn = 40, 2000, 500
    for betas, check in ((_ratio_ladder(1.5, 1e-3), "lnz"), (default_betas(d), "dlnz")):
        T = len(betas)
        c, lp = _start(f, T, W, d, d)
        r = pr.run(f, c, lp, betas, n, seed=100 + d)
        cold = r["chain"][burn:, 0].reshape(-1, d)
        assert np.all(np.abs(cold.mean(axis=0)) < 0.06), cold.mean(axis=0)
        assert np.all(np.abs(cold.var(axis=0) - 1.0) < 0.08), cold.var(axis=0)
        lnz, dlnz = log_evidence(betas, r["lnp_chain"][burn:])
        if check == "lnz":
            assert abs(lnz - exact) < 0.1, (lnz, exact)
        else:
            assert dlnz >= abs(lnz - exact), (lnz, dlnz, exact)


def test_two_modes_mix_only_with_tempering():
    """Weights 0.3 / 0.7 at x0 = -4 / +4 (sigma 0.5): from a start in the light mode the cold PT chain finds both in
    their proportions; one ensemble from the same start never leaves its mode."""
    d, W = 2, 32
    s2 = 0.25

    def f(x):
        x = np.atleast_2d(x)
        r1 = np.sum((x - np.array([-4.0, 0.0])) ** 2, axis=1)
        r2 = np.sum((x - np.array([4.0, 0.0])) ** 2, axis=1)
        out = np.logaddexp(np.log(0.3) - 0.5 * r1 / s2, np.log(0.7) - 0.5 * r2 / s2)
        out[np.any(np.abs(x) > 10.0, axis=1)] = -np.inf
        return out

    betas = _ratio_ladder(1.5, 1e-3)
    T = len(betas)
    c = np.random.default_rng(4).normal(size=(T, W, d)) * 0.3 + np.array([-4.0, 0.0])
    lp = f(c.reshape(-1, d)).reshape(T, W)
    r = pr.run(f, c, lp, betas, 2000, seed=21)
    frac = np.mean(r["chain"][500:, 0, :, 0] > 0)
    assert abs(frac - 0.7) < 0.1, frac
    one = pr.run(f, c[:1], lp[:1], [1.0], 2000, seed=21)
    assert np.all(one["chain"][:, 0, :, 0] < 0)


def test_adaptation_evens_out_the_swap_acceptance():
    d, W, n = 3, 32, 1500
    f = _gauss(d)
    betas = np.array([1.0, 0.9, 0.8, 0.1, 0.05, 0.04, 0.0])     # uneven: some pairs almost always swap, some never
    T = len(betas)
    c, lp = _start(f, T, W, d, 5)
    ad = pr.run(f, c, lp, betas, n, seed=8, adapt=True, tau=10.0)
    assert np.all(np.diff(ad["betas"]) < 0) and ad["betas"][0] == 1.0 and ad["betas"][-1] == 0.0
    before = pr.run(f, c, lp, betas, 500, seed=9)["n_swaps"] / (500 * W)
    after = pr.run(f, ad["coords"], ad["lnp"], ad["betas"], 500, seed=9)["n_swaps"] / (500 * W)
    assert np.std(after) < 0.5 * np.std(before), (before, after)


def test_log_evidence_closed_forms():
    betas = np.array([1.0, 0.5, 0.25])
    logl = np.full((5, 3, 4), -2.5)
    assert log_evidence(betas, logl) == (-2.5, 0.0)                 # constant lnL: lnZ = lnL, beta_min > 0 closed
    # <lnL>_beta linear in beta, Var constant: the trapezoid is exact and the correction vanishes
    b = np.array([1.0, 0.6, 0.3, 0.0])
    x = np.array([[-1.0, 1.0]])                                      # mean 0, variance 1 around E(beta)
    logl = (3.0 * b - 2.0)[None, :, None] + x[:, None, :]
    lnz, dlnz = log_evidence(b, logl)
    assert lnz == pytest.approx(1.5 - 2.0, abs=1e-14) and dlnz == pytest.approx(0.0, abs=1e-14)
    with pytest.raises(ValueError):
        log_evidence(b, logl[:, :3])


def test_default_ladder():
    for d in (1, 3, 6, 30):
        b = default_betas(d)
        r = 1.0 + 2.0 * np.sqrt(np.log(4.0) / d)
        assert b[0] == 1.0 and b[-1] == 0.0 and b[-2] < 1e-6 <= b[-3]
        assert np.allclose(b[:-2] / b[1:-1], r)


def test_pt_sampler_accessors_without_device():
    """Bookkeeping of DeviceParallelTemperingSampler on a hand-filled history -- no device involved."""

    class _Like:                     # what the sampler reads from a GpuLikelihood before sampling
        engine, ndim = object(), 2

    T, W, nd, n = 3, 4, 2, 10
    betas = [1.0, 0.5, 0.0]
    smp = DeviceParallelTemperingSampler(W, nd, _Like(), betas=betas, seed=1)
    assert smp.ntemps == T and smp.acceptance_fraction.shape == (T, W) and smp.tswap_acceptance_fraction.shape == (2,)
    assert smp.get_log_like().shape == (0, T, W)
    chain = np.arange(n * 2 * W * nd, dtype=float).reshape(n, 2, W, nd)
    logl = -np.arange(n * T * W, dtype=float).reshape(n, T, W)
    bh = np.tile(betas, (n, 1))
    smp._chunks = [(chain[:4], logl[:4], bh[:4], np.ones(4, bool)), (chain[4:], logl[4:], bh[4:], np.zeros(6, bool))]
    smp.n_record, smp.iteration = 2, n
    smp._accepted[:] = np.arange(T * W).reshape(T, W)
    smp._swaps[:] = [20, 8]
    assert np.array_equal(smp.get_chain(discard=2, thin=2, temp=1), chain[3::2, 1])
    assert np.array_equal(smp.get_chain(flat=True), chain[:, 0].reshape(-1, nd))
    assert np.array_equal(smp.get_log_like(discard=1), logl[1:])
    assert smp.get_log_like(flat=True).shape == (T, n * W)
    assert np.array_equal(smp.beta_history, bh)
    assert np.allclose(smp.tswap_acceptance_fraction, [20 / (n * W), 8 / (n * W)])
    v = smp.cold()
    assert (v.nwalkers, v.ndim, v.iteration) == (W, nd, n)
    assert np.array_equal(v.get_chain(discard=3, flat=True), chain[3:, 0].reshape(-1, nd))
    assert np.array_equal(v.get_log_prob(), logl[:, 0])
    assert v.chain.shape == (W, n, nd) and v.flatchain.shape == (n * W, nd) and v.lnprobability.shape == (W, n)
    assert np.array_equal(v.acceptance_fraction, np.arange(W) / n)
    assert v.get_autocorr_time(quiet=True).shape == (nd,)
    assert smp.log_evidence_estimate(discard=4) == log_evidence(betas, logl[4:])
    with pytest.raises(ValueError, match="adapt"):
        smp.log_evidence_estimate(discard=3)                        # a kept step ran with adaptation
    with pytest.raises(ValueError):
        smp.get_chain(temp=3)                                        # no such temperature
    with pytest.raises(ValueError):
        smp.get_chain(temp=2)                                        # not recorded
    for bad in ([0.9, 0.5], [1.0, 0.5, 0.5], [1.0, 0.5, -0.1], [[1.0]]):
        with pytest.raises(ValueError):
            DeviceParallelTemperingSampler(W, nd, _Like(), betas=bad)
    with pytest.raises(ValueError):
        DeviceParallelTemperingSampler(W, nd + 1, _Like())
    with pytest.raises(TypeError):
        DeviceParallelTemperingSampler(W, nd, object())
