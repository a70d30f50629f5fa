"""CPU: survey-mode parallel tempering without a device -- the replay's walker offset, the moment accumulator the
device restates, the evidence from moments, and the host-side checks of SightlineParallelTemperingSampler."""
import numpy as np
import pytest

from oracle import pt_replay as pr
from oracle import pt_replay_sightlines as prs
from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler, evidence_from_moments, log_evidence

BOX = 5.0


def _gauss(d):
    def f(x):
        x = np.atleast_2d(x)
        out = -0.5 * np.sum(x * x, axis=1) - 0.5 * d * np.log(2 * np.pi)
        out[np.any(np.abs(x) > BOX, axis=1)] = -np.inf
        return out
    return f


def _start(f, T, W, d, seed):
    c = np.random.default_rng(seed).uniform(-1.0, 1.0, size=(T, W, d))
    return c, f(c.reshape(-1, d)).reshape(T, W)


@pytest.mark.parametrize("W", [16, 13])
def test_offset_zero_is_the_replay_and_an_offset_changes_the_draws(W):
    """walker_offset=0 reproduces oracle/pt_replay.run bit for bit (chain, lnprob, counters, ladder with
    adaptation); a survey sightline's offset s T W gives other draws."""
    d, T, n = 3, 4, 25
    f = _gauss(d)
    c, lp = _start(f, T, W, d, W)
    betas = [1.0, 0.4, 0.1, 0.0]
    for adapt in (False, True):
        ref = pr.run(f, c, lp, betas, n, seed=7, n_record=2, adapt=adapt, tau=5.0)
        got = prs.run(f, c, lp, betas, n, seed=7, n_record=2, adapt=adapt, tau=5.0, walker_offset=0)
        for k in ("chain", "lnp_chain", "n_accepted", "n_swaps", "beta_history", "betas", "coords", "lnp"):
            assert np.array_equal(ref[k], got[k]), k
    other = prs.run(f, c, lp, betas, n, seed=7, n_record=2, walker_offset=3 * T * W)
    assert not np.array_equal(other["chain"], ref["chain"])
    assert not np.array_equal(other["n_swaps"], ref["n_swaps"])
    # the draws are those of the shifted counters
    h0, sw0 = prs._draws(7, np.arange(3), T, W, 0)
    h1, sw1 = prs._draws(7, np.arange(3), 1, W, 2 * W)
    assert np.array_equal(h0[0][2][:, 2], h1[0][2][:, 0])       # stretch uniforms of temperature 2 = ensemble 2


def test_merge_moments_matches_numpy_mean_and_var():
    """Blocks of W values merged one after another equal np.mean / np.var of all of them: values near +-5e3 with a
    spread of a few units, as lnL of a survey sightline."""
    rng = np.random.default_rng(3)
    for centre in (-5e3, 5e3):
        for W in (2, 13, 32):
            x = centre + 3.0 * rng.standard_normal((400, 5, W))       # [steps, T, W]
            mom = np.zeros((5, 3))
            for step in x:
                mom = prs.merge_moments(mom, step)
            flat = np.swapaxes(x, 0, 1).reshape(5, -1)
            assert np.array_equal(mom[:, 0], np.full(5, 400.0 * W))
            assert np.max(np.abs(mom[:, 1] / flat.mean(axis=1) - 1)) <= 1e-13
            assert np.max(np.abs((mom[:, 2] / mom[:, 0]) / flat.var(axis=1) - 1)) <= 1e-10


def test_merge_moments_first_block_is_exact_and_nonfinite_propagates():
    x = np.array([[1.5, -2.25, 7.0, 0.125]])
    m = prs.merge_moments(np.zeros((1, 3)), x)
    total = ((1.5 + -2.25) + 7.0) + 0.125
    mean = total / 4.0
    q = sum((v - mean) * (v - mean) for v in x[0])
    assert m[0, 0] == 4.0 and m[0, 1] == mean and m[0, 2] == q
    bad = prs.merge_moments(m, np.array([[1.0, -np.inf, 2.0, 3.0]]))
    assert not np.all(np.isfinite(bad))
    assert not np.all(np.isfinite(prs.merge_moments(bad, x)))


def test_evidence_from_moments_is_log_evidence():
    rng = np.random.default_rng(1)
    for betas in ([1.0, 0.5, 0.2, 0.0], [1.0, 0.6, 0.3, 0.1, 0.02], [1.0]):
        T = len(betas)
        logl = -100.0 + 5 * np.arange(T)[None, :, None] + rng.standard_normal((50, T, 8))
        x = np.swapaxes(logl, 0, 1).reshape(T, -1)
        assert evidence_from_moments(betas, x.mean(axis=1), x.var(axis=1)) == log_evidence(betas, logl)
    with pytest.raises(ValueError):
        evidence_from_moments([1.0, 0.5], [0.0], [1.0, 1.0])


def test_replay_moments_give_the_chain_evidence():
    d, W = 2, 10
    f = _gauss(d)
    betas = np.array([1.0, 0.3, 0.05, 0.0])
    c, lp = _start(f, 4, W, d, 9)
    r = prs.run(f, c, lp, betas, 200, seed=4)
    E, V = r["ti"][:, 1], r["ti"][:, 2] / r["ti"][:, 0]
    a, b = evidence_from_moments(betas, E, V), log_evidence(betas, r["lnp_chain"])
    assert abs(a[0] - b[0]) < 1e-10 and abs(a[1] - b[1]) < 1e-10


class _Batch:                        # what the sampler reads from a SightlineBatch before sampling
    engine, ndim, n_sightlines = object(), 2, 3


def test_sightline_sampler_host_checks():
    S, W = 3, 6
    smp = SightlineParallelTemperingSampler(W, 2, _Batch(), betas=[1.0, 0.5, 0.0])
    assert smp.ntemps == 3 and smp.betas.shape == (S, 3) and np.all(smp.betas == [1.0, 0.5, 0.0])
    assert smp.acceptance_fraction.shape == (S, 3, W) and smp.tswap_acceptance_fraction.shape == (S, 2)
    assert smp.evidence_steps == 0 and smp.ti_moments.shape == (S, 3, 3)
    ladders = np.array([[1.0, 0.5, 0.0], [1.0, 0.3, 0.0], [1.0, 0.6, 0.1]])
    assert np.array_equal(SightlineParallelTemperingSampler(W, 2, _Batch(), betas=ladders).betas, ladders)
    assert SightlineParallelTemperingSampler(W, 2, _Batch()).ntemps > 10            # default ladder
    bad = ladders.copy()
    bad[1, 2] = 0.4
    with pytest.raises(ValueError, match="sightline 1"):
        SightlineParallelTemperingSampler(W, 2, _Batch(), betas=bad)
    for b in (ladders[:2], [[[1.0]]], [0.9, 0.5], [1.0, 0.5, 0.5]):
        with pytest.raises(ValueError):
            SightlineParallelTemperingSampler(W, 2, _Batch(), betas=b)
    with pytest.raises(ValueError, match="adapt"):
        smp.run_mcmc(np.zeros((S, W, 2)), 5, adapt=True, accumulate=True)
    with pytest.raises(ValueError):
        smp.run_mcmc(np.zeros((S, W, 2)), 5, n_record=4)
    with pytest.raises(ValueError, match="no moments"):
        smp.log_evidence_estimate()
    with pytest.raises(ValueError):
        smp.get_log_like()                                                           # record_log_like=False
    with pytest.raises(ValueError):
        SightlineParallelTemperingSampler(W, 3, _Batch())
    with pytest.raises(ValueError):
        SightlineParallelTemperingSampler(1, 2, _Batch())
    with pytest.raises(TypeError):
        SightlineParallelTemperingSampler(W, 2, object())
    with pytest.raises(IndexError):
        smp.sightline(S)


def test_sightline_sampler_evidence_from_hand_filled_moments():
    """log_evidence_estimate on hand-filled moments: per-sightline evidence_from_moments; a non-finite sightline
    gets NaN and one warning naming it; the view returns scalars."""
    S, W = 3, 6
    betas = [1.0, 0.5, 0.0]
    smp = SightlineParallelTemperingSampler(W, 2, _Batch(), betas=betas)
    rng = np.random.default_rng(2)
    E, V = -10.0 + rng.standard_normal((S, 3)), rng.uniform(0.5, 2.0, (S, 3))
    n = 60.0
    smp._ti = np.stack([np.full((S, 3), n), E, V * n], axis=-1)
    smp._ti_betas, smp.evidence_steps = smp.betas, 10
    lnz, dlnz = smp.log_evidence_estimate()
    for s in range(S):
        assert (lnz[s], dlnz[s]) == evidence_from_moments(betas, E[s], (V[s] * n) / n)
    assert smp.sightline(1).log_evidence_estimate() == (lnz[1], dlnz[1])
    smp._ti[2, 1, 2] = np.nan
    with pytest.warns(RuntimeWarning, match=r"\[2\]"):
        lnz2, dlnz2 = smp.log_evidence_estimate()
    assert np.array_equal(lnz2[:2], lnz[:2]) and np.isnan(lnz2[2]) and np.isnan(dlnz2[2])
