"""oracle/slice_replay_sightlines.py (CPU only): the survey-mode replay -- the walker-counter offset of ensemble e and
the per-half-step batch counts that rbv_slice_run_sightlines is checked against."""
import numpy as np

MU = np.array([1.0, -2.0, 0.5])
COV = np.array([[0.25, 0.3, 0.0], [0.3, 4.0, 0.5], [0.0, 0.5, 1.0]])
ICOV = np.linalg.inv(COV)


def _lnp(x):
    d = np.atleast_2d(x) - MU
    return -0.5 * np.einsum("ni,ij,nj->n", d, ICOV, d)


def _start(seed=4, W=10):
    return MU + 0.1 * np.random.default_rng(seed).standard_normal((W, 3))


def test_slice_replay_default_offset_reproduces_single_ensemble_run():
    """walker_offset=0 is the single-ensemble replay (oracle/slice_replay.py) bit for bit, at both depths (depth
    changes only the number of batches), and matches the counters, mu and chain pinned from it."""
    from oracle import slice_replay, slice_replay_sightlines as sl
    p0 = _start()
    for depth, nbatches in ((1, 687), (2, 400)):
        out = sl.run(_lnp, p0, _lnp(p0), 60, seed=99, depth=depth)
        ref = slice_replay.run(_lnp, p0, _lnp(p0), 60, seed=99, depth=depth)
        for key in ("chain", "lnp_chain", "mus"):
            assert np.array_equal(out[key], ref[key]), key
        for key in ("mu", "tune", "good", "nexp", "ncon", "ncall", "nbatches"):
            assert out[key] == ref[key], key
        assert (out["nexp"], out["ncon"], out["ncall"], out["nbatches"]) == (695, 568, 3063, nbatches)
        assert (out["tune"], out["good"]) == (False, 6)
        assert abs(out["mu"] - 0.8093344506506087) <= 1e-14
        assert abs(out["chain"][-1].sum() - -0.3658812389966257) <= 1e-12
    # a continued run with the carried tuning state equals one long run, as for the single-ensemble replay
    a = sl.run(_lnp, p0, _lnp(p0), 25, seed=99, walker_offset=30)
    b = sl.run(_lnp, a["chain"][-1], a["lnp_chain"][-1], 35, seed=99, mu=a["mu"], tune=a["tune"], good=a["good"],
               first_step=25, walker_offset=30)
    whole = sl.run(_lnp, p0, _lnp(p0), 60, seed=99, walker_offset=30)
    assert np.array_equal(np.concatenate([a["chain"], b["chain"]]), whole["chain"])
    assert np.array_equal(np.concatenate([a["batches_per_half"], b["batches_per_half"]]), whole["batches_per_half"])


def test_slice_replay_walker_offset_changes_the_streams_and_batches_sum():
    """An offset gives ensemble e its own random streams (another chain from the same start); the batches of every
    half-step sum to nbatches, every half-step needs at least two, and the lockstep launch count of several ensembles
    is the per-half-step maximum."""
    from oracle import slice_replay_sightlines as sl
    p0 = _start()
    W, nsteps = len(p0), 40
    runs = [sl.run(_lnp, p0, _lnp(p0), nsteps, seed=7, walker_offset=e * W) for e in range(3)]
    assert not np.array_equal(runs[0]["chain"], runs[1]["chain"])
    assert not np.array_equal(runs[1]["chain"], runs[2]["chain"])
    for out in runs:
        per = out["batches_per_half"]
        assert per.shape == (2 * nsteps,) and per.sum() == out["nbatches"] and per.min() >= 2
        assert np.allclose(out["lnp_chain"], _lnp(out["chain"].reshape(-1, 3)).reshape(out["lnp_chain"].shape))
    lockstep = np.max([out["batches_per_half"] for out in runs], axis=0).sum()
    assert max(out["nbatches"] for out in runs) <= lockstep <= sum(out["nbatches"] for out in runs)
    # depth 2 serves the same chain in fewer batches per half-step
    two = sl.run(_lnp, p0, _lnp(p0), nsteps, seed=7, walker_offset=W, depth=2)
    assert np.array_equal(two["chain"], runs[1]["chain"])
    assert np.all(two["batches_per_half"] <= runs[1]["batches_per_half"])
