"""GPU: the batch sizes and run lengths at which the launch configuration, not the arithmetic, decides the result.

A. Row counts past 65 535, the CUDA limit of gridDim.y / gridDim.z: the gradient, Fisher and Jacobian launches put the
   row in grid y or z and go over the rows in slices (DESIGN.md sections 14, 15).  Every row must be bit-identical to
   the same row in a small batch, and the rows at the slice seams must match the oracles.
B. The stretch-move chain handed to the host in many blocks (rbv_stretch_run_sink): ring reuse, short and one-step
   last blocks, the cooperative kernel per block, the cooperative path without a sink, the captured-graph path, and
   continuation across block boundaries -- bit for bit against the plain per-step loop."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_fisher import FISHER_TOL, JAC_TOL, _c1_on_grid  # noqa: E402
from test_gpu_gradient import GRAD_TOL, VALUE_RTOL  # noqa: E402

pytestmark = pytest.mark.gpu

GRID_ROWS = 65535                  # gridDim.y / gridDim.z limit
SIZES = [65535, 65536, 131071]     # the last size one slice covers, the first that needs two, two seams + 1 ragged row
NAN_ROW, BAD_B_ROW, OUT_ROW = 65534, 65535, 65536
CHUNK = 4096


def _slices(W):
    return -(-W // GRID_ROWS)


def _rows(W):
    """C1 ensemble of W rows with a NaN row, a b < 0 row and an out-of-bounds row straddling the first seam, and an
    in-bounds last row (where W leaves room for them)."""
    from rbvfit_b200 import workloads as wl
    w = wl.get_workload("C1")
    th = wl.make_ensemble(w, W)
    C = th.shape[1] // 3
    good = np.clip(w["theta_true"] + np.array([0.05, -0.03, 2.0, -1.5, 3.0, -4.0]), w["lb"], w["ub"])
    # every row of the seam starts in bounds (make_ensemble pushes ~1 % of its rows out), then gets its one change
    for i in (NAN_ROW - 1, NAN_ROW, BAD_B_ROW, OUT_ROW, OUT_ROW + 1, W - 1):
        if i < W:
            th[i] = good + 1e-3 * i / W
    if NAN_ROW < W:
        th[NAN_ROW, 1] = np.nan
    if BAD_B_ROW < W:
        th[BAD_B_ROW, C] = -1.0
    if OUT_ROW < W:
        th[OUT_ROW, 0] = w["ub"][0] + 1.0
    return th


def _seam_rows(W):
    """Finite rows on both sides of every seam, plus the first and the last row."""
    return sorted({i for i in (0, NAN_ROW - 1, OUT_ROW, OUT_ROW + 1, W - 1) if i < W} - {NAN_ROW, BAD_B_ROW})


def _chunked(fn, th, n=CHUNK):
    parts = [fn(th[i:i + n]) for i in range(0, len(th), n)]
    if isinstance(parts[0], tuple):
        return tuple(np.concatenate(p) for p in zip(*parts))
    return np.concatenate(parts)


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.fixture(scope="module", params=[5, 1], ids=["K5", "K1"])
def grid_problem(request):
    """C1's lines on 64 pixels with a 5-tap LSF, or one tap (no LSF: fisher_lsf_kernel is not launched)."""
    like, comp, _theta = _c1_on_grid(64, request.param)
    yield request.param, like, comp
    like.close()


# ------------------------------------------------------------------------------------------ A. rows past the grid limit
@pytest.mark.parametrize("W", SIZES)
def test_gradient_past_the_grid_limit(grid_problem, W):
    import torch
    from oracle import voigt_grad_oracle as vg
    _K, like, comp = grid_problem
    th = _rows(W)
    C = th.shape[1] // 3
    n0 = like.engine.launch_count
    v, g = like.lnprob_and_grad(th)
    assert like.engine.launch_count - n0 == 2 + 4 * _slices(W)       # prep, finalize + 4 per slice of rows
    vc, gc = _chunked(like.lnprob_and_grad, th)
    assert _same(v, vc) and _same(g, gc)
    vl, gl = like.lnlike_and_grad(th)
    vlc, glc = _chunked(like.lnlike_and_grad, th)
    assert _same(vl, vlc) and _same(gl, glc)
    t = torch.tensor(th, dtype=torch.float64, device=like.engine.tdev, requires_grad=True)
    out = like.lnprob_torch(t)
    out.sum().backward()
    assert _same(out.detach().cpu().numpy(), v) and _same(t.grad.cpu().numpy(), g)
    # special rows: NaN stays NaN, out of bounds gives -inf and a zero gradient (with the prior)
    if NAN_ROW < W:
        assert np.isnan(v[NAN_ROW]) and np.isnan(vl[NAN_ROW]) and np.isnan(g[NAN_ROW, :3 * C]).any()
    if BAD_B_ROW < W:
        assert v[BAD_B_ROW] == -np.inf and np.all(g[BAD_B_ROW] == 0.0)
        assert np.isnan(vl[BAD_B_ROW]) and np.isnan(gl[BAD_B_ROW, :3 * C]).any()
    if OUT_ROW < W:
        assert v[OUT_ROW] == -np.inf and np.all(g[OUT_ROW] == 0.0)
        assert np.isfinite(vl[OUT_ROW]) and np.all(np.isfinite(gl[OUT_ROW]))
    oob = ~np.isfinite(v) & ~np.isnan(v)
    assert np.all(g[oob] == 0.0)
    # value against the forward path, gradient at the seams against the oracle
    fin = np.isfinite(vl)
    ref = like.lnlike(th)
    assert np.max(np.abs(vl[fin] - ref[fin]) / np.abs(ref[fin])) <= VALUE_RTOL
    worst = 0.0
    for i in _seam_rows(W):
        G = vg.grad_scale(comp, th[i])
        ok = G > 0
        assert np.all(gl[i][~ok] == 0.0)
        worst = max(worst, float(np.max(np.abs(gl[i][ok] - vg.lnlike_grad(comp, th[i])[ok]) / G[ok])))
    print(W, "seam rows", _seam_rows(W), "max |dg| / G", worst)
    assert worst <= GRAD_TOL


@pytest.mark.parametrize("W", SIZES)
def test_fisher_and_jacobian_past_the_grid_limit(grid_problem, W):
    from oracle import voigt_fisher_oracle as vf
    K, like, comp = grid_problem
    eng = like.engine
    th = _rows(W)
    C = th.shape[1] // 3
    ref_v, ref_g, ref_F = like.lnlike_and_fisher(th)             # default chunks: fewer rows than the grid limit
    ref_J = like.model_jacobian(th, 0)
    assert eng._fisher_rows_per_chunk() < GRID_ROWS
    eng.fisher_chunk_bytes = 1 << 40                               # the whole batch in one launch sequence
    try:
        n0 = eng.launch_count
        v, g, F = like.lnlike_and_fisher(th)
        per_slice = 4 + (1 if K > 1 else 0)                        # flux, resid, col [, lsf], gram
        assert eng.launch_count - n0 == 2 + per_slice * _slices(W)
        J = like.model_jacobian(th, 0)
    finally:
        eng.fisher_chunk_bytes = type(eng).fisher_chunk_bytes
    assert _same(v, ref_v) and _same(g, ref_g) and _same(F, ref_F)
    assert _same(J, ref_J)
    if NAN_ROW < W:
        assert np.isnan(v[NAN_ROW]) and np.isnan(F[NAN_ROW, :3 * C, :3 * C]).any()
    if BAD_B_ROW < W:
        assert np.isnan(v[BAD_B_ROW]) and np.isnan(J[BAD_B_ROW][:, :3 * C]).all()
    dd = next(iter(comp.values()))
    for i in _seam_rows(W):
        ll, _g, F_or = vf.lnlike_fisher(comp, th[i])
        assert abs(v[i] - ll) <= 3e-11 * abs(ll)                    # the forward model's own error (test_gpu_fisher)
        d = np.sqrt(np.outer(np.diag(F_or), np.diag(F_or)))
        ok = d > 0
        assert np.all(F[i][~ok] == 0.0)
        assert np.max(np.abs(F[i] - F_or)[ok] / d[ok]) <= FISHER_TOL
        J_or = vf.model_jacobian(dd, th[i])
        scale = np.max(np.abs(J_or[:3 * C]), axis=1)
        assert np.max(np.max(np.abs(J[i].T[:3 * C] - J_or[:3 * C]), axis=1) / scale) <= JAC_TOL


def _c1_sightline(P, K, seed):
    """One sightline of C1's structure on a P-pixel grid with a K-tap LSF and its own noise realisation."""
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    w = wl.get_workload("C1")
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    for (z, ion, trans, comps) in w["systems"]:
        cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        ocfg.add_system(z, ion, trans, comps)
    taps = vo.cos_like_lsf(K)
    wave = np.linspace(3770.0, 3780.0, P)
    rng = np.random.default_rng(seed)
    flux = vo.model_flux(vo.lower(ocfg, custom_taps=taps), w["theta_true"], wave) + 0.02 * rng.standard_normal(P)
    return w, dict(model=GpuVoigtModel(cfg, FWHM=None, lsf_taps=taps), wave=wave, flux=flux, error=np.full(P, 0.02))


def test_sightline_fisher_past_the_grid_limit():
    """3 sightlines x 21 847 walkers = 65 541 rows in one launch sequence: the seam at row 65 535 falls inside
    sightline 2, so every row must still be evaluated against inst0 + w / wps."""
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    S, wps = 3, 21847
    specs = [_c1_sightline(64, 5, 40 + s) for s in range(S)]
    w = specs[0][0]
    batch = SightlineBatch([d for _w, d in specs], w["lb"], w["ub"])
    singles = [GpuLikelihood({"COS": d}, w["lb"], w["ub"]) for _w, d in specs]
    th = _rows(S * wps).reshape(S, wps, -1)
    batch.engine.fisher_chunk_bytes = 1 << 40
    n0 = batch.engine.launch_count
    v, g, F = batch.lnlike_and_fisher(th)
    assert batch.engine.launch_count - n0 == 2 + 5 * _slices(S * wps)
    for s in range(S):
        vs, gs, Fs = singles[s].lnlike_and_fisher(th[s])
        assert _same(v[s], vs) and _same(g[s], gs) and _same(F[s], Fs), s
    batch.close()
    for like in singles:
        like.close()


def test_sightline_lm_past_the_grid_limit():
    """SightlineBatch.fit_quick over 66 000 one-component 64-pixel sightlines with the whole batch in one device loop
    (every Fisher launch of the loop and of the covariance fallback covers 66 000 rows) against the default blocks of
    whole sightlines, and sightlines at both ends and the seam against one-sightline runs."""
    import time
    import warnings
    from oracle import voigt_oracle as vo
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
    S, P, sigma = 66000, 64, 0.02
    z, ion, trans = 0.348, "MgII", [2796.3, 2803.5]
    t = np.array([14.2, 40.0, -25.0])
    lb, ub = wl.default_bounds(t[:1], t[1:2], t[2:])
    cfg, ocfg = FitConfiguration(), vo.OracleConfig()
    cfg.add_system(z=z, ion=ion, transitions=trans, components=1)
    ocfg.add_system(z, ion, trans, 1)
    taps = vo.cos_like_lsf(5)
    wave = np.linspace(3765.0, 3785.0, P)
    clean = vo.model_flux(vo.lower(ocfg, custom_taps=taps), t, wave)
    rng = np.random.default_rng(66000)
    flux = clean[None, :] + sigma * rng.standard_normal((S, P))
    x0 = np.clip(t + np.array([0.05, 3.0, 3.0]) * rng.standard_normal((S, 3)), lb, ub)
    model = GpuVoigtModel(cfg, FWHM=None, lsf_taps=taps).compile(verbose=False)
    t0 = time.perf_counter()
    batch = SightlineBatch([dict(model=model, wave=wave, flux=f, error=np.full(P, sigma)) for f in flux], lb, ub)
    print(f"{S} sightlines set up in {time.perf_counter() - t0:.1f} s")
    eng = batch.engine
    one = eng._sl_bytes(eng.lib.rbv_lm_workspace_bytes_sightlines, 1, "rbv_lm_workspace_bytes_sightlines")
    assert eng.fisher_chunk_bytes // one < GRID_ROWS < S                # the default blocks stay below the limit
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                                 # sightlines that do not converge
        ref = batch.fit_quick(x0)
        eng.fisher_chunk_bytes = 1 << 40
        try:
            got = batch.fit_quick(x0)
        finally:
            eng.fisher_chunk_bytes = type(eng).fisher_chunk_bytes
    print("status counts", np.unique(got.status, return_counts=True), "max n_evals", got.n_evals.max())
    assert np.mean(got.status > 0) > 0.9
    for a, b in zip(got, ref):
        assert _same(a, b)
    # one row per sightline is a 66 000-row Fisher launch whatever the budget
    v, g, F = batch.lnlike_and_fisher(got.x[:, None, :])
    for s in (0, GRID_ROWS - 1, GRID_ROWS, S - 1):
        single = eng.lm_sightlines(x0[s:s + 1], s, 1)
        for i, field in enumerate(("x", "chi2", "n_evals", "status")):
            assert _same(single[(0, 1, 3, 4)[i]][0], getattr(got, field)[s]), (s, field)
        if not single[5][0] & 1:                  # fit_quick replaces a non-positive-definite F_ff's covariance
            assert _same(single[2][0], got.cov[s]), s
        like = GpuLikelihood({"COS": dict(model=model, wave=wave, flux=flux[s], error=np.full(P, sigma))}, lb, ub)
        vs, gs, Fs = like.lnlike_and_fisher(got.x[s])
        assert vs == v[s, 0] and _same(gs, g[s, 0]) and _same(Fs, F[s, 0]), s
        like.close()
    batch.close()


@pytest.mark.parametrize("stream", ["0", "1"])
def test_forward_paths_past_the_grid_limit(monkeypatch, stream):
    """lnprob (tile and streaming kernel), the sightline lnprob and model_flux put rows in grid x or a work queue:
    131 071 rows in one launch give what batches of 4096 give."""
    from rbvfit_b200.likelihood import SightlineBatch
    monkeypatch.setenv("RBVFIT_B200_STREAM", stream)
    like, _comp, _theta = _c1_on_grid(64, 5)
    th = _rows(131071)
    assert _same(like.lnprob(th), _chunked(like.lnprob, th))
    assert like.engine.last_kernel == ("stream" if stream == "1" else "tile")
    assert _same(like.engine.model_flux(0, th), _chunked(lambda t: like.engine.model_flux(0, t), th))
    like.close()
    S, wps = 3, 43691
    specs = [_c1_sightline(64, 5, 40 + s) for s in range(S)]
    w = specs[0][0]
    batch = SightlineBatch([d for _w, d in specs], w["lb"], w["ub"])
    ths = _rows(S * wps).reshape(S, wps, -1)
    full = batch.lnprob(ths)
    parts = np.concatenate([batch.lnprob(np.ascontiguousarray(ths[:, j:j + CHUNK]))
                            for j in range(0, wps, CHUNK)], axis=1)
    assert _same(full, parts)
    batch.close()


# ------------------------------------------------------------------------------------------ B. the chain sink
def _p0(w, W, seed):
    rng = np.random.default_rng(seed)
    return np.clip(w["theta_true"] + 1e-3 * rng.standard_normal((W, 6)), w["lb"], w["ub"])


def _sink_block(W, nsteps):
    """Engine.stretch_run_to_host's block length for W walkers of C1."""
    return int(min(256, max(1, (6 << 20) // (W * 7 * 8)), max(1, (nsteps + 1) // 2)))


def _run(like, p0, nsteps, seed, use_graph, split_at=None):
    """(chain, log-prob, acceptance, launches) of a DeviceEnsembleSampler run; split_at: run(split_at) then
    run(None, nsteps - split_at)."""
    from rbvfit_b200.sampler import DeviceEnsembleSampler
    smp = DeviceEnsembleSampler(p0.shape[0], p0.shape[1], like, seed=seed, use_graph=use_graph)
    n0 = like.engine.launch_count
    if split_at is None:
        smp.run_mcmc(p0, nsteps)
    else:
        smp.run_mcmc(p0, split_at)
        smp.run_mcmc(None, nsteps - split_at)
    return smp.get_chain(), smp.get_log_prob(), smp.acceptance_fraction, like.engine.launch_count - n0, smp._seed


def _assert_same_run(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


@pytest.fixture(scope="module")
def c1_sampler_problem():
    """C1 (2048 pixels) with 50 walkers: 25-row half-steps, the cooperative voigt_mcmc_kernel's size."""
    from test_gpu_vfit import _c1_fitter
    mp = pytest.MonkeyPatch()
    mp.delenv("RBVFIT_B200_STREAM", raising=False)       # the streaming kernel would rule the cooperative one out
    mp.delenv("RBVFIT_B200_MCMC_PERSISTENT", raising=False)
    w, fitter, _comp, _t = _c1_fitter(nwalkers=50)
    mp.undo()
    like = fitter._like
    p0 = _p0(w, 50, 12)
    ref = {n: _run(like, p0, n, 31, use_graph=False) for n in (1100, 513)}
    yield w, like, p0, ref
    like.close()


def _launches_of_initial_lnprob(like, W):
    import torch
    n0 = like.engine.launch_count
    like.engine.lnprob_device(torch.zeros((W, like.ndim), dtype=torch.float64, device=like.engine.tdev) +
                              torch.as_tensor(like.lb, device=like.engine.tdev))
    return like.engine.launch_count - n0


@pytest.mark.parametrize("nsteps", [1100, 513])
def test_sink_ring_reuse_cooperative_kernel(c1_sampler_problem, nsteps):
    """1100 steps = blocks of 256, 256, 256, 256, 76 (the ring halves are refilled twice); 513 = 256, 256, 1."""
    from oracle import stretch_replay as sr
    _w, like, p0, ref = c1_sampler_problem
    K = _sink_block(50, nsteps)
    assert K == 256
    got = _run(like, p0, nsteps, 31, use_graph=True)
    _assert_same_run(got, ref[nsteps])
    # one cooperative launch per block (besides the ensemble's initial lnprob)
    assert got[3] - _launches_of_initial_lnprob(like, 50) == -(-nsteps // K)
    chain, lps = got[0], got[1]
    for s in sorted({0, K - 1, K, 2 * K, 4 * K, nsteps - 1} & set(range(nsteps))):
        assert np.array_equal(like.lnprob(chain[s]), lps[s]), s
    if nsteps == 1100:
        n = 120
        rc, rl, nacc = sr.run(like.lnprob, p0, like.lnprob(p0), n, got[4])
        assert np.allclose(chain[:n], rc, rtol=0, atol=1e-9)
        assert np.max(np.abs(lps[:n] - rl) / np.abs(rl)) <= 1e-9
        moved = np.any(chain[1:n] != chain[:n - 1], axis=2).sum(axis=0) + np.any(chain[0] != p0, axis=1)
        assert np.array_equal(moved, nacc)


@pytest.mark.parametrize("persistent", ["0", "1"])
def test_sink_graph_and_cooperative_paths_agree(c1_sampler_problem, monkeypatch, persistent):
    """The same runs with the cooperative kernel switched off (captured graph of one step per replay) or on, each in a
    fresh likelihood."""
    from test_gpu_vfit import _c1_fitter
    _w, _like, p0, ref = c1_sampler_problem
    monkeypatch.delenv("RBVFIT_B200_STREAM", raising=False)
    monkeypatch.setenv("RBVFIT_B200_MCMC_PERSISTENT", persistent)
    _w2, fitter, _comp, _t = _c1_fitter(nwalkers=50)
    like = fitter._like
    init = _launches_of_initial_lnprob(like, 50)
    for nsteps in (1100, 513):
        got = _run(like, p0, nsteps, 31, use_graph=True)
        _assert_same_run(got, ref[nsteps])
        blocks = -(-nsteps // _sink_block(50, nsteps))
        if persistent == "1":
            assert got[3] - init == blocks
        else:
            assert got[3] - init >= 2 * nsteps                     # >= 2 kernels per step, replayed from the graph
    like.close()


def test_cooperative_run_without_sink(c1_sampler_problem):
    """Engine.stretch_run(use_graph=True) of 2100 steps: cooperative launches of 1024, 1024 and 52 steps with no
    sink, against the sink run of the same seed (2100 steps = 8 blocks of 256 and one of 52)."""
    import torch
    _w, like, p0, _ref = c1_sampler_problem
    eng = like.engine
    n = 2100
    sink = _run(like, p0, n, 31, use_graph=True)
    dev = eng.tdev
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.current_stream(dev).synchronize()
    with torch.cuda.stream(stream):
        coords_t = torch.as_tensor(p0, device=dev)
        lnp_t = eng.lnprob_device(coords_t)
        chain_t = torch.empty((n, 50, 6), dtype=torch.float64, device=dev)
        lps_t = torch.empty((n, 50), dtype=torch.float64, device=dev)
        nacc_t = torch.zeros(50, dtype=torch.int32, device=dev)
        flag_t = torch.zeros(1, dtype=torch.int32, device=dev)
        n0 = eng.launch_count
        eng.stretch_run(coords_t, lnp_t, n, 2.0, sink[4], 0, chain_t, lps_t, nacc_t, flag_t, use_graph=True)
        launches = eng.launch_count - n0
        stream.synchronize()
    assert int(flag_t.item()) == 0                                    # bit 2: a grid-barrier timeout
    assert launches == 3
    assert np.array_equal(chain_t.cpu().numpy(), sink[0]) and np.array_equal(lps_t.cpu().numpy(), sink[1])
    assert np.array_equal(nacc_t.cpu().numpy() / n, sink[2])
    assert np.array_equal(coords_t.cpu().numpy(), sink[0][-1]) and np.array_equal(lnp_t.cpu().numpy(), sink[1][-1])


def test_sink_continuation_across_blocks(c1_sampler_problem):
    """run(600) (blocks 256, 256, 88) then run(None, 500) (250, 250, first_step 600) is run(1100)."""
    _w, like, p0, ref = c1_sampler_problem
    _assert_same_run(_run(like, p0, 1100, 31, use_graph=True, split_at=600), ref[1100])


def test_sink_many_short_blocks_large_ensemble():
    """4096 walkers: blocks of 27 steps (27, 27, 27, 19 for 100 steps) on the captured-graph path with a separate
    finalisation launch, against the plain per-step loop."""
    from test_gpu_vfit import _c1_fitter
    w, fitter, _comp, _t = _c1_fitter(nwalkers=4096)
    like = fitter._like
    assert _sink_block(4096, 100) == 27
    p0 = _p0(w, 4096, 13)
    a = _run(like, p0, 100, 17, use_graph=True)
    b = _run(like, p0, 100, 17, use_graph=False)
    _assert_same_run(a, b)
    # recomputed as one 4096-row batch, which may take another tile geometry or kernel than the 2048-row half-steps
    for s in (0, 26, 27, 54, 81, 99):
        assert np.max(np.abs(like.lnprob(a[0][s]) - a[1][s]) / np.abs(a[1][s])) <= 1e-12, s
    like.close()
