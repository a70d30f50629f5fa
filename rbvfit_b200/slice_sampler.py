"""Batched ensemble slice sampler with zeus's semantics and sampler-object contract.

The reference hands ``vfit.lnprob`` to ``zeus.EnsembleSampler(nwalkers, ndim, lnprob, pool=pool)``
(src/rbvfit/vfit_mcmc.py:425-440) when ``sampler='zeus'``.  zeus-mcmc is a third-party dependency that is not
vendored (requirements.txt:11, ``zeus-mcmc>=2.3.0``) and is not installed here, so the algorithm is restated
from its published description (Karamanis & Beutler 2021, "Ensemble slice sampling", Algorithm 2-3; zeus 2.x
defaults: DifferentialMove, mu = 1 tuned by stochastic approximation, tolerance 0.05, patience 5):

  per iteration, for each half of the (shuffled) ensemble with the other half as the complementary set C:
      direction_k = 2 mu (C_j - C_l),  j != l drawn from C                       (differential move)
      slice level  y_k = lnp(X_k) - Exp(1)
      stepping out: [L, R] = [-U, 1 - U]; widen L (R) by 1 while lnp(X_k + L dir_k) > y_k, counting expansions
      shrinking:   draw t ~ U(L, R); accept X_k + t dir_k if lnp >= y_k, else shrink the bracket towards 0
      tuning:      mu <- mu * 2 n_exp / (n_exp + n_con) until the expansion fraction sits at 1/2 +- tolerance

Every lnp evaluation inside the two loops is ONE device batch over the walkers that are still active in
that loop (``vectorize=True`` contract) -- the long tail of small batches is latency-bound on the GPU
(SURVEY.md section 7.3).  ``DeviceEnsembleSliceSampler`` keeps the whole loop on the device instead
(``rbv_slice_run``): the walkers of a half advance in lockstep through their own widen / shrink state machines, one
masked device batch per iteration, and only a 24-byte counter block is read back between iterations.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np

from .sampler import _ChunkedHistory, integrated_time


class EnsembleSliceSampler(_ChunkedHistory):
    def __init__(self, nwalkers: int, ndim: int, log_prob_fn: Callable, mu: float = 1.0, tune: bool = True,
                 tolerance: float = 0.05, patience: int = 5, maxsteps: int = 10000, maxiter: int = 10000,
                 pool=None, vectorize: bool = True, seed: Optional[int] = None):
        if nwalkers < 2 * ndim or nwalkers % 2:
            raise ValueError("Please provide at least (2 * ndim) walkers, and an even number of them.")
        self.nwalkers, self.ndim = int(nwalkers), int(ndim)
        self.log_prob_fn = log_prob_fn
        self.vectorize = vectorize
        self.pool = pool
        self.mu, self.mu0 = float(mu), float(mu)
        self.tune, self.tolerance, self.patience = bool(tune), float(tolerance), int(patience)
        self.maxsteps, self.maxiter = int(maxsteps), int(maxiter)
        self._random = np.random.default_rng(seed)
        self.reset()

    def reset(self):
        self._chain = np.empty((0, self.nwalkers, self.ndim))
        self._log_prob = np.empty((0, self.nwalkers))
        self.iteration = 0
        self.ncall = 0          # lnp evaluations (rows)
        self.nbatches = 0       # lnp calls (device batches)
        self.mus = []
        self._last = None

    def compute_log_prob(self, coords):
        coords = np.atleast_2d(coords)
        if self.vectorize:
            lp = np.asarray(self.log_prob_fn(coords), dtype=np.float64)
        else:
            lp = np.array([float(self.log_prob_fn(c)) for c in coords])
        self.ncall += len(coords)
        self.nbatches += 1
        if np.any(np.isnan(lp)):
            raise ValueError("Probability function returned NaN")
        return lp

    # ------------------------------------------------------------------ one iteration
    def _iterate(self, X, Z):
        nw, rng = self.nwalkers, self._random
        half = nw // 2
        order = rng.permutation(nw)
        nexp = ncon = 0
        for split in range(2):
            active = order[split * half:(split + 1) * half]
            inactive = order[(1 - split) * half:(2 - split) * half] if split == 0 else order[:half]
            n = len(active)
            # differential move: two distinct complementary walkers per active walker
            j = rng.integers(0, len(inactive), size=n)
            l = (j + rng.integers(1, len(inactive), size=n)) % len(inactive)
            directions = 2.0 * self.mu * (X[inactive[j]] - X[inactive[l]])
            X0, Z0 = X[active].copy(), Z[active] - rng.exponential(size=n)
            L = -rng.random(n)
            R = L + 1.0
            # stepping out, left then right (batched over the walkers still expanding)
            J = np.floor(self.maxsteps * rng.random(n)).astype(int)
            K = (self.maxsteps - 1) - J
            for side, budget in ((L, J), (R, K)):
                step = -1.0 if side is L else 1.0
                mask = np.ones(n, dtype=bool)
                while np.any(mask):
                    idx = np.flatnonzero(mask)
                    Zs = self.compute_log_prob(X0[idx] + side[idx, None] * directions[idx])
                    grow = (Zs >= Z0[idx]) & (budget[idx] >= 1)
                    side[idx[grow]] += step
                    budget[idx[grow]] -= 1
                    nexp += int(grow.sum())
                    mask[idx[~grow]] = False
            # shrinking
            Xp, Zp = X0.copy(), np.empty(n)
            mask = np.ones(n, dtype=bool)
            it = 0
            while np.any(mask):
                idx = np.flatnonzero(mask)
                t = L[idx] + rng.random(len(idx)) * (R[idx] - L[idx])
                cand = X0[idx] + t[:, None] * directions[idx]
                Zc = self.compute_log_prob(cand)
                ok = Zc >= Z0[idx]
                Xp[idx[ok]] = cand[ok]
                Zp[idx[ok]] = Zc[ok]
                mask[idx[ok]] = False
                rej = idx[~ok]
                tl = t[~ok]
                L[rej[tl < 0]] = tl[tl < 0]
                R[rej[tl >= 0]] = tl[tl >= 0]
                ncon += len(rej)
                it += 1
                if it > self.maxiter:
                    raise RuntimeError("Number of contractions exceeded maximum limit!")
            X[active], Z[active] = Xp, Zp
        return X, Z, nexp, ncon

    def run_mcmc(self, start, nsteps, progress=False, **_ignored):
        if start is None:
            if self._last is None:
                raise ValueError("Cannot have `start=None` if run_mcmc has never been called.")
            X, Z = self._last
        else:
            X = np.array(start, dtype=np.float64, copy=True)
            if X.shape != (self.nwalkers, self.ndim):
                raise ValueError("Incompatible input dimensions! Please provide array of shape (nwalkers, ndim)")
            Z = self.compute_log_prob(X)
            if not np.all(np.isfinite(Z)):
                raise ValueError("Invalid walker initial positions! Initialise walkers from positions of finite "
                                 "log probability.")
        chain = np.empty((nsteps, self.nwalkers, self.ndim))
        lps = np.empty((nsteps, self.nwalkers))
        it = range(nsteps)
        if progress:
            try:
                from tqdm import tqdm
                it = tqdm(it, total=nsteps)
            except ImportError:
                pass
        good = 0
        for i in it:
            X, Z, nexp, ncon = self._iterate(X, Z)
            if self.tune:
                nexp = max(1, nexp)
                self.mu *= 2.0 * nexp / (nexp + ncon)
                self.mus.append(self.mu)
                if abs(nexp / (nexp + ncon) - 0.5) < self.tolerance:
                    good += 1
                if good > self.patience:
                    self.tune = False
            chain[i], lps[i] = X, Z
        self._hist_append(chain, lps)
        self.iteration += nsteps
        self._last = (X, Z)
        return X, Z

    # ------------------------------------------------------------------ zeus-shaped accessors
    def _get(self, arr, discard=0, thin=1, flat=False):
        v = arr[discard::thin]
        if flat:
            return v.reshape((-1,) + v.shape[2:])
        return v

    def get_chain(self, flat=False, thin=1, discard=0):
        return self._get(self._chain, discard, thin, flat)

    def get_log_prob(self, flat=False, thin=1, discard=0):
        return self._get(self._log_prob, discard, thin, flat)

    @property
    def chain(self):
        return self._chain

    @property
    def acceptance_fraction(self):
        """Fraction of (walker, step) pairs that moved -- what the reference derives for zeus chains
        (vfit_mcmc.py:470-486); slice sampling always moves, so this is ~1."""
        c = self._chain
        if len(c) < 2:
            return np.ones(self.nwalkers)
        return np.mean(np.any(c[1:] != c[:-1], axis=2), axis=0)

    @property
    def efficiency(self):
        return self.iteration * self.nwalkers / max(self.ncall, 1)

    def get_autocorr_time(self, discard=0, thin=1, **kwargs):
        return thin * integrated_time(self.get_chain(discard=discard, thin=thin), **kwargs)

    def get_last_sample(self):
        return self._last


class DeviceEnsembleSliceSampler(EnsembleSliceSampler):
    """Same move, same accessor contract, but the whole loop runs on the GPU (``rbv_slice_run``, C ABI): directions,
    slice levels, brackets, the per-walker widen / shrink state machines and the adaptation of mu live in device
    memory, every iteration is one masked likelihood batch over the active half -- the body of a CUDA-graph WHILE
    node whose condition the device sets (``use_graph=False``: the host polls a counter block instead) -- and the
    chain is copied to the host once per ``run_mcmc`` call.  ``likelihood`` is a ``GpuLikelihood``; random numbers
    come from the counter-based Philox streams of the device stretch move, so a run is reproducible and can be
    continued (``run_mcmc(None, n)``) without changing the stream of one long run (``oracle/slice_replay.py``
    restates it in numpy for the tests).  ``depth``: logical iterations served per launch (1 or 2, default 2 -- the
    second one's candidates are evaluated speculatively, ``csrc/rbv_slice.cuh``); chains, ``mu`` and the counters
    ``ncall`` / ``nexp`` / ``ncon`` do not depend on it, only ``nbatches`` does."""

    def __init__(self, nwalkers: int, ndim: int, likelihood, mu: float = 1.0, tune: bool = True,
                 tolerance: float = 0.05, patience: int = 5, maxsteps: int = 10000, maxiter: int = 10000,
                 seed: Optional[int] = None, use_graph: bool = True, depth: int = 2, **_ignored):
        if not hasattr(likelihood, "engine"):
            raise TypeError("DeviceEnsembleSliceSampler needs a GpuLikelihood (the log-probability must run on "
                            "the device)")
        if likelihood.ndim != ndim:
            raise ValueError(f"likelihood has ndim={likelihood.ndim}, sampler was given ndim={ndim}")
        self.likelihood = likelihood
        self._seed = int(np.random.SeedSequence(seed).generate_state(1, dtype=np.uint64)[0])
        self._stream = None
        self._state = None
        self.good = 0
        self.use_graph = bool(use_graph)
        if depth not in (1, 2):
            raise ValueError("depth must be 1 or 2")
        self.depth = int(depth)
        super().__init__(nwalkers, ndim, likelihood.lnprob, mu=mu, tune=tune, tolerance=tolerance,
                         patience=patience, maxsteps=maxsteps, maxiter=maxiter, seed=seed)

    def reset(self):
        super().reset()
        self._state = None
        self.nexp = self.ncon = 0

    def run_mcmc(self, start, nsteps, progress=False, **_ignored):
        import torch
        from ._lib import RbvSliceTuning
        eng = self.likelihood.engine
        dev = eng.tdev
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        torch.cuda.current_stream(dev).synchronize()
        with torch.cuda.stream(self._stream):
            if start is None:
                if self._state is None:
                    raise ValueError("Cannot have `start=None` if run_mcmc has never been called.")
                coords_t, lnp_t = self._state
            else:
                X = np.array(start, dtype=np.float64, copy=True)
                if X.shape != (self.nwalkers, self.ndim):
                    raise ValueError("Incompatible input dimensions! Please provide array of shape (nwalkers, ndim)")
                coords_t = torch.as_tensor(X, device=dev)
                lnp_t = eng.lnprob_device(coords_t)
                self.ncall += self.nwalkers
                self.nbatches += 1
                if not bool(torch.isfinite(lnp_t).all()):
                    raise ValueError("Invalid walker initial positions! Initialise walkers from positions of "
                                     "finite log probability.")
            chain_t = torch.empty((nsteps, self.nwalkers, self.ndim), dtype=torch.float64, device=dev)
            lps_t = torch.empty((nsteps, self.nwalkers), dtype=torch.float64, device=dev)
            flag_t = torch.zeros(1, dtype=torch.int32, device=dev)
            tuning = RbvSliceTuning(mu=self.mu, tolerance=self.tolerance, tune=int(self.tune), good=int(self.good),
                                    patience=self.patience, maxsteps=self.maxsteps, maxiter=self.maxiter,
                                    depth=self.depth)
            mus = eng.slice_run(coords_t, lnp_t, nsteps, tuning, self._seed, self.iteration, chain_t, lps_t, flag_t,
                                use_graph=self.use_graph)
            self._stream.synchronize()
            if int(flag_t.item()) & 1:
                raise ValueError("Probability function returned NaN")
            was_tuning = self.tune
            self.mu, self.tune, self.good = float(tuning.mu), bool(tuning.tune), int(tuning.good)
            if was_tuning:
                self.mus.extend(float(m) for m in mus)
            self.ncall += int(tuning.n_calls)
            self.nbatches += int(tuning.n_batches)
            self.nexp += int(tuning.n_expansions)
            self.ncon += int(tuning.n_contractions)
            self._state = (coords_t, lnp_t)
            chain, lps = chain_t.cpu().numpy(), lps_t.cpu().numpy()
        self._hist_append(chain, lps)
        self.iteration += nsteps
        if nsteps:
            self._last = (chain[-1].copy(), lps[-1].copy())
        return self._last


class DistributedDeviceSliceSampler(DeviceEnsembleSliceSampler):
    """The device-resident ensemble slice sampler over several GPUs (one process per GPU, NCCL): with a communicator
    attached to the engine (``Engine.comm_init``, done here) ``rbv_slice_run`` splits the rows of every iteration's
    masked likelihood batch over the ranks and all-gathers their lnprob in place inside the library; walker state,
    directions, brackets and the adaptation of mu are replicated, every rank takes the same decisions from the same
    counter-based random streams, so the chain is the single-GPU chain bit for bit.  The seed (None = OS entropy) and
    the initial ensemble are taken from rank 0 and broadcast.  The per-half-step loop is host-polled by default (every
    rank reads the same replicated counters); ``RBVFIT_B200_SLICE_DIST_GRAPH=1`` keeps it a CUDA-graph WHILE node."""

    def __init__(self, nwalkers: int, ndim: int, likelihood, partition, **kwargs):
        from .dist import replicate_seed
        seed = kwargs.pop("seed", None)
        super().__init__(nwalkers, ndim, likelihood, seed=seed, **kwargs)
        self.partition = partition
        self._seed = replicate_seed(seed, partition.rank, partition.world, partition.group)
        eng = likelihood.engine
        if partition.world > 1 and not eng.has_comm:
            eng.comm_init(partition.group)

    def run_mcmc(self, start, nsteps, progress=False, **kw):
        from .dist import replicate_array
        if start is not None:
            p = self.partition
            start = replicate_array(start, p.rank, p.world, p.group)
        out = super().run_mcmc(start, nsteps, progress=progress, **kw)
        eng = self.likelihood.engine
        if getattr(eng, "peer_attached", False) and eng.peer_error():
            from ._lib import RbvError
            raise RbvError("the peer-memory all-gather gave up waiting for a rank (30 s without its rows)")
        return out


class _SliceSightlineView:
    """One sightline of a ``SightlineEnsembleSliceSampler`` behind ``DeviceEnsembleSliceSampler``'s (zeus's) accessor
    contract -- what a caller hands to the reference's ``UnifiedResults`` for that sightline."""

    def __init__(self, parent, index: int):
        self._p, self._s = parent, int(index)
        self.nwalkers, self.ndim = parent.nwalkers, parent.ndim

    @property
    def iteration(self):
        return self._p.iteration

    def get_chain(self, flat=False, thin=1, discard=0):
        return self._p.get_chain(flat=flat, thin=thin, discard=discard, sightline=self._s)

    def get_log_prob(self, flat=False, thin=1, discard=0):
        return self._p.get_log_prob(flat=flat, thin=thin, discard=discard, sightline=self._s)

    @property
    def chain(self):
        return self.get_chain()

    @property
    def acceptance_fraction(self):
        return self._p.acceptance_fraction[self._s]

    @property
    def efficiency(self):
        return float(self._p.efficiency[self._s])

    @property
    def mu(self):
        return float(self._p.mu[self._s])

    @property
    def tune(self):
        return bool(self._p.tune[self._s])

    @property
    def mus(self):
        return self._p.mus[:, self._s]

    @property
    def ncall(self):
        return int(self._p.ncall[self._s])

    @property
    def nexp(self):
        return int(self._p.nexp[self._s])

    @property
    def ncon(self):
        return int(self._p.ncon[self._s])

    @property
    def nbatches(self):
        return self._p.nbatches

    def get_autocorr_time(self, discard=0, thin=1, **kwargs):
        return thin * integrated_time(self.get_chain(discard=discard, thin=thin), **kwargs)

    def get_last_sample(self):
        last = self._p.get_last_sample()
        return None if last is None else (last[0][self._s], last[1][self._s])


class SightlineEnsembleSliceSampler(_ChunkedHistory):
    """Survey mode of ``DeviceEnsembleSliceSampler``: one zeus ensemble PER SIGHTLINE of a ``SightlineBatch``, all S
    ensembles advancing in lockstep on the device (``rbv_slice_run_sightlines``) -- the reference would run S separate
    ``vfit(..., sampler='zeus')`` fits one after the other.  Every iteration of a half-step is ONE sightline
    likelihood launch over the candidate rows of every sightline; a sightline whose walkers have finished masks its
    rows.  Each sightline keeps its own mu, tuning state and counters, exactly as S separate samplers would: its chain
    does not depend on the other sightlines, and sightline 0 reproduces ``DeviceEnsembleSliceSampler`` with the same
    seed on that sightline alone (same random streams, walker counter offset by s W for sightline s).  Sightlines
    shard across GPUs with no collective: every rank runs this sampler over its own ``SightlineBatch``.

    Accessors follow zeus (``arr[discard::thin]``): ``get_chain`` [steps, S, W, ndim], ``sightline=s`` -> [steps, W,
    ndim]; ``flat`` merges the steps and walkers of each sightline, never across sightlines.  Per sightline: ``mu``,
    ``tune``, ``ncall``, ``nexp``, ``ncon``, ``efficiency`` [S], ``mus`` [steps, S] (mu after every step),
    ``acceptance_fraction`` [S, W]; ``nbatches`` counts likelihood launches.  ``sightline(s)`` returns a one-sightline
    view with ``DeviceEnsembleSliceSampler``'s accessors."""

    def __init__(self, nwalkers: int, ndim: int, batch, mu: float = 1.0, tune: bool = True,
                 tolerance: float = 0.05, patience: int = 5, maxsteps: int = 10000, maxiter: int = 10000,
                 seed: Optional[int] = None, use_graph: bool = True, depth: int = 2):
        from .likelihood import SightlineBatch
        if not isinstance(batch, SightlineBatch):
            raise TypeError("SightlineEnsembleSliceSampler needs a SightlineBatch")
        if batch.ndim != ndim:
            raise ValueError(f"the sightline batch has ndim={batch.ndim}, sampler was given ndim={ndim}")
        if nwalkers < 2 * ndim or nwalkers % 2:
            raise ValueError("Please provide at least (2 * ndim) walkers, and an even number of them.")
        if not mu > 0:
            raise ValueError("mu must be positive")
        if depth not in (1, 2):
            raise ValueError("depth must be 1 or 2")
        self.batch = batch
        self.n_sightlines = int(batch.n_sightlines)
        self.nwalkers, self.ndim = int(nwalkers), int(ndim)
        self.mu0, self.tune0 = float(mu), bool(tune)
        self.tolerance, self.patience = float(tolerance), int(patience)
        self.maxsteps, self.maxiter = int(maxsteps), int(maxiter)
        self.use_graph, self.depth = bool(use_graph), int(depth)
        self._seed = int(np.random.SeedSequence(seed).generate_state(1, dtype=np.uint64)[0])
        self._stream = None
        self.reset()

    def reset(self):
        import torch
        S, W, nd = self.n_sightlines, self.nwalkers, self.ndim
        dev = self.batch.engine.tdev
        self._chain = np.empty((0, S, W, nd))
        self._log_prob = np.empty((0, S, W))
        self._mus = []
        self.iteration = 0
        self.nbatches = 0
        self._init_calls = np.zeros(S, dtype=np.int64)
        # per-sightline state of rbv_slice_run_sightlines, kept on the device between runs
        self._mu_t = torch.full((S,), self.mu0, dtype=torch.float64, device=dev)
        self._tune_good_t = torch.zeros((S, 2), dtype=torch.int32, device=dev)
        self._tune_good_t[:, 0] = int(self.tune0)
        self._totals_t = torch.zeros((S, 3), dtype=torch.int64, device=dev)
        self._pull_state()
        self._state = None
        self._last = None

    def _pull_state(self):
        self.mu = self._mu_t.cpu().numpy()
        tg = self._tune_good_t.cpu().numpy()
        self.tune, self.good = tg[:, 0] != 0, tg[:, 1].copy()
        tot = self._totals_t.cpu().numpy()
        self.nexp, self.ncon = tot[:, 0].copy(), tot[:, 1].copy()
        self.ncall = self._init_calls + tot[:, 2]

    def run_mcmc(self, start, nsteps, progress=False, **_ignored):
        """``start`` [S, W, ndim], or None to continue the last run; returns the last sample (coords [S, W, ndim],
        lnprob [S, W])."""
        import torch
        from ._lib import RbvSliceTuning
        eng = self.batch.engine
        dev = eng.tdev
        S, W, nd = self.n_sightlines, self.nwalkers, self.ndim
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        torch.cuda.current_stream(dev).synchronize()
        with torch.cuda.stream(self._stream):
            if start is None:
                if self._state is None:
                    raise ValueError("Cannot have `start=None` if run_mcmc has never been called.")
                coords_t, lnp_t = self._state
            else:
                X = np.array(start, dtype=np.float64, copy=True)
                if X.shape != (S, W, nd):
                    raise ValueError(f"Incompatible input dimensions! Please provide array of shape ({S}, {W}, {nd})")
                coords_t = torch.as_tensor(X, device=dev)
                lnp_t = eng.lnprob_sightlines_device(coords_t.view(S * W, nd), W).view(S, W)
                self._init_calls += W
                self.nbatches += 1
                if not bool(torch.isfinite(lnp_t).all()):
                    raise ValueError("Invalid walker initial positions! Initialise walkers from positions of "
                                     "finite log probability.")
            chain_t = torch.empty((nsteps, S, W, nd), dtype=torch.float64, device=dev)
            lps_t = torch.empty((nsteps, S, W), dtype=torch.float64, device=dev)
            mus_t = torch.empty((nsteps, S), dtype=torch.float64, device=dev)
            flag_t = torch.zeros(1, dtype=torch.int32, device=dev)
            tuning = RbvSliceTuning(tolerance=self.tolerance, patience=self.patience, maxsteps=self.maxsteps,
                                    maxiter=self.maxiter, depth=self.depth)
            try:
                eng.slice_run_sightlines(coords_t, lnp_t, nsteps, tuning, self._mu_t, self._tune_good_t,
                                         self._totals_t, self._seed, self.iteration, chain_t, lps_t, mus_t, flag_t,
                                         use_graph=self.use_graph)
            finally:
                self._stream.synchronize()
                self.nbatches += int(tuning.n_batches)
                self._pull_state()
            if int(flag_t.item()) & 1:
                raise ValueError("Probability function returned NaN")
            self._state = (coords_t, lnp_t)
            chain, lps = chain_t.cpu().numpy(), lps_t.cpu().numpy()
            self._mus.append(mus_t.cpu().numpy())
        self._hist_append(chain, lps)
        self.iteration += nsteps
        if nsteps:
            self._last = (chain[-1].copy(), lps[-1].copy())
        return self._last

    # ------------------------------------------------------------------ zeus-shaped accessors
    def _get(self, arr, discard, thin, flat, sightline):
        v = arr[discard::thin]
        if sightline is not None:
            v = v[:, int(sightline)]
            if flat:
                return v.reshape((-1,) + v.shape[2:])
            return v
        if flat:                                  # [S, steps * W, ...]: flat per sightline, never across sightlines
            v = np.swapaxes(v, 0, 1)
            return v.reshape((v.shape[0], -1) + v.shape[3:])
        return v

    def get_chain(self, flat=False, thin=1, discard=0, sightline=None):
        """[steps, S, W, ndim]; ``sightline=s`` -> [steps, W, ndim]; ``flat`` merges the steps and walkers of each
        sightline (never across sightlines)."""
        return self._get(self._chain, discard, thin, flat, sightline)

    def get_log_prob(self, flat=False, thin=1, discard=0, sightline=None):
        return self._get(self._log_prob, discard, thin, flat, sightline)

    @property
    def chain(self):
        return self._chain

    @property
    def mus(self):
        """[steps, S]: every sightline's mu after each step"""
        if not self._mus:
            return np.empty((0, self.n_sightlines))
        if len(self._mus) > 1:
            self._mus[:] = [np.concatenate(self._mus, axis=0)]
        return self._mus[0]

    @property
    def acceptance_fraction(self):
        """[S, W]: fraction of steps in which the walker moved (slice moves always move, so ~1)"""
        c = self._chain
        if len(c) < 2:
            return np.ones((self.n_sightlines, self.nwalkers))
        return np.mean(np.any(c[1:] != c[:-1], axis=3), axis=0)

    @property
    def efficiency(self):
        """[S]"""
        return self.iteration * self.nwalkers / np.maximum(self.ncall, 1)

    def sightline(self, index: int) -> _SliceSightlineView:
        if not 0 <= int(index) < self.n_sightlines:
            raise IndexError(index)
        return _SliceSightlineView(self, index)

    def get_last_sample(self):
        return self._last
