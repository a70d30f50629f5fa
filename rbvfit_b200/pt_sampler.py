"""Parallel-tempered ensemble sampling on the device, with the Bayesian evidence by thermodynamic integration.

The reference offers emcee and zeus only (vfit_mcmc.py:408-440) and no evidence estimate.  The algorithm here is
ptemcee's (Vousden, Farr & Mandel 2016, MNRAS 455, 1919): T stretch-move ensembles sample prior x L^beta_t on a
ladder 1 = beta_0 > beta_1 > ... >= 0 and exchange states between adjacent temperatures once per step, so the cold
(beta = 1) chain can cross between modes that a single ensemble never leaves.  The whole step runs on the device
(``rbv_pt_run``, rbvfit_b200/csrc/rbv_pt.cuh); with T = 1 it is ``DeviceEnsembleSampler``'s chain bit for bit.

The mean log-likelihood the run records at every temperature gives

    ln Z = int_0^1 <ln L>_beta d beta

(thermodynamic integration); ``log_evidence`` evaluates it with the trapezoid rule and its derivative correction
(Friel, Hurn & Wyse 2014: d<ln L>/d beta = Var(ln L)), Z being normalised to the box prior of the bounds.

``SightlineParallelTemperingSampler`` runs one ladder per sightline of a ``SightlineBatch`` in one device loop
(``rbv_pt_run_sightlines``) and accumulates the mean and variance of ln L of every sightline and temperature on the
device, so the evidence of a survey never needs its [steps, S, T, W] lnprob chain (``evidence_from_moments``).
"""
from __future__ import annotations

import warnings
from typing import Optional

import numpy as np

from .sampler import integrated_time, walkers_independent


def default_betas(ndim: int, beta_min: float = 1e-6) -> np.ndarray:
    """Geometric ladder from 1 down past ``beta_min`` with ratio 1 + 2 sqrt(ln 4 / ndim), then beta = 0 (the hottest
    ensemble samples the prior).  The ratio is the Gaussian rule for 25 % swap acceptance that ptemcee uses beyond its
    table for small ndim (DESIGN.md section 18)."""
    if ndim < 1 or not beta_min > 0.0:
        raise ValueError("need ndim >= 1 and beta_min > 0")
    r = 1.0 + 2.0 * np.sqrt(np.log(4.0) / ndim)
    betas = [1.0]
    while betas[-1] >= beta_min:
        betas.append(betas[-1] / r)
    betas.append(0.0)
    return np.array(betas)


def check_betas(betas) -> np.ndarray:
    """The ladder as float64, or ValueError: 1-D, betas[0] = 1, strictly decreasing, >= 0."""
    b = np.array(betas, dtype=np.float64, copy=True)
    if b.ndim != 1 or len(b) < 1:
        raise ValueError("betas must be a non-empty 1-D array")
    if b[0] != 1.0:
        raise ValueError("betas[0] must be 1 (the posterior itself)")
    if not (np.all(np.diff(b) < 0) and np.all(b >= 0)):
        raise ValueError("betas must be strictly decreasing and >= 0")
    return b


def _ti(betas, E, V):
    """Trapezoid in beta with the derivative correction; [0, beta_min] closed with the hottest E and V."""
    if betas[-1] > 0:
        betas, E, V = np.append(betas, 0.0), np.append(E, E[-1]), np.append(V, V[-1])
    db = betas[:-1] - betas[1:]
    return float(np.sum(db / 2.0 * (E[:-1] + E[1:])) - np.sum(db ** 2 / 12.0 * (V[:-1] - V[1:])))


def evidence_from_moments(betas, E, V):
    """(lnZ, dlnZ) from the mean ``E`` [T] and variance ``V`` [T] of the untempered log-likelihood at each
    temperature of the ladder ``betas`` [T].  dlnZ is ptemcee's: |lnZ - lnZ(every other temperature)|, which also
    exposes the discretisation error of a coarse ladder."""
    betas = check_betas(betas)
    E, V = np.asarray(E, dtype=np.float64), np.asarray(V, dtype=np.float64)
    if E.shape != betas.shape or V.shape != betas.shape:
        raise ValueError(f"E and V must be [{len(betas)}]")
    lnz = _ti(betas, E, V)
    if betas[-1] > 0:
        coarse = np.arange(0, len(betas), 2)
    else:        # keep beta = 0 itself
        coarse = np.append(np.arange(0, len(betas) - 1, 2), len(betas) - 1)
    lnz2 = _ti(betas[coarse], E[coarse], V[coarse])
    return lnz, abs(lnz - lnz2)


def log_evidence(betas, logl):
    """(lnZ, dlnZ) from ``logl`` [steps, T, W], the untempered log-likelihood at each temperature of the ladder
    ``betas`` [T] (``evidence_from_moments`` of its per-temperature mean and variance)."""
    betas = check_betas(betas)
    logl = np.asarray(logl, dtype=np.float64)
    if logl.ndim != 3 or logl.shape[1] != len(betas) or logl.shape[0] * logl.shape[2] == 0:
        raise ValueError(f"logl must be [steps, {len(betas)}, walkers] with at least one sample")
    x = np.swapaxes(logl, 0, 1).reshape(len(betas), -1)
    return evidence_from_moments(betas, x.mean(axis=1), x.var(axis=1))


class _TemperatureView:
    """One recorded temperature behind emcee's accessor contract (what ``vfit`` / ``UnifiedResults`` read from
    ``fitter.sampler``, core/unified_results.py:163-299).  ``get_log_prob`` is the untempered lnprob."""

    def __init__(self, parent, temp: int):
        self._p, self._t = parent, int(temp)
        self.nwalkers, self.ndim = parent.nwalkers, parent.ndim

    @property
    def iteration(self):
        return self._p.iteration

    def get_chain(self, discard=0, thin=1, flat=False):
        return self._p.get_chain(discard=discard, thin=thin, flat=flat, temp=self._t)

    def get_log_prob(self, discard=0, thin=1, flat=False):
        v = self._p.get_log_like(discard=discard, thin=thin)[:, self._t]
        return v.reshape(-1) if flat else v

    @property
    def chain(self):
        return np.swapaxes(self.get_chain(), 0, 1)

    @property
    def flatchain(self):
        return self.get_chain(flat=True)

    @property
    def lnprobability(self):
        return self.get_log_prob().T

    @property
    def acceptance_fraction(self):
        return self._p.acceptance_fraction[self._t]

    def get_autocorr_time(self, discard=0, thin=1, **kwargs):
        return thin * integrated_time(self.get_chain(discard=discard, thin=thin), **kwargs)


class DeviceParallelTemperingSampler:
    """Parallel-tempered stretch-move sampler on the device (``rbv_pt_run``).  ``likelihood`` is a
    ``GpuLikelihood``; ``betas`` the ladder (default ``default_betas(ndim)``).  Random numbers come from the
    counter-based streams of ``DeviceEnsembleSampler`` keyed by ``seed``, so a run is reproducible and
    ``run_mcmc(None, n)`` continues it without changing the stream of a single long run.

    ``run_mcmc(p0, nsteps, adapt=False, n_record=1)``: ``p0`` is [T, W, ndim], or [W, ndim] replicated to every
    temperature; ``adapt`` adjusts the interior of the ladder after every step (ptemcee's rule; burn-in only, it
    breaks detailed balance); the coordinates of the ``n_record`` coldest temperatures are kept, lnprob of all."""

    def __init__(self, nwalkers: int, ndim: int, likelihood, betas=None, a: float = 2.0, seed: Optional[int] = None,
                 use_graph: bool = True, adaptation_lag: float = 10000.0, adaptation_time: float = 100.0):
        if not hasattr(likelihood, "engine"):
            raise TypeError("DeviceParallelTemperingSampler needs a GpuLikelihood (the log-probability must run on "
                            "the device)")
        if likelihood.ndim != ndim:
            raise ValueError(f"likelihood has ndim={likelihood.ndim}, sampler was given ndim={ndim}")
        if nwalkers < 2:
            raise ValueError("need at least two walkers per temperature")
        if not a > 1.0:
            raise ValueError("the stretch scale a must be > 1")
        if not (adaptation_lag > 0 and adaptation_time > 0):
            raise ValueError("adaptation_lag and adaptation_time must be > 0")
        self.likelihood = likelihood
        self.nwalkers, self.ndim, self.a = int(nwalkers), int(ndim), float(a)
        self._betas0 = check_betas(default_betas(ndim) if betas is None else betas)
        self.ntemps = len(self._betas0)
        self.use_graph = bool(use_graph)
        self.adaptation_lag, self.adaptation_time = float(adaptation_lag), float(adaptation_time)
        self._seed = int(np.random.SeedSequence(seed).generate_state(1, dtype=np.uint64)[0])
        self._stream = None
        self.reset()

    def reset(self):
        T, W = self.ntemps, self.nwalkers
        self._chunks = []           # per run: chain [n, n_record, W, ndim], logl [n, T, W], betas [n, T], adapted [n]
        self._accepted = np.zeros((T, W))
        self._swaps = np.zeros(max(T - 1, 0))
        self._betas = self._betas0.copy()
        self.iteration = 0
        self.adapt_steps = 0
        self.n_record = None
        self._state = None

    def run_mcmc(self, initial_state, nsteps, adapt=False, n_record=1, skip_initial_state_check=False, **_ignored):
        import torch
        eng = self.likelihood.engine
        dev = eng.tdev
        T, W, nd = self.ntemps, self.nwalkers, self.ndim
        nsteps, n_record = int(nsteps), int(n_record)
        if nsteps < 0:
            raise ValueError("nsteps must be >= 0")
        if not 1 <= n_record <= T:
            raise ValueError(f"n_record must lie in 1 .. {T}")
        if self.n_record is not None and n_record != self.n_record:
            raise ValueError(f"this run records n_record={self.n_record} temperatures; reset() to change it")
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        torch.cuda.current_stream(dev).synchronize()
        with torch.cuda.stream(self._stream):
            if initial_state is None:
                if self._state is None:
                    raise ValueError("Cannot have `initial_state=None` if run_mcmc has never been called.")
                coords_t, lnp_t, betas_t = self._state
            else:
                coords = np.array(initial_state, dtype=np.float64, copy=True)
                if coords.shape == (W, nd):
                    coords = np.broadcast_to(coords, (T, W, nd)).copy()
                if coords.shape != (T, W, nd):
                    raise ValueError("incompatible input dimensions {0}: need [{1}, {2}, {3}] or [{2}, {3}]".format(
                        coords.shape, T, W, nd))
                if np.any(np.isinf(coords)):
                    raise ValueError("At least one parameter value was infinite")
                if np.any(np.isnan(coords)):
                    raise ValueError("At least one parameter value was NaN")
                if not skip_initial_state_check and not all(walkers_independent(c) for c in coords):
                    raise ValueError("Initial state has a large condition number. Make sure that your walkers are "
                                     "linearly independent for the best performance")
                coords_t = torch.as_tensor(coords, device=dev)
                lnp_t = eng.lnprob_device(coords_t.view(T * W, nd)).view(T, W).contiguous()
                if bool(torch.isnan(lnp_t).any()):
                    raise ValueError("Probability function returned NaN")
                betas_t = torch.as_tensor(self._betas, device=dev).clone()
            nacc_t = torch.zeros((T, W), dtype=torch.int32, device=dev)
            nswap_t = torch.zeros(max(T - 1, 1), dtype=torch.int64, device=dev)
            flag_t = torch.zeros(1, dtype=torch.int32, device=dev)
            bh_t = torch.empty((nsteps, T), dtype=torch.float64, device=dev)
            kw = dict(adapt=adapt, adaptation_lag=self.adaptation_lag, adaptation_time=self.adaptation_time,
                      adapt_steps_done=self.adapt_steps, n_record=n_record)
            if self.use_graph and nsteps >= 4:
                # the chain streams to the host in blocks while the run goes on (the chain sink)
                chain, logl = eng.pt_run_to_host(coords_t, lnp_t, betas_t, nsteps, self.a, self._seed, self.iteration,
                                                 bh_t, nacc_t, nswap_t, flag_t, **kw)
            else:
                chain_t = torch.empty((nsteps, n_record, W, nd), dtype=torch.float64, device=dev)
                logl_t = torch.empty((nsteps, T, W), dtype=torch.float64, device=dev)
                eng.pt_run(coords_t, lnp_t, betas_t, nsteps, self.a, self._seed, self.iteration, chain_t, logl_t,
                           bh_t, nacc_t, nswap_t, flag_t, use_graph=self.use_graph, **kw)
                chain, logl = chain_t.cpu().numpy(), logl_t.cpu().numpy()
            self._stream.synchronize()
            if int(flag_t.item()) & 1:
                raise ValueError("Probability function returned NaN")
            self._state = (coords_t, lnp_t, betas_t)
            self._accepted += nacc_t.cpu().numpy()
            if T > 1:
                self._swaps += nswap_t.cpu().numpy()
            self._betas = betas_t.cpu().numpy()
            bh = bh_t.cpu().numpy()
        self.n_record = n_record
        self._chunks.append((chain, logl, bh, np.full(nsteps, bool(adapt))))
        self.iteration += nsteps
        if adapt:
            self.adapt_steps += nsteps
        return (chain[-1].copy(), logl[-1].copy()) if nsteps else None

    # -- accessors
    def _all(self):
        """(chain [steps, n_record, W, ndim], logl [steps, T, W], beta history [steps, T], adapted [steps]): the
        per-run chunks are concatenated once, when first read."""
        if len(self._chunks) != 1:
            T, W, nd = self.ntemps, self.nwalkers, self.ndim
            if not self._chunks:
                return (np.empty((0, self.n_record or 1, W, nd)), np.empty((0, T, W)), np.empty((0, T)),
                        np.empty(0, dtype=bool))
            self._chunks = [tuple(np.concatenate([c[k] for c in self._chunks]) for k in range(4))]
        return self._chunks[0]

    @staticmethod
    def _sel(v, discard, thin):
        return v[discard + thin - 1:: thin]

    def get_chain(self, discard=0, thin=1, flat=False, temp=0):
        """[steps, W, ndim] of temperature ``temp`` (0 = beta 1); ``flat`` merges steps and walkers."""
        if not 0 <= int(temp) < self.ntemps:
            raise ValueError(f"temp must lie in 0 .. {self.ntemps - 1}")
        if self.n_record is not None and int(temp) >= self.n_record:
            raise ValueError(f"temperature {temp} was not recorded: run with n_record > {temp}")
        v = self._sel(self._all()[0], discard, thin)[:, int(temp)]
        return v.reshape((-1, self.ndim)) if flat else v

    def get_log_like(self, discard=0, thin=1, flat=False):
        """[steps, T, W] untempered log-likelihood (lnprob) of every temperature; ``flat`` -> [T, steps * W]."""
        v = self._sel(self._all()[1], discard, thin)
        return np.swapaxes(v, 0, 1).reshape(self.ntemps, -1) if flat else v

    @property
    def betas(self) -> np.ndarray:
        """The current ladder (adapted by runs with ``adapt=True``)."""
        return self._betas.copy()

    @property
    def beta_history(self) -> np.ndarray:
        """[steps, T]: the ladder each step ran with."""
        return self._all()[2]

    @property
    def acceptance_fraction(self) -> np.ndarray:
        """[T, W] accepted stretch moves per step."""
        return self._accepted / max(self.iteration, 1)

    @property
    def tswap_acceptance_fraction(self) -> np.ndarray:
        """[T - 1] accepted swaps of pair (i, i + 1) per step and walker."""
        return self._swaps / max(self.iteration * self.nwalkers, 1)

    def cold(self) -> _TemperatureView:
        """emcee-shaped view of the beta = 1 chain."""
        return _TemperatureView(self, 0)

    def log_evidence_estimate(self, discard=0):
        """(lnZ, dlnZ) by thermodynamic integration over the steps after ``discard`` (see ``log_evidence``).
        Raises ValueError when a kept step ran with ``adapt=True``: adaptation breaks detailed balance."""
        _chain, logl, bh, adapted = self._all()
        discard = int(discard)
        if discard < 0 or discard >= len(logl):
            raise ValueError(f"discard must lie in 0 .. {len(logl) - 1} (steps run: {len(logl)})")
        if np.any(adapted[discard:]):
            raise ValueError("the kept steps include steps run with adapt=True: discard them (adaptation breaks "
                             "detailed balance) or run more steps with adapt=False")
        return log_evidence(bh[discard], logl[discard:])

    def get_last_sample(self):
        return None if self._state is None else tuple(t.cpu().numpy() for t in self._state[:2])


def _ladders(betas, S, ndim) -> np.ndarray:
    """[S, T] ladders from None (``default_betas(ndim)``), one [T] ladder shared by every sightline, or [S, T]."""
    if betas is None:
        return np.tile(default_betas(ndim), (S, 1))
    b = np.asarray(betas, dtype=np.float64)
    if b.ndim == 1:
        return np.tile(check_betas(b), (S, 1))
    if b.ndim != 2 or b.shape[0] != S:
        raise ValueError(f"betas must be [T] or [{S}, T]")
    out = np.empty_like(b)
    for s in range(S):
        try:
            out[s] = check_betas(b[s])
        except ValueError as e:
            raise ValueError(f"sightline {s}: {e}") from None
    return out


class _SightlinePtView:
    """One sightline of a ``SightlineParallelTemperingSampler`` behind ``DeviceParallelTemperingSampler``'s
    accessors; ``log_evidence_estimate()`` is that sightline's (lnZ, dlnZ) from the device moments."""

    def __init__(self, parent, index: int):
        self._p, self._s = parent, int(index)
        self.nwalkers, self.ndim, self.ntemps = parent.nwalkers, parent.ndim, parent.ntemps

    @property
    def iteration(self):
        return self._p.iteration

    @property
    def n_record(self):
        return self._p.n_record

    def get_chain(self, discard=0, thin=1, flat=False, temp=0):
        return self._p.get_chain(discard=discard, thin=thin, flat=flat, temp=temp, sightline=self._s)

    def get_log_like(self, discard=0, thin=1, flat=False):
        return self._p.get_log_like(discard=discard, thin=thin, flat=flat, sightline=self._s)

    @property
    def betas(self) -> np.ndarray:
        return self._p.betas[self._s]

    @property
    def beta_history(self) -> np.ndarray:
        return self._p.beta_history[:, self._s]

    @property
    def acceptance_fraction(self) -> np.ndarray:
        return self._p.acceptance_fraction[self._s]

    @property
    def tswap_acceptance_fraction(self) -> np.ndarray:
        return self._p.tswap_acceptance_fraction[self._s]

    def cold(self) -> _TemperatureView:
        return _TemperatureView(self, 0)

    def log_evidence_estimate(self):
        lnz, dlnz = self._p.log_evidence_estimate(sightlines=[self._s])
        return float(lnz[0]), float(dlnz[0])

    def get_last_sample(self):
        last = self._p.get_last_sample()
        return None if last is None else tuple(v[self._s] for v in last)


class SightlineParallelTemperingSampler:
    """Survey-mode parallel tempering (``rbv_pt_run_sightlines``): ``DeviceParallelTemperingSampler`` for every
    sightline of a ``SightlineBatch``, all S ladders of T ensembles advancing in lockstep in one device loop.  Sightline
    s uses the random streams of a one-sightline run with every walker counter offset by s T W, so sightline 0
    reproduces ``DeviceParallelTemperingSampler`` on that sightline alone with the same seed, and sightlines never mix.

    ``betas`` is one ladder [T] every sightline starts from, or [S, T] (default ``default_betas(ndim)``).  The
    evidence comes from moments of ln L accumulated on the device ([S, T] means and variances), not from the lnprob
    chain: ``run_mcmc(p0, nsteps, adapt=False, accumulate=None, n_record=1)`` accumulates when ``accumulate`` (default
    ``not adapt``; adaptation breaks detailed balance, so both at once are refused).  A burn-in is therefore a run
    with ``accumulate=False`` (or ``reset_evidence()`` after it).  ``p0`` is [S, W, ndim] (replicated to every
    temperature) or [S, T, W, ndim].

    ``record_chain`` keeps the coordinates of the ``n_record`` coldest temperatures on the host, ``record_log_like``
    the lnprob of every temperature ([steps, S, T, W]: large for a survey, off by default).  ``sightline(s)``
    returns a view with ``DeviceParallelTemperingSampler``'s accessors."""

    def __init__(self, nwalkers: int, ndim: int, batch, betas=None, a: float = 2.0, seed: Optional[int] = None,
                 use_graph: bool = True, record_chain: bool = True, record_log_like: bool = False,
                 adaptation_lag: float = 10000.0, adaptation_time: float = 100.0):
        if not hasattr(batch, "engine") or not hasattr(batch, "n_sightlines"):
            raise TypeError("SightlineParallelTemperingSampler needs a SightlineBatch")
        if batch.ndim != ndim:
            raise ValueError(f"the sightline batch has ndim={batch.ndim}, sampler was given ndim={ndim}")
        if nwalkers < 2:
            raise ValueError("need at least two walkers per temperature")
        if not a > 1.0:
            raise ValueError("the stretch scale a must be > 1")
        if not (adaptation_lag > 0 and adaptation_time > 0):
            raise ValueError("adaptation_lag and adaptation_time must be > 0")
        self.batch = batch
        self.n_sightlines = int(batch.n_sightlines)
        self.nwalkers, self.ndim, self.a = int(nwalkers), int(ndim), float(a)
        self._betas0 = _ladders(betas, self.n_sightlines, self.ndim)
        self.ntemps = self._betas0.shape[1]
        self.use_graph = bool(use_graph)
        self.record_chain, self.record_log_like = bool(record_chain), bool(record_log_like)
        self.adaptation_lag, self.adaptation_time = float(adaptation_lag), float(adaptation_time)
        self._seed = int(np.random.SeedSequence(seed).generate_state(1, dtype=np.uint64)[0])
        self._stream = None
        self.reset()

    def reset(self):
        S, T, W = self.n_sightlines, self.ntemps, self.nwalkers
        self._chunks = []           # per run: chain, logl (or None), betas [n, S, T], adapted [n]
        self._accepted = np.zeros((S, T, W))
        self._swaps = np.zeros((S, max(T - 1, 0)))
        self._betas = self._betas0.copy()
        self.iteration = 0
        self.adapt_steps = 0
        self.n_record = None
        self._state = None
        self.reset_evidence()

    def reset_evidence(self):
        """Drop the accumulated moments (e.g. after a burn-in run)."""
        self._ti = np.zeros((self.n_sightlines, self.ntemps, 3))
        self._ti_betas = None
        self.evidence_steps = 0

    def run_mcmc(self, initial_state, nsteps, adapt=False, accumulate=None, n_record=1,
                 skip_initial_state_check=False, **_ignored):
        S, T, W, nd = self.n_sightlines, self.ntemps, self.nwalkers, self.ndim
        nsteps, n_record = int(nsteps), int(n_record)
        if accumulate is None:
            accumulate = not adapt
        if adapt and accumulate:
            raise ValueError("adapt and accumulate cannot both be set: adaptation breaks detailed balance, so its steps "
                             "must not enter the evidence")
        if nsteps < 0:
            raise ValueError("nsteps must be >= 0")
        if not 1 <= n_record <= T:
            raise ValueError(f"n_record must lie in 1 .. {T}")
        if self.n_record is not None and n_record != self.n_record:
            raise ValueError(f"this run records n_record={self.n_record} temperatures; reset() to change it")
        if accumulate and self._ti_betas is not None and not np.array_equal(self._ti_betas, self._betas):
            raise ValueError("the ladders changed since the moments began accumulating: reset_evidence() first")
        import torch
        eng = self.batch.engine
        dev = eng.tdev
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        torch.cuda.current_stream(dev).synchronize()
        with torch.cuda.stream(self._stream):
            if initial_state is None:
                if self._state is None:
                    raise ValueError("Cannot have `initial_state=None` if run_mcmc has never been called.")
                coords_t, lnp_t, betas_t = self._state
            else:
                coords = np.array(initial_state, dtype=np.float64, copy=True)
                if coords.shape == (S, W, nd):
                    coords = np.broadcast_to(coords[:, None], (S, T, W, nd)).copy()
                if coords.shape != (S, T, W, nd):
                    raise ValueError("incompatible input dimensions {0}: need [{1}, {2}, {3}, {4}] or [{1}, {3}, {4}]"
                                     .format(coords.shape, S, T, W, nd))
                if not np.all(np.isfinite(coords)):
                    raise ValueError("At least one parameter value was infinite or NaN")
                if not skip_initial_state_check and not all(walkers_independent(c)
                                                            for c in coords.reshape(S * T, W, nd)):
                    raise ValueError("Initial state has a large condition number. Make sure that your walkers are "
                                     "linearly independent for the best performance")
                coords_t = torch.as_tensor(coords, device=dev)
                lnp_t = eng.lnprob_sightlines_device(coords_t.view(S * T * W, nd), T * W).view(S, T, W).contiguous()
                if bool(torch.isnan(lnp_t).any()):
                    raise ValueError("Probability function returned NaN")
                betas_t = torch.as_tensor(self._betas, device=dev).clone()
            nacc_t = torch.zeros((S, T, W), dtype=torch.int32, device=dev)
            nswap_t = torch.zeros((S, max(T - 1, 1)), dtype=torch.int64, device=dev)
            flag_t = torch.zeros(1, dtype=torch.int32, device=dev)
            bh_t = torch.empty((nsteps, S, T), dtype=torch.float64, device=dev)
            ti_t = torch.as_tensor(self._ti, device=dev).clone() if accumulate else None
            kw = dict(adapt=adapt, adaptation_lag=self.adaptation_lag, adaptation_time=self.adaptation_time,
                      adapt_steps_done=self.adapt_steps, n_record=n_record)
            rc, rl = self.record_chain, self.record_log_like
            if self.use_graph and nsteps >= 4 and (rc or rl):
                # the chain streams to the host in blocks while the run goes on (the chain sink)
                chain, logl = eng.pt_run_sightlines_to_host(coords_t, lnp_t, betas_t, nsteps, self.a, self._seed,
                                                            self.iteration, bh_t, ti_t, nacc_t, nswap_t, flag_t,
                                                            record_chain=rc, record_log_like=rl, **kw)
            else:
                chain_t = torch.empty((nsteps, S, n_record, W, nd), dtype=torch.float64, device=dev) if rc else None
                logl_t = torch.empty((nsteps, S, T, W), dtype=torch.float64, device=dev) if rl else None
                eng.pt_run_sightlines(coords_t, lnp_t, betas_t, nsteps, self.a, self._seed, self.iteration, chain_t,
                                      logl_t, bh_t, ti_t, nacc_t, nswap_t, flag_t, use_graph=self.use_graph, **kw)
                chain = chain_t.cpu().numpy() if rc else None
                logl = logl_t.cpu().numpy() if rl else None
            self._stream.synchronize()
            if int(flag_t.item()) & 1:
                raise ValueError("Probability function returned NaN")
            self._state = (coords_t, lnp_t, betas_t)
            self._accepted += nacc_t.cpu().numpy()
            if T > 1:
                self._swaps += nswap_t.cpu().numpy()
            if accumulate and nsteps:
                self._ti = ti_t.cpu().numpy()
                self._ti_betas = self._betas.copy()
                self.evidence_steps += nsteps
            self._betas = betas_t.cpu().numpy()
            bh = bh_t.cpu().numpy()
        self.n_record = n_record
        self._chunks.append((chain, logl, bh, np.full(nsteps, bool(adapt))))
        self.iteration += nsteps
        if adapt:
            self.adapt_steps += nsteps
        if not nsteps:
            return None
        return (chain[-1].copy() if chain is not None else None, logl[-1].copy() if logl is not None else None)

    # -- accessors
    def _all(self, k):
        """Field k of the concatenated per-run chunks (0 chain, 1 logl, 2 beta history, 3 adapted)."""
        if len(self._chunks) != 1:
            S, T, W, nd = self.n_sightlines, self.ntemps, self.nwalkers, self.ndim
            if not self._chunks:
                return (np.empty((0, S, self.n_record or 1, W, nd)), np.empty((0, S, T, W)), np.empty((0, S, T)),
                        np.empty(0, dtype=bool))[k]
            self._chunks = [tuple(None if self._chunks[0][j] is None else
                                  np.concatenate([c[j] for c in self._chunks]) for j in range(4))]
        return self._chunks[0][k]

    @staticmethod
    def _sel(v, discard, thin):
        return v[discard + thin - 1:: thin]

    def get_chain(self, discard=0, thin=1, flat=False, temp=0, sightline=None):
        """[steps, S, W, ndim] of temperature ``temp`` (0 = beta 1); ``sightline=s`` -> [steps, W, ndim]; ``flat``
        merges the steps and walkers of each sightline (never across sightlines)."""
        if not self.record_chain:
            raise ValueError("the chain was not recorded (record_chain=False)")
        if not 0 <= int(temp) < self.ntemps:
            raise ValueError(f"temp must lie in 0 .. {self.ntemps - 1}")
        if self.n_record is not None and int(temp) >= self.n_record:
            raise ValueError(f"temperature {temp} was not recorded: run with n_record > {temp}")
        v = self._sel(self._all(0), discard, thin)[:, :, int(temp)]
        if sightline is not None:
            v = v[:, int(sightline)]
            return v.reshape((-1, self.ndim)) if flat else v
        if flat:
            return np.swapaxes(v, 0, 1).reshape(self.n_sightlines, -1, self.ndim)
        return v

    def get_log_like(self, discard=0, thin=1, flat=False, sightline=None):
        """[steps, S, T, W] untempered log-likelihood (lnprob) of every temperature (``record_log_like``);
        ``sightline=s`` -> [steps, T, W]; ``flat`` -> [S, T, steps * W] ([T, steps * W] for one sightline)."""
        if not self.record_log_like:
            raise ValueError("the lnprob chain was not recorded (record_log_like=False)")
        v = self._sel(self._all(1), discard, thin)
        if sightline is not None:
            v = v[:, int(sightline)]
            return np.swapaxes(v, 0, 1).reshape(self.ntemps, -1) if flat else v
        return np.moveaxis(v, 0, 2).reshape(self.n_sightlines, self.ntemps, -1) if flat else v

    @property
    def betas(self) -> np.ndarray:
        """[S, T] the current ladders (adapted by runs with ``adapt=True``)."""
        return self._betas.copy()

    @property
    def beta_history(self) -> np.ndarray:
        """[steps, S, T]: the ladders each step ran with."""
        return self._all(2)

    @property
    def acceptance_fraction(self) -> np.ndarray:
        """[S, T, W] accepted stretch moves per step."""
        return self._accepted / max(self.iteration, 1)

    @property
    def tswap_acceptance_fraction(self) -> np.ndarray:
        """[S, T - 1] accepted swaps of pair (i, i + 1) per step and walker."""
        return self._swaps / max(self.iteration * self.nwalkers, 1)

    @property
    def ti_moments(self) -> np.ndarray:
        """[S, T, 3] the accumulated (n, mean, M2) of ln L (Var = M2 / n)."""
        return self._ti.copy()

    def log_evidence_estimate(self, sightlines=None):
        """(lnZ [S], dlnZ [S]) by thermodynamic integration of the moments accumulated on the device (see
        ``evidence_from_moments``).  A sightline whose moments are not finite (a walker that stayed outside the
        bounds, for instance) gets NaN, and one warning names every such sightline."""
        if self.evidence_steps == 0:
            raise ValueError("no moments accumulated: run_mcmc with accumulate=True (the default without adapt)")
        idx = np.arange(self.n_sightlines) if sightlines is None else np.asarray(sightlines, dtype=np.int64)
        lnz, dlnz = np.full(len(idx), np.nan), np.full(len(idx), np.nan)
        bad = []
        for j, s in enumerate(idx):
            n, E, M2 = self._ti[s, :, 0], self._ti[s, :, 1], self._ti[s, :, 2]
            V = M2 / n
            if not (np.all(np.isfinite(E)) and np.all(np.isfinite(V))):
                bad.append(int(s))
                continue
            lnz[j], dlnz[j] = evidence_from_moments(self._ti_betas[s], E, V)
        if bad:
            warnings.warn(f"non-finite ln L moments (lnZ = NaN) on sightlines {bad}", RuntimeWarning)
        return lnz, dlnz

    def sightline(self, index: int) -> _SightlinePtView:
        if not 0 <= int(index) < self.n_sightlines:
            raise IndexError(index)
        return _SightlinePtView(self, index)

    def get_last_sample(self):
        """(coords [S, T, W, ndim], lnprob [S, T, W]) of the current state, or None before the first run."""
        return None if self._state is None else tuple(t.cpu().numpy() for t in self._state[:2])
