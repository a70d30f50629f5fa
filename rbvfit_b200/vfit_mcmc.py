"""GPU drop-in for rbvfit's ``vfit`` fitter (reference: src/rbvfit/vfit_mcmc.py:102-692) and ``set_bounds``
(:695-787, traditional branch).

Same constructor, attributes and methods as the reference for the likelihood path and its immediate
callers: ``lnprior / lnlike / lnprob``, ``optimize_guess``, ``_initialize_walkers``, ``runmcmc``,
``compute_best_theta``, ``get_samples``.  What changes is *where the batch is*: every place the reference
loops over theta rows one at a time (walker initialisation :442-466, the finite-difference gradient of
L-BFGS-B :355-360, the sampler's half-steps :536-540) hands the whole batch to the GPU in one call.
``use_pool=True`` is accepted and ignored -- a CUDA context must not be forked; the device batch replaces
the process pool.
"""
from __future__ import annotations

import copy
import warnings
from typing import Dict

import numpy as np

from .likelihood import GpuLikelihood
from .sampler import DeviceEnsembleSampler, EnsembleSampler


def gelman_rubin(chains) -> np.ndarray:
    """Gelman-Rubin potential scale reduction per parameter; ``chains`` is [n_chains, n_steps, ndim] (the walkers as
    chains, the call the reference makes: zeus.diagnostics.gelman_rubin(chain.transpose(1, 0, 2)), vfit_mcmc.py:637-639).
    W = mean within-chain variance, B/n = variance of the chain means, V = (n-1)/n W + B/n + B/(n m), R = sqrt(V / W)."""
    x = np.asarray(chains, dtype=np.float64)
    m, n = x.shape[0], x.shape[1]
    if m < 2 or n < 2:
        raise ValueError("need at least two chains of at least two steps")
    means = x.mean(axis=1)
    W = x.var(axis=1, ddof=1).mean(axis=0)
    B_over_n = means.var(axis=0, ddof=1)
    V = (n - 1.0) / n * W + B_over_n + B_over_n / m
    return np.sqrt(V / W)


class vfit:
    def __init__(self, instrument_data: Dict, theta, lb, ub, no_of_Chain=50, no_of_steps=1000,
                 perturbation=1e-4, sampler="emcee", skip_initial_state_check=False, device=None, seed=None,
                 device_sampler=True, betas=None):
        self._validate_unified_instrument_data(instrument_data)
        self._validate_guesses(theta, lb, ub)
        self.theta = np.asarray(theta)
        self.lb = np.asarray(lb)
        self.ub = np.asarray(ub)
        self._like = GpuLikelihood(instrument_data, self.lb, self.ub, device=device)   # _compile_models
        self.instrument_data = self._like.instrument_data
        self.instrument_configs = self._extract_configs(instrument_data)
        self.multi_instrument = len(instrument_data) > 1
        self.no_of_Chain = no_of_Chain
        self.no_of_steps = no_of_steps
        self.perturbation = perturbation
        self.skip_initial_state_check = skip_initial_state_check
        self.sampler_name = sampler.lower()
        if self.sampler_name not in ["emcee", "zeus", "pt"]:
            raise ValueError(f"Unknown sampler '{sampler}'. Use 'emcee', 'zeus' or 'pt'.")
        if self.sampler_name == "pt" and not device_sampler:
            raise ValueError("sampler='pt' (parallel tempering) runs on the device only")
        self.betas = betas                 # sampler='pt': the temperature ladder (None: default_betas(ndim))
        self.pt_sampler = None             # sampler='pt': the DeviceParallelTemperingSampler (fitter.sampler = its cold view)
        self.mcmc_flag = False
        self.sampler = None
        self.best_theta = None
        self.samples = None
        self.ndim = len(self.theta)
        self.nwalkers = no_of_Chain
        self._rng = np.random.default_rng(seed)
        self._seed = seed
        self.device_sampler = bool(device_sampler)   # sampling loop on the GPU (rbv_stretch_run / rbv_slice_run)

    # ------------------------------------------------------------------ validation (vfit_mcmc.py:199-229)
    def _validate_unified_instrument_data(self, instrument_data):
        if not isinstance(instrument_data, dict):
            raise TypeError("instrument_data must be a dictionary")
        if len(instrument_data) == 0:
            raise ValueError("instrument_data cannot be empty")
        required = {"model", "wave", "flux", "error"}
        for name, data in instrument_data.items():
            if not isinstance(data, dict):
                raise TypeError(f"instrument_data['{name}'] must be a dictionary")
            missing = required - set(data.keys())
            if missing:
                raise ValueError(f"instrument_data['{name}'] missing keys: {missing}")
            n = len(data["wave"])
            if len(data["flux"]) != n or len(data["error"]) != n:
                raise ValueError(f"instrument_data['{name}']: wave, flux, and error must have same length")

    def _validate_guesses(self, theta, lb, ub):
        theta, lb, ub = np.asarray(theta), np.asarray(lb), np.asarray(ub)
        if len(theta) != len(lb) or len(theta) != len(ub):
            raise ValueError("theta, lb, and ub must have the same length")
        if np.any(theta < lb) or np.any(theta > ub):
            raise ValueError("Initial guess theta must be within bounds lb and ub")

    def _extract_configs(self, instrument_data):
        configs = {}
        for name, data in instrument_data.items():
            model = data["model"]
            if hasattr(model, "config"):
                cfg = copy.deepcopy(model.config)
                if not hasattr(cfg, "instrumental_params"):
                    cfg.instrumental_params = {}
                if getattr(model, "FWHM", None) is not None:
                    cfg.instrumental_params["FWHM"] = model.FWHM
                for p in ("grating", "life_position", "cen_wave"):
                    if getattr(model, p, None) is not None:
                        cfg.instrumental_params[p] = getattr(model, p)
                configs[name] = cfg
        return configs

    # ------------------------------------------------------------------ likelihood (vfit_mcmc.py:291-353)
    def lnprior(self, theta):
        return self._like.lnprior(theta)

    def lnprob(self, theta):
        """(ndim,) -> float, (n, ndim) -> (n,): prior and likelihood are fused on the device."""
        return self._like.lnprob(theta)

    def lnlike(self, theta):
        """lnlike alone (vfit_mcmc.py:297-319): the reference's lnlike does not look at the bounds, so rows outside
        them are evaluated too (``rbv_lnlike_batch``: the lnprob launch without the prior, no shared state touched)."""
        return self._like.lnlike(theta)

    # ------------------------------------------------------------------ optimiser (vfit_mcmc.py:355-360)
    def optimize_guess(self, theta, gradient="fd"):
        """L-BFGS-B on -lnprob with scipy's 2-point finite differences (absolute step 1e-8, flipped at the
        upper bound), exactly what ``op.minimize(nll, theta, method='L-BFGS-B', bounds=bounds)`` does -- but
        f(x) and its ndim forward-difference probes are ONE device batch per iteration instead of ndim+1
        serial calls.  ``gradient="device"``: f and its exact gradient from one device row per call
        (``rbv_lnprob_grad_batch``)."""
        import scipy.optimize as op
        if gradient not in ("fd", "device"):
            raise ValueError("gradient must be 'fd' or 'device'")
        lb, ub = self.lb.astype(float), self.ub.astype(float)
        h = 1e-8

        if gradient == "device":
            def fun_and_grad(x):
                v, g = self._like.lnprob_and_grad(np.asarray(x, dtype=np.float64))
                return -v, -g

            result = op.minimize(fun_and_grad, np.asarray(theta, dtype=np.float64), jac=True, method="L-BFGS-B",
                                 bounds=list(zip(lb, ub)))
            return result.x

        def fun_and_grad(x):
            x = np.asarray(x, dtype=np.float64)
            steps = np.full(self.ndim, h)
            steps[x + h > ub] = -h                      # one-sided step stays inside the bounds
            batch = np.vstack([x, x[None, :] + np.diag(steps)])
            vals = -np.asarray(self.lnprob(batch))
            return vals[0], (vals[1:] - vals[0]) / steps

        result = op.minimize(fun_and_grad, np.asarray(theta, dtype=np.float64), jac=True, method="L-BFGS-B",
                             bounds=list(zip(lb, ub)))
        return result.x

    # ------------------------------------------------------------------ quick fit (vfit_mcmc.py:362-406)
    def _chi2_batch(self, thetas):
        """chi^2 summed over instruments for every row (quick_fit_interface.py:30-51), without the prior:
        chi^2 = -2 lnlike + sum_px log_inv_sigma2, the second term being constant.  One device batch."""
        thetas = np.atleast_2d(np.asarray(thetas, dtype=np.float64))
        const = sum(float(np.sum(np.asarray(d["log_inv_sigma2"], dtype=np.float64)))
                    for d in self.instrument_data.values())
        ll = np.atleast_1d(self.lnlike(thetas))
        chi2 = -2.0 * ll + const
        return np.where(np.isfinite(chi2), chi2, 1e10)            # the reference returns 1e10 when evaluation fails

    def fit_quick(self, verbose=True, gradient="fd", method="lbfgsb"):
        """Deterministic chi^2 fit (L-BFGS-B, maxfun 5000) with finite-difference 1-sigma errors -- same
        objective, optimiser, step rule and fallbacks as core/quick_fit_interface.py:10-128; the objective, its
        gradient probes and the 2 ndim + 1 curvature probes are device batches.  ``gradient="device"``: chi^2 and
        its exact gradient (-2 d lnlike) from one device row per call; the error bars keep the rule above.

        ``method="lm"``: bounded Levenberg-Marquardt (``rbvfit_b200.lm``) on the device's Gauss-Newton matrix, one
        ``lnlike_and_fisher`` row per point evaluated; the errors are sqrt(diag) of the full covariance
        (J^T W J)^-1 over the free parameters, also stored as ``theta_best_covariance`` (NaN for parameters pinned
        on a bound or not constrained by the data).  ``gradient`` applies to L-BFGS-B only."""
        import scipy.optimize as op
        if gradient not in ("fd", "device"):
            raise ValueError("gradient must be 'fd' or 'device'")
        if method not in ("lbfgsb", "lm"):
            raise ValueError("method must be 'lbfgsb' or 'lm'")
        if method == "lm":
            if gradient != "fd":
                raise ValueError("gradient applies to method='lbfgsb' only")
            return self._fit_quick_lm(verbose)
        self.mcmc_flag = False
        lb, ub = self.lb.astype(float), self.ub.astype(float)
        h = 1e-8
        theta0 = np.asarray(self.theta, dtype=np.float64)

        def fun_and_grad(x):
            x = np.asarray(x, dtype=np.float64)
            steps = np.full(self.ndim, h)
            steps[x + h > ub] = -h
            vals = self._chi2_batch(np.vstack([x, x[None, :] + np.diag(steps)]))
            return vals[0], (vals[1:] - vals[0]) / steps

        if gradient == "device":
            const = sum(float(np.sum(np.asarray(d["log_inv_sigma2"], dtype=np.float64)))
                        for d in self.instrument_data.values())

            def fun_and_grad(x):      # noqa: F811 -- the exact-gradient objective replaces the FD one
                ll, g = self._like.lnlike_and_grad(np.asarray(x, dtype=np.float64))
                chi2 = -2.0 * ll + const
                if not np.isfinite(chi2):
                    return 1e10, np.zeros_like(g)          # the reference returns 1e10 when evaluation fails
                return chi2, -2.0 * g

        try:
            result = op.minimize(fun_and_grad, theta0, jac=True, bounds=list(zip(lb, ub)), method="L-BFGS-B",
                                 options={"maxfun": 5000})
            best = result.x
            if not result.success:
                warnings.warn(f"Optimization may not have converged: {result.message}")
            # _estimate_parameter_errors (:93-128): central second difference, chi2 + 1 criterion
            delta = np.maximum(np.maximum(np.abs(best) * 0.01, np.abs(theta0) * 0.01), 1e-6)
            probes = np.vstack([best, best[None, :] + np.diag(delta), best[None, :] - np.diag(delta)])
            c = self._chi2_batch(probes)
            d2 = (c[1:self.ndim + 1] - 2.0 * c[0] + c[self.ndim + 1:]) / delta ** 2
            with np.errstate(divide="ignore", invalid="ignore"):
                err = np.where(d2 > 0, np.sqrt(1.0 / d2), np.abs(best - theta0))
        except Exception as e:   # pragma: no cover - mirrors the reference's fallback
            warnings.warn(f"Minimize fitting failed: {e}")
            best, err = theta0.copy(), np.zeros_like(theta0)
        if verbose:
            print("Quick fit completed")
            if np.any(np.isnan(err)):
                print("WARNING: Some uncertainties are NaN")
        self.theta_best, self.theta_best_error = best, err
        return best, err

    def _fit_quick_lm(self, verbose):
        from .lm import levenberg_marquardt
        self.mcmc_flag = False
        res = levenberg_marquardt(self._like.lnlike_and_fisher, np.asarray(self.theta, dtype=np.float64),
                                  self.lb.astype(float), self.ub.astype(float))
        if res.status <= 0:
            warnings.warn(f"Optimization may not have converged: {res.message}")
        err = np.sqrt(np.diag(res.cov))
        if verbose:
            print("Quick fit completed")
            if np.any(np.isnan(err)):
                print("WARNING: Some uncertainties are NaN")
        self.theta_best, self.theta_best_error, self.theta_best_covariance = res.x, err, res.cov
        return res.x, err

    def covariance(self, theta=None):
        """Inverse Gauss-Newton matrix (J^T W J)^-1 at ``theta`` (default ``theta_best``, else ``theta``) from one
        device row: the Delta chi^2 = 1 covariance over the free parameters, NaN rows / columns for parameters
        pinned on a bound (gradient pointing out of the box) or not constrained by the data."""
        from . import lm
        if theta is None:
            theta = getattr(self, "theta_best", None)
            if theta is None:
                theta = self.theta
        theta = np.asarray(theta, dtype=np.float64)
        _ll, g, F = self._like.lnlike_and_fisher(theta)
        return lm.covariance(F, lm.free_set(theta, g, F, self.lb.astype(float), self.ub.astype(float)))

    # ------------------------------------------------------------------ walkers (vfit_mcmc.py:442-466)
    def _initialize_walkers(self, popt):
        """Same distribution and bounds clipping as the reference; validity is checked for all walkers in one
        batch and only the invalid ones are redrawn."""
        guesses = np.empty((self.nwalkers, self.ndim))
        todo = np.arange(self.nwalkers)
        for _attempt in range(1000):
            g = popt + self.perturbation * self._rng.standard_normal((len(todo), self.ndim))
            g = np.clip(g, self.lb + 1e-10, self.ub - 1e-10)
            ok = np.isfinite(np.atleast_1d(self.lnprob(g)))
            guesses[todo[ok]] = g[ok]
            todo = todo[~ok]
            if len(todo) == 0:
                return guesses
        raise RuntimeError(f"Could not initialize walker {todo[0]} after 1000 attempts")

    # ------------------------------------------------------------------ MCMC (vfit_mcmc.py:492-561)
    def runmcmc(self, optimize=True, verbose=True, use_pool=True, progress=True):
        if optimize:
            if verbose:
                print("  Optimizing starting guess...")
            self.theta = self.optimize_guess(self.theta)
            if verbose:
                print("✓ Starting guess optimized")
        guesses = self._initialize_walkers(self.theta)
        if self.sampler_name == "pt":
            from .pt_sampler import DeviceParallelTemperingSampler
            sampler = DeviceParallelTemperingSampler(self.nwalkers, self.ndim, self._like, betas=self.betas,
                                                     seed=self._seed)
            guesses = np.stack([guesses] + [self._initialize_walkers(self.theta) for _ in range(sampler.ntemps - 1)])
        elif self.sampler_name == "zeus":
            from .slice_sampler import DeviceEnsembleSliceSampler, EnsembleSliceSampler
            if self.device_sampler:
                sampler = DeviceEnsembleSliceSampler(self.nwalkers, self.ndim, self._like, seed=self._seed)
            else:
                sampler = EnsembleSliceSampler(self.nwalkers, self.ndim, self.lnprob, seed=self._seed)
        elif self.device_sampler:
            sampler = DeviceEnsembleSampler(self.nwalkers, self.ndim, self._like, seed=self._seed)
        else:
            sampler = EnsembleSampler(self.nwalkers, self.ndim, self.lnprob, seed=self._seed)
        if verbose:
            print(f"  Starting {self.sampler_name} MCMC (device batches)...")
            print(f"   Walkers: {self.nwalkers}")
            print(f"   Steps: {self.no_of_steps}")
            print(f"   Instruments: {len(self.instrument_data)}")
        try:
            if self.sampler_name in ("emcee", "pt"):
                sampler.run_mcmc(guesses, self.no_of_steps, progress=progress,
                                 skip_initial_state_check=self.skip_initial_state_check)
            else:
                sampler.run_mcmc(guesses, self.no_of_steps, progress=progress)
        except Exception as e:
            raise RuntimeError(f"MCMC sampling failed: {e}")
        if self.sampler_name == "pt":
            self.pt_sampler, sampler = sampler, sampler.cold()
        self.sampler = sampler
        self.mcmc_flag = True
        self.samples = None
        self.compute_best_theta()
        if verbose:
            print("  MCMC completed")
            self._print_diagnostics()

    def compute_best_theta(self, burntime=100):
        if self.samples is None:
            self.samples = self._extract_samples(self.sampler, burntime)
        self.best_theta = np.percentile(self.samples, 50, axis=0)
        self.low_theta = np.percentile(self.samples, 16, axis=0)
        self.high_theta = np.percentile(self.samples, 84, axis=0)

    def _extract_samples(self, sampler, burntime):
        try:
            return sampler.get_chain(discard=burntime, flat=True)
        except Exception as e:   # pragma: no cover
            warnings.warn(f"Could not extract samples: {e}")
            return np.array([])

    def _get_acceptance_fraction(self, sampler):
        return sampler.acceptance_fraction

    def _print_diagnostics(self):
        """vfit_mcmc.py:589-655: acceptance fraction, emcee's integrated auto-correlation time, zeus's Gelman-Rubin
        statistic (zeus.diagnostics.gelman_rubin is not vendored in the reference; `gelman_rubin` below restates the
        standard estimator on the walkers as chains)."""
        print("\n" + "=" * 60 + "\nMCMC DIAGNOSTICS\n" + "=" * 60)
        try:
            af = np.mean(self._get_acceptance_fraction(self.sampler))
            print(f"Mean acceptance fraction: {af:.3f}")
            if af < 0.2:
                print("⚠️  Low acceptance fraction (<0.2). Consider reducing step size.")
            elif af > 0.7:
                print("⚠️  High acceptance fraction (>0.7). Consider increasing step size.")
            else:
                print("✅ Good acceptance fraction (0.2-0.7)")
        except Exception:
            print("Acceptance fraction not available")
        if self.sampler_name == "pt":
            try:
                print("Swap acceptance (coldest pair first): "
                      + " ".join(f"{x:.2f}" for x in self.pt_sampler.tswap_acceptance_fraction))
                lnz, dlnz = self.log_evidence()
                print(f"ln Z (thermodynamic integration, second half of the chain): {lnz:.3f} +- {dlnz:.3f}")
            except Exception:
                print("Evidence not available")
        if self.sampler_name in ("emcee", "pt"):
            try:
                tau = np.nanmean(self.sampler.get_autocorr_time())
                print(f"Mean auto-correlation time: {tau:.3f} steps")
                if self.no_of_steps < 50 * tau:
                    print("⚠️  Warning: Chain may be too short for reliable results")
                    print(f"   Recommended: >{50 * tau:.0f} steps")
                else:
                    print("✅ Chain length adequate")
            except Exception:
                print("⚠️  Warning: Could not calculate auto-correlation time")
        if self.sampler_name == "zeus":
            try:
                max_rhat = float(np.max(gelman_rubin(self.sampler.get_chain().transpose(1, 0, 2))))
                print(f"Gelman-Rubin R-hat: {max_rhat:.3f}")
                if max_rhat > 1.1:
                    print("⚠️  Warning: R-hat > 1.1, chains may not have converged")
                else:
                    print("✅ Good convergence (R-hat < 1.1)")
            except Exception:
                print("Could not calculate Gelman-Rubin diagnostic")
        if self.best_theta is not None:
            print("\nParameter Summary:")
            print(f"Best-fit parameters: {len(self.best_theta)} values")
            if self.samples is not None:
                print(f"Effective samples: {len(self.samples)}")
        print("=" * 60)

    def chi_squared(self, theta=None, instrument_name=None):
        """Reduced chi-squared per instrument (and 'combined' for several) at ``theta`` (default: best_theta, else
        the current guess) -- the computation of UnifiedResults.chi_squared (core/unified_results.py:305-369):
        chi2 = sum(((flux - model) / error)**2), dof = max(n_data - n_params, 1); the model comes from the GPU."""
        if theta is None:
            theta = self.best_theta if self.best_theta is not None else self.theta
        theta = np.asarray(theta, dtype=np.float64)
        if instrument_name is not None and instrument_name not in self.instrument_data:
            raise ValueError(f"Instrument '{instrument_name}' not found. Available: {list(self.instrument_data)}")
        names = [instrument_name] if instrument_name is not None else list(self.instrument_data)
        results, total_chi2, total_n = {}, 0.0, 0
        for name in names:
            d = self.instrument_data[name]
            model = d["model"](theta, d["wave"])
            keep = d.get("weight_mask")             # extension: masked pixels (piecewise-LSF halos) do not count
            keep = np.ones(len(d["wave"]), dtype=bool) if keep is None else np.asarray(keep, dtype=bool)
            chi2 = float(np.sum((((d["flux"] - model) / d["error"]) ** 2)[keep]))
            results[name] = chi2 / max(int(keep.sum()) - len(theta), 1)
            total_chi2 += chi2
            total_n += int(keep.sum())
        if instrument_name is None and len(names) > 1:
            results["combined"] = total_chi2 / max(total_n - len(theta), 1)
        return results

    def log_evidence(self, burn_in=0.5):
        """sampler='pt': (ln Z, d ln Z) by thermodynamic integration over the steps after the first ``burn_in``
        fraction (``DeviceParallelTemperingSampler.log_evidence_estimate``); Z is normalised to the box prior of the
        bounds, so two line sets fitted to the same data compare by ln Z."""
        if not self.mcmc_flag:
            raise RuntimeError("MCMC has not been run")
        if self.pt_sampler is None:
            raise RuntimeError("the evidence needs sampler='pt' (parallel tempering)")
        return self.pt_sampler.log_evidence_estimate(discard=int(burn_in * self.no_of_steps))

    def get_samples(self, flat=True, burn_in=0.5):
        if not self.mcmc_flag:
            raise RuntimeError("MCMC has not been run")
        return self.sampler.get_chain(discard=int(burn_in * self.no_of_steps), flat=flat)


def set_bounds(nguess, bguess, vguess, **kwargs):
    """Traditional branch of the reference's ``set_bounds`` (vfit_mcmc.py:760-787): N +- 2 dex,
    b in [max(2, b-40), min(150, b+40)], v +- 50 km/s, with the same keyword overrides.
    (The reference's ``ions=`` branch is mis-indented and leaves most bounds at zero -- SURVEY.md appendix B;
    it is not replicated.)"""
    if kwargs.get("ions") is not None:
        raise NotImplementedError("ion-aware bounds are outside the hot path (and broken in the reference)")
    nguess, bguess, vguess = np.asarray(nguess), np.asarray(bguess), np.asarray(vguess)
    Nlow, NHI = nguess - 2.0, nguess + 2.0
    blow, bHI = np.clip(bguess - 40.0, 2.0, None), np.clip(bguess + 40.0, None, 150.0)
    vlow, vHI = vguess - 50.0, vguess + 50.0
    Nlow = np.asarray(kwargs.get("Nlow", Nlow))
    blow = np.asarray(kwargs.get("blow", blow))
    vlow = np.asarray(kwargs.get("vlow", vlow))
    NHI = np.asarray(kwargs.get("Nhi", NHI))
    bHI = np.asarray(kwargs.get("bhi", bHI))
    vHI = np.asarray(kwargs.get("vhi", vHI))
    lb = np.concatenate([Nlow, blow, vlow])
    ub = np.concatenate([NHI, bHI, vHI])
    return [lb, ub], lb, ub
