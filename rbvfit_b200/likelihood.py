"""Batched GPU likelihood: the B200 replacement of ``vfit._compile_models`` + ``lnprior/lnlike/lnprob``
(reference: src/rbvfit/vfit_mcmc.py:234-259, 291-353).

``GpuLikelihood.lnprob`` honours emcee's / zeus's ``vectorize=True`` contract -- ``(n, ndim) -> (n,)`` --
and still returns a plain float for a single ``(ndim,)`` row, so it can be handed to either sampler or
called by an optimiser exactly like the reference's bound method.
"""
from __future__ import annotations

import warnings
from typing import Dict, NamedTuple, Optional

import numpy as np

from ._lib import RbvError
from .engine import Engine
from .model import GpuCompiledVoigtModel, GpuVoigtModel


def _weights(error):
    """inv_sigma2 / log_inv_sigma2 with the reference's expressions AND dtype (vfit_mcmc.py:255-256):
    a float32 error array gives float32-rounded weights, which are then promoted to float64."""
    err = np.asarray(error)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv_sigma2 = 1.0 / (err ** 2)
        log_inv_sigma2 = np.log(1.0 / (err ** 2))
    return inv_sigma2, log_inv_sigma2


class _LnprobFunction:
    """``torch.autograd.Function`` for ``GpuLikelihood.lnprob_torch``, built on first use (torch is imported lazily
    throughout the package)."""
    _cls = None

    @classmethod
    def apply(cls, theta_t, engine):
        if cls._cls is None:
            import torch

            class LnprobFunction(torch.autograd.Function):
                @staticmethod
                def forward(ctx, theta, eng):
                    rows = theta.detach()
                    rows = (rows[None, :] if rows.dim() == 1 else rows).contiguous()
                    value, grad = eng.lnprob_grad_device(rows, True)
                    ctx.save_for_backward(grad)
                    ctx.squeeze = theta.dim() == 1
                    return value[0] if ctx.squeeze else value

                @staticmethod
                def backward(ctx, grad_output):
                    (grad,) = ctx.saved_tensors
                    if ctx.squeeze:
                        return grad_output * grad[0], None
                    return grad_output[:, None] * grad, None

            cls._cls = LnprobFunction
        return cls._cls.apply(theta_t, engine)


class GpuLikelihood:
    """All instruments of one fit on one GPU."""

    def __init__(self, instrument_data: Dict[str, dict], lb, ub, device: Optional[int] = None):
        if not isinstance(instrument_data, dict):
            raise TypeError("instrument_data must be a dictionary")
        if len(instrument_data) == 0:
            raise ValueError("instrument_data cannot be empty")
        self.engine = Engine(device)
        self.names = []
        self.pixels = []
        self.instrument_data = {}
        for name, d in instrument_data.items():
            model = d["model"]
            if isinstance(model, GpuVoigtModel):                 # vfit_mcmc.py:241-245
                compiled = model.compile(verbose=False)
            elif isinstance(model, GpuCompiledVoigtModel):
                compiled = model
            else:
                raise TypeError(
                    f"instrument_data['{name}']['model'] must be a GpuVoigtModel / GpuCompiledVoigtModel: "
                    "arbitrary Python callables cannot run on the device and rbvfit_b200 has no CPU fallback")
            wave, flux, error = (np.asarray(d[k]) for k in ("wave", "flux", "error"))
            if len(flux) != len(wave) or len(error) != len(wave):
                raise ValueError(f"instrument_data['{name}']: wave, flux, and error must have same length")
            inv_sigma2, log_inv_sigma2 = _weights(error)
            mask = d.get("weight_mask")
            if mask is not None:     # extension: pixels with False do not enter the likelihood (both terms exactly 0)
                mask = np.asarray(mask, dtype=bool)
                if mask.shape != wave.shape:
                    raise ValueError(f"instrument_data['{name}']: weight_mask must have the shape of wave")
                inv_sigma2 = np.where(mask, inv_sigma2, inv_sigma2.dtype.type(0))
                log_inv_sigma2 = np.where(mask, log_inv_sigma2, log_inv_sigma2.dtype.type(0))
            data = compiled.data
            self.engine.add_instrument(data, wave, flux=flux, inv_sigma2=inv_sigma2,
                                       log_inv_sigma2=log_inv_sigma2, taps=data.kernel,
                                       normalize_taps=data.kernel_normalize)
            self.names.append(name)
            self.pixels.append(len(wave))
            self.instrument_data[name] = {"model": compiled.model_flux, "wave": wave, "flux": flux,
                                          "error": error, "inv_sigma2": inv_sigma2,
                                          "log_inv_sigma2": log_inv_sigma2, "weight_mask": mask}
        self.lb = np.asarray(lb, dtype=np.float64)
        self.ub = np.asarray(ub, dtype=np.float64)
        self.engine.set_bounds(self.lb, self.ub)
        self.ndim = self.lb.size
        self.total_pixels = int(sum(self.pixels))
        self.precision = "fp64"
        self.far_field = "chebyshev"
        self.last_precision_check = None

    # ------------------------------------------------------------------ reference-shaped API
    def lnprob(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim == 1:
            return float(self.engine.lnprob_host(theta[None, :])[0])
        if theta.ndim != 2:
            raise ValueError("theta must be (ndim,) or (n, ndim)")
        if theta.shape[0] == 0:
            return np.zeros(0)
        return self.engine.lnprob_host(np.ascontiguousarray(theta))

    __call__ = lnprob

    def pinned_theta(self, n: int) -> np.ndarray:
        """Page-locked [n, ndim] array for ensembles that are evaluated repeatedly: ``lnprob`` reads a page-locked
        theta in place (no staging copy on the host)."""
        return self.engine.pinned_theta(n)

    def lnlike(self, theta):
        """The likelihood without the prior (``vfit.lnlike``, vfit_mcmc.py:297-319): rows outside the bounds are
        evaluated like any other.  One launch, no shared state touched."""
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim == 1:
            return float(self.engine.lnlike_host(theta[None, :])[0])
        if theta.shape[0] == 0:
            return np.zeros(0)
        return self.engine.lnlike_host(theta)

    def lnprior(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        bad = np.any(theta < self.lb, axis=-1) | np.any(theta > self.ub, axis=-1)
        out = np.where(bad, -np.inf, 0.0)
        return float(out) if out.ndim == 0 else out

    def lnprob_device(self, theta_t, out_t=None):
        """Device-resident variant (torch tensors in / out, asynchronous)."""
        return self.engine.lnprob_device(theta_t, out_t)

    # ------------------------------------------------------------------ analytic gradient (DESIGN.md section 14)
    def _value_and_grad(self, theta, apply_prior: bool):
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim not in (1, 2) or theta.shape[-1] != self.ndim:
            raise ValueError(f"theta must be ({self.ndim},) or (n, {self.ndim})")
        if theta.ndim == 2 and theta.shape[0] == 0:
            return np.zeros(0), np.zeros((0, self.ndim))
        v, g = self.engine.lnprob_grad_host(np.atleast_2d(theta), apply_prior)
        if theta.ndim == 1:
            return float(v[0]), g[0]
        return v, g

    def lnprob_and_grad(self, theta):
        """lnprob and its exact gradient from one device row per theta row: ``(ndim,) -> (float, (ndim,))``,
        ``(n, ndim) -> ((n,), (n, ndim))``.  Rows outside the bounds give -inf and a zero gradient."""
        return self._value_and_grad(theta, True)

    def lnlike_and_grad(self, theta):
        """lnlike (no prior: every row evaluated) and its exact gradient; shapes as ``lnprob_and_grad``."""
        return self._value_and_grad(theta, False)

    def lnprob_torch(self, theta_t):
        """lnprob as a differentiable torch function of a DEVICE float64 tensor (``(n, ndim) -> (n,)``,
        ``(ndim,) -> 0-d``): the forward pass is one ``rbv_lnprob_grad_batch`` launch, the backward pass scales the
        saved gradient by ``grad_output``."""
        return _LnprobFunction.apply(theta_t, self.engine)

    # ------------------------------------------------------------------ Jacobian / Fisher (DESIGN.md section 15)
    def _rows(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim not in (1, 2) or theta.shape[-1] != self.ndim:
            raise ValueError(f"theta must be ({self.ndim},) or (n, {self.ndim})")
        return theta

    def lnlike_and_fisher(self, theta):
        """lnlike (no prior), its gradient and its Gauss-Newton matrix sum_p w_p dM_p/dtheta_i dM_p/dtheta_j from one
        device row per theta row: ``(ndim,) -> (float, (ndim,), (ndim, ndim))``,
        ``(n, ndim) -> ((n,), (n, ndim), (n, ndim, ndim))``.  -2 lnlike is chi^2 up to a constant, so the inverse
        of the matrix is the Delta chi^2 = 1 covariance of the parameters."""
        theta = self._rows(theta)
        if theta.ndim == 2 and theta.shape[0] == 0:
            return np.zeros(0), np.zeros((0, self.ndim)), np.zeros((0, self.ndim, self.ndim))
        v, g, f = self.engine.lnlike_fisher_host(np.atleast_2d(theta))
        if theta.ndim == 1:
            return float(v[0]), g[0], f[0]
        return v, g, f

    def model_jacobian(self, theta, instrument):
        """d(model flux)/dtheta of one instrument (name or index), LSF applied: ``(ndim,) -> [P, ndim]``,
        ``(n, ndim) -> [n, P, ndim]`` (the layout of scipy's ``least_squares``)."""
        theta = self._rows(theta)
        inst = self.names.index(instrument) if isinstance(instrument, str) else int(instrument)
        if theta.ndim == 2 and theta.shape[0] == 0:
            return np.zeros((0, self.pixels[inst], self.ndim))
        jac = np.swapaxes(self.engine.model_jacobian(inst, np.atleast_2d(theta)), 1, 2)
        return jac[0] if theta.ndim == 1 else jac

    def set_far_field(self, mode: str = "chebyshev"):
        """``"chebyshev"`` (default): the summed far wings (lines >= 24 Doppler widths away) of each 1024-pixel
        super-chunk are evaluated at 8 Chebyshev nodes and interpolated; a line takes part only where an
        a-priori bound keeps its interpolation error <= 1e-12 / L in optical depth (DESIGN.md section 4c).
        ``"direct"``: every (line, pixel) pair is evaluated on its own."""
        if mode not in ("chebyshev", "direct"):
            raise ValueError("far field mode must be 'chebyshev' or 'direct'")
        self.engine.set_farfield(mode)
        self.far_field = mode

    def set_precision(self, precision: str = "fp64", check_thetas=None, rtol: float = 1e-9) -> bool:
        """Select the far-wing arithmetic.  ``"fp32-gated"`` moves far-wing lines whose contribution is provably
        tiny (a-priori bound: their sum stays <= 4e-6 per pixel, i.e. |dtau| <= 1e-11) to the FP32 pipe.
        With ``check_thetas`` the gate is also verified a posteriori: the batch is evaluated in both modes and
        the FP32 variant is kept only if every finite lnprob agrees to ``rtol``; otherwise the likelihood
        falls back to FP64 (never to the CPU).  Returns True when the requested precision is active."""
        if precision not in ("fp64", "fp32-gated"):
            raise ValueError("precision must be 'fp64' or 'fp32-gated'")
        self.engine.set_precision("fp64")
        self.precision = "fp64"
        if precision == "fp64":
            return True
        ref = None if check_thetas is None else self.lnprob(np.atleast_2d(check_thetas))
        self.engine.set_precision("fp32-gated")
        self.precision = "fp32-gated"
        if ref is not None:
            got = self.lnprob(np.atleast_2d(check_thetas))
            fin = np.isfinite(ref)
            same_pattern = np.array_equal(np.isfinite(got), fin)
            err = np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin])) if fin.any() else 0.0
            self.last_precision_check = float(err)
            if not same_pattern or not (err <= rtol):
                self.engine.set_precision("fp64")
                self.precision = "fp64"
                return False
        return True

    def close(self):
        self.engine.close()


class SightlineFit(NamedTuple):
    """Per-sightline results of ``SightlineBatch.fit_quick``, each field with the meaning of ``lm.LMResult``."""
    x: np.ndarray          # [S, ndim] best points
    chi2: np.ndarray       # [S] -2 lnlike at x
    cov: np.ndarray        # [S, ndim, ndim] inv(F_ff) over the free set; NaN rows / columns elsewhere
    n_evals: np.ndarray    # [S] Fisher evaluations
    status: np.ndarray     # [S] lm.STATUS_*: > 0 converged
    errors: np.ndarray     # [S, ndim] sqrt(diag(cov))


class SightlineBatch:
    """Survey mode (BASELINE.json config 5, "1024 independent sightlines batched"): S independent fits that share
    the model *structure* (same number of lines / components / pixels / LSF taps) but have their own redshift,
    spectrum and walker ensemble.  One launch evaluates every walker of every sightline; walker row
    ``s * walkers_per_sightline + k`` belongs to sightline ``s``.  Sightlines shard across GPUs with no
    collective (each rank builds a SightlineBatch over its own subset)."""

    def __init__(self, sightlines, lb, ub, device: Optional[int] = None):
        """``sightlines``: list of dicts {'model', 'wave', 'flux', 'error'} (one instrument each)."""
        if len(sightlines) == 0:
            raise ValueError("sightlines cannot be empty")
        self.engine = Engine(device)
        self.n_sightlines = len(sightlines)
        for i, d in enumerate(sightlines):
            model = d["model"]
            compiled = model.compile(verbose=False) if isinstance(model, GpuVoigtModel) else model
            if not isinstance(compiled, GpuCompiledVoigtModel):
                raise TypeError(f"sightline {i}: 'model' must be a GpuVoigtModel / GpuCompiledVoigtModel")
            wave, flux, error = (np.asarray(d[k]) for k in ("wave", "flux", "error"))
            if len(flux) != len(wave) or len(error) != len(wave):
                raise ValueError(f"sightline {i}: wave, flux, and error must have same length")
            inv_sigma2, log_inv_sigma2 = _weights(error)
            mask = d.get("weight_mask")
            if mask is not None:     # extension: pixels with False do not enter the likelihood (both terms exactly 0)
                mask = np.asarray(mask, dtype=bool)
                if mask.shape != wave.shape:
                    raise ValueError(f"sightline {i}: weight_mask must have the shape of wave")
                inv_sigma2 = np.where(mask, inv_sigma2, inv_sigma2.dtype.type(0))
                log_inv_sigma2 = np.where(mask, log_inv_sigma2, log_inv_sigma2.dtype.type(0))
            data = compiled.data
            self.engine.add_instrument(data, wave, flux=flux, inv_sigma2=inv_sigma2, log_inv_sigma2=log_inv_sigma2,
                                       taps=data.kernel, normalize_taps=data.kernel_normalize)
        self.pixels = self.engine.pixels[0]
        self.lb = np.asarray(lb, dtype=np.float64)
        self.ub = np.asarray(ub, dtype=np.float64)
        self.engine.set_bounds(self.lb, self.ub)
        self.ndim = self.lb.size

    def lnprob(self, theta):
        """theta [S, Ws, ndim] -> lnprob [S, Ws]."""
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim != 3 or theta.shape[0] != self.n_sightlines or theta.shape[2] != self.ndim:
            raise ValueError(f"theta must be [{self.n_sightlines}, walkers_per_sightline, {self.ndim}]")
        S, Ws, nd = theta.shape
        return self.engine.lnprob_sightlines_host(theta.reshape(S * Ws, nd), Ws).reshape(S, Ws)

    def pinned_theta(self, walkers_per_sightline: int) -> np.ndarray:
        """Page-locked [S, walkers_per_sightline, ndim] array: ``lnprob`` copies it to the device in place."""
        a = self.engine.pinned_theta(self.n_sightlines * int(walkers_per_sightline))
        return a.reshape(self.n_sightlines, int(walkers_per_sightline), self.ndim)

    def lnprob_device(self, theta_t, wps: int, out_t=None):
        return self.engine.lnprob_sightlines_device(theta_t, wps, out_t)

    def lnlike_and_fisher(self, theta):
        """theta [S, Ws, ndim] -> (lnlike [S, Ws], gradient [S, Ws, ndim], Gauss-Newton matrix [S, Ws, ndim, ndim]),
        every row against its own sightline (``GpuLikelihood.lnlike_and_fisher`` of that sightline, bit for bit)."""
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim != 3 or theta.shape[0] != self.n_sightlines or theta.shape[2] != self.ndim:
            raise ValueError(f"theta must be [{self.n_sightlines}, walkers_per_sightline, {self.ndim}]")
        S, Ws, nd = theta.shape
        v, g, f = self.engine.lnlike_fisher_sightlines_host(theta.reshape(S * Ws, nd), Ws)
        return v.reshape(S, Ws), g.reshape(S, Ws, nd), f.reshape(S, Ws, nd, nd)

    def fit_quick(self, theta0, max_evals: int = 200, ftol: float = 1e-10, xtol: float = 1e-10) -> SightlineFit:
        """Bounded Levenberg-Marquardt fit of every sightline (the rules of ``lm.levenberg_marquardt``) in one device
        loop: each iteration is one Fisher evaluation of the sightlines still iterating and one update kernel
        (DESIGN.md section 16).  ``theta0``: [S, ndim] starts, or one [ndim] start for every sightline.  Sightlines
        whose F_ff is not positive definite at the end get ``lm.covariance``'s pinv (with its warning)."""
        from . import lm
        S, nd = self.n_sightlines, self.ndim
        theta0 = np.asarray(theta0, dtype=np.float64)
        if theta0.shape == (nd,):
            theta0 = np.broadcast_to(theta0, (S, nd))
        if theta0.shape != (S, nd):
            raise ValueError(f"theta0 must be [{S}, {nd}] or [{nd}]")
        x, chi2, cov, n_evals, status, flags = self.engine.lm_sightlines(theta0, 0, S, max_evals, ftol, xtol)
        bad = np.flatnonzero(flags & 1)
        if bad.size:
            _v, g, F = self.engine.lnlike_fisher_sightlines_host(x, 1)
            for s in bad:
                cov[s] = lm.covariance(F[s], lm.free_set(x[s], g[s], F[s], self.lb, self.ub))
        n_bad = int(np.count_nonzero(status <= 0))
        if n_bad:
            warnings.warn(f"Optimization may not have converged on {n_bad} of {S} sightlines (status <= 0)")
        with np.errstate(invalid="ignore"):
            errors = np.sqrt(np.diagonal(cov, axis1=1, axis2=2))
        return SightlineFit(x, chi2, cov, n_evals, status, errors)

    def close(self):
        self.engine.close()
