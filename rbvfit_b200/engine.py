"""Thin owner of one ``RbvContext`` (C ABI) and of the PyTorch tensors it points at.

PyTorch is used for exactly three things here: device / pinned-host buffer ownership, the CUDA stream
handle, and (in ``rbvfit_b200.dist``) torch.distributed.  All arithmetic happens in the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional

import numpy as np

from . import _lib
from ._lib import RbvChainSink, RbvError, RbvLineTable, RbvPtControl, RbvSpectrum, check

VOIGT_METHODS = {"wofz": 0, "fast": 1}


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RbvError("rbvfit_b200 needs a CUDA device: torch.cuda.is_available() is False and there is "
                       "no CPU fallback")
    return torch


def _dptr(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Engine:
    """One likelihood context on one device."""

    def _dev_tensor(self, t, dtype, what: str, shape=None):
        """Every tensor whose ``data_ptr()`` crosses the C ABI: right dtype, contiguous, on this engine's device
        (anything else would be read as raw doubles / ints by the library)."""
        if t is None:
            return None
        if t.dtype != dtype or not t.is_contiguous() or t.device != self.tdev:
            raise ValueError(f"{what} must be a contiguous {dtype} tensor on {self.tdev}")
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise ValueError(f"{what} must have shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    def __init__(self, device: Optional[int] = None):
        torch = _torch()
        self.lib = _lib.load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.tdev = torch.device("cuda", self.device)
        self._h = C.c_void_p()
        check(self.lib.rbv_create(self.device, C.byref(self._h)), "rbv_create")
        self._keep: List[object] = []        # device tensors the context points at
        self.pixels: List[int] = []
        self.components: List[int] = []
        self.ndim = 0
        self._cap = 0                         # walker capacity of the staging buffers
        self._theta_dev = self._lnp_dev = self._ws = None
        self._theta_pin = self._lnp_pin = None
        self._ws_bytes = 0
        self._ws_sightlines = False
        self._stretch_ws = None               # workspace of the device-resident sampler
        self._slice_ws = None                 # workspace of the device-resident slice sampler
        self.comm_rank, self.comm_world = 0, 1   # rbv_comm_init (multi-GPU: the library issues the all-gather)
        self.peer_attached = False               # rbv_peer_attach: the all-gather over NVLink peer memory
        self._sink_ring = None                # (block_steps, device ring, pinned ring) of rbv_stretch_run_sink

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.rbv_destroy(self._h)
            self._h = C.c_void_p()
        self._keep = []

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ set-up
    def add_instrument(self, lowered, wave, flux=None, inv_sigma2=None, log_inv_sigma2=None,
                       taps=None, normalize_taps=False) -> int:
        """``lowered``: object with atomic_lambda0/atomic_gamma/atomic_f/z_factors/N_indices/
        total_components/voigt_method (CompiledModelData layout, voigt_model.py:265-280)."""
        torch = _torch()
        lam = np.ascontiguousarray(lowered.atomic_lambda0, dtype=np.float64)
        gam = np.ascontiguousarray(np.asarray(lowered.atomic_gamma), dtype=np.float64)   # f32 -> f64 promotion
        fos = np.ascontiguousarray(np.asarray(lowered.atomic_f), dtype=np.float64)
        zf = np.ascontiguousarray(lowered.z_factors, dtype=np.float64)
        comp = np.ascontiguousarray(lowered.N_indices, dtype=np.int32)
        lt = RbvLineTable(len(lam), int(lowered.total_components), _dptr(lam), _dptr(gam), _dptr(fos), _dptr(zf),
                          comp.ctypes.data_as(C.POINTER(C.c_int)), VOIGT_METHODS[lowered.voigt_method])

        def dev(a):
            if a is None:
                return None
            t = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.tdev)
            self._keep.append(t)
            return t

        wave_t = dev(wave)
        P = int(wave_t.numel())
        inv_wave_t = torch.empty(P, dtype=torch.float64, device=self.tdev)
        self._keep.append(inv_wave_t)
        flux_t, w_t, l_t = dev(flux), dev(inv_sigma2), dev(log_inv_sigma2)
        if taps is not None:
            taps = np.ascontiguousarray(taps, dtype=np.float64)
            taps_p, n_taps = _dptr(taps), int(taps.size)
        else:
            taps_p, n_taps = None, 0
        sp = RbvSpectrum(P, wave_t.data_ptr(),
                         flux_t.data_ptr() if flux_t is not None else None,
                         w_t.data_ptr() if w_t is not None else None,
                         l_t.data_ptr() if l_t is not None else None,
                         inv_wave_t.data_ptr(), taps_p, n_taps, int(bool(normalize_taps)))
        idx = C.c_int(-1)
        check(self.lib.rbv_add_instrument(self._h, C.byref(lt), C.byref(sp), C.byref(idx)), "rbv_add_instrument")
        self.pixels.append(P)
        self.components.append(int(lowered.total_components))
        self._cap = 0   # tile count changed -> workspace must be re-sized
        return idx.value

    def set_bounds(self, lb, ub):
        lb = np.ascontiguousarray(lb, dtype=np.float64)
        ub = np.ascontiguousarray(ub, dtype=np.float64)
        if lb.shape != ub.shape or lb.ndim != 1:
            raise ValueError("lb and ub must be 1-D arrays of equal length")
        check(self.lib.rbv_set_bounds(self._h, _dptr(lb), _dptr(ub), lb.size), "rbv_set_bounds")
        self.ndim = int(lb.size)
        self._cap = 0

    def set_precision(self, precision: str):
        check(self.lib.rbv_set_precision(self._h, {"fp64": 0, "fp32-gated": 1}[precision]), "rbv_set_precision")

    def set_farfield(self, mode: str):
        """'chebyshev' (default) or 'direct' -- how far line wings are accumulated (DESIGN.md section 4c)."""
        check(self.lib.rbv_set_farfield(self._h, {"direct": 0, "chebyshev": 1}[mode]), "rbv_set_farfield")

    # ------------------------------------------------------------------ buffers
    def _reserve(self, W: int, ndim: int, sightlines: bool = False):
        torch = _torch()
        if (W <= self._cap and self._theta_dev is not None and self._theta_dev.shape[1] == ndim
                and self._ws_sightlines == sightlines):
            return
        cap = max(W, 64, int(self._cap * 1.5))
        nbytes = C.c_size_t(0)
        fn = self.lib.rbv_workspace_bytes_sightlines if sightlines else self.lib.rbv_workspace_bytes
        check(fn(self._h, cap, C.byref(nbytes)), "rbv_workspace_bytes")
        self._ws_sightlines = sightlines
        self._ws_bytes = int(nbytes.value)
        self._ws = torch.empty(max(self._ws_bytes, 8), dtype=torch.uint8, device=self.tdev)
        self._theta_dev = torch.empty((cap, ndim), dtype=torch.float64, device=self.tdev)
        self._lnp_dev = torch.empty(cap, dtype=torch.float64, device=self.tdev)
        self._theta_pin = torch.empty((cap, ndim), dtype=torch.float64, pin_memory=True)
        self._lnp_pin = torch.empty(cap, dtype=torch.float64, pin_memory=True)
        self._theta_pin_np = self._theta_pin.numpy()
        self._lnp_pin_np = self._lnp_pin.numpy()
        self._cap = cap

    def _stream(self):
        return _torch().cuda.current_stream(self.tdev).cuda_stream

    # ------------------------------------------------------------------ hot path
    def lnprob_host(self, theta: np.ndarray) -> np.ndarray:
        """HOST theta [W, ndim] -> HOST lnprob [W]; H2D, kernel, D2H and the sync happen inside the C call."""
        W, ndim = theta.shape
        if ndim != self.ndim:
            raise ValueError(f"theta has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._reserve(W, ndim, sightlines=False)
        src = self._theta_pin.data_ptr()
        if (theta.dtype == np.float64 and theta.flags.c_contiguous
                and self.lib.rbv_host_pinned(theta.ctypes.data)):
            src = theta.ctypes.data            # page-locked already (pinned_theta, a pinned torch tensor): DMA in place
        else:
            self._theta_pin_np[:W] = theta     # staging copy of a pageable array
        check(self.lib.rbv_lnprob_batch_host(self._h, src, W, self._lnp_pin.data_ptr(),
                                             self._theta_dev.data_ptr(), self._lnp_dev.data_ptr(),
                                             self._ws.data_ptr(), self._ws_bytes, self._stream()),
              "rbv_lnprob_batch_host")
        return self._lnp_pin_np[:W].copy()

    def pinned_theta(self, W: int) -> np.ndarray:
        """A page-locked float64 array [W, ndim] the caller can fill in place: ``lnprob_host`` on it (or on any other
        page-locked array) skips the staging copy.  The array owns its memory (a pinned torch tensor behind it, freed
        with the array)."""
        torch = _torch()
        return torch.empty((int(W), self.ndim), dtype=torch.float64, pin_memory=True).numpy()   # the array keeps it alive

    def lnprob_device(self, theta_t, out_t=None):
        """DEVICE theta tensor [W, ndim] (float64, contiguous) -> DEVICE lnprob tensor [W]; asynchronous."""
        torch = _torch()
        self._dev_tensor(theta_t, torch.float64, "theta")
        W, ndim = theta_t.shape
        if ndim != self.ndim:
            raise ValueError(f"theta has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._reserve(W, ndim, sightlines=False)
        if out_t is None:
            out_t = torch.empty(W, dtype=torch.float64, device=self.tdev)
        self._dev_tensor(out_t, torch.float64, "out", (W,))
        check(self.lib.rbv_lnprob_batch(self._h, theta_t.data_ptr(), W, out_t.data_ptr(), self._ws.data_ptr(),
                                        self._ws_bytes, self._stream()), "rbv_lnprob_batch")
        return out_t

    def lnprob_grad_device(self, theta_t, apply_prior: bool, value_t=None, grad_t=None):
        """DEVICE theta [W, ndim] -> (value [W], gradient [W, ndim]) DEVICE tensors (``rbv_lnprob_grad_batch``):
        lnprob and its gradient with ``apply_prior``, lnlike and its gradient without; asynchronous."""
        torch = _torch()
        self._dev_tensor(theta_t, torch.float64, "theta")
        if theta_t.dim() != 2 or theta_t.shape[1] != self.ndim:
            raise ValueError(f"theta must be [W, {self.ndim}]")
        W = int(theta_t.shape[0])
        if value_t is None:
            value_t = torch.empty(W, dtype=torch.float64, device=self.tdev)
        if grad_t is None:
            grad_t = torch.empty((W, self.ndim), dtype=torch.float64, device=self.tdev)
        self._dev_tensor(value_t, torch.float64, "value", (W,))
        self._dev_tensor(grad_t, torch.float64, "grad", (W, self.ndim))
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_grad_workspace_bytes(self._h, max(W, 1), C.byref(nbytes)), "rbv_grad_workspace_bytes")
        if getattr(self, "_grad_ws", None) is None or self._grad_ws.numel() < nbytes.value:
            self._grad_ws = torch.empty(max(int(nbytes.value), 8), dtype=torch.uint8, device=self.tdev)
        check(self.lib.rbv_lnprob_grad_batch(self._h, theta_t.data_ptr(), W, int(bool(apply_prior)),
                                             value_t.data_ptr(), grad_t.data_ptr(), self._grad_ws.data_ptr(),
                                             self._grad_ws.numel(), self._stream()), "rbv_lnprob_grad_batch")
        return value_t, grad_t

    def lnprob_grad_host(self, theta: np.ndarray, apply_prior: bool):
        """HOST theta [W, ndim] -> HOST (value [W], gradient [W, ndim])."""
        torch = _torch()
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        if theta.ndim != 2:
            raise ValueError("theta must be [W, ndim]")
        th = torch.as_tensor(theta, device=self.tdev)
        v, g = self.lnprob_grad_device(th, apply_prior)
        return v.cpu().numpy(), g.cpu().numpy()

    # host calls split a batch so that the Jacobian workspace (about 2 * 3C * P doubles per row) stays below this
    fisher_chunk_bytes = 1 << 30

    def _fisher_ws(self, W: int):
        torch = _torch()
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_fisher_workspace_bytes(self._h, max(W, 1), C.byref(nbytes)), "rbv_fisher_workspace_bytes")
        if getattr(self, "_fisher_ws_t", None) is None or self._fisher_ws_t.numel() < nbytes.value:
            self._fisher_ws_t = None
            self._fisher_ws_t = torch.empty(max(int(nbytes.value), 8), dtype=torch.uint8, device=self.tdev)
        return self._fisher_ws_t

    def _fisher_rows_per_chunk(self) -> int:
        one = C.c_size_t(0)
        check(self.lib.rbv_fisher_workspace_bytes(self._h, 1, C.byref(one)), "rbv_fisher_workspace_bytes")
        return max(1, int(self.fisher_chunk_bytes // max(int(one.value), 1)))

    def lnlike_fisher_device(self, theta_t, value_t=None, grad_t=None, fisher_t=None):
        """DEVICE theta [W, ndim] -> (lnlike [W], gradient [W, ndim], Gauss-Newton matrix [W, ndim, ndim]) DEVICE
        tensors (``rbv_lnlike_fisher_batch``); asynchronous."""
        torch = _torch()
        self._dev_tensor(theta_t, torch.float64, "theta")
        if theta_t.dim() != 2 or theta_t.shape[1] != self.ndim:
            raise ValueError(f"theta must be [W, {self.ndim}]")
        W, n = int(theta_t.shape[0]), self.ndim
        if value_t is None:
            value_t = torch.empty(W, dtype=torch.float64, device=self.tdev)
        if grad_t is None:
            grad_t = torch.empty((W, n), dtype=torch.float64, device=self.tdev)
        if fisher_t is None:
            fisher_t = torch.empty((W, n, n), dtype=torch.float64, device=self.tdev)
        self._dev_tensor(value_t, torch.float64, "value", (W,))
        self._dev_tensor(grad_t, torch.float64, "grad", (W, n))
        self._dev_tensor(fisher_t, torch.float64, "fisher", (W, n, n))
        ws = self._fisher_ws(W)
        check(self.lib.rbv_lnlike_fisher_batch(self._h, theta_t.data_ptr(), W, value_t.data_ptr(), grad_t.data_ptr(),
                                               fisher_t.data_ptr(), ws.data_ptr(), ws.numel(), self._stream()),
              "rbv_lnlike_fisher_batch")
        return value_t, grad_t, fisher_t

    def lnlike_fisher_host(self, theta: np.ndarray):
        """HOST theta [W, ndim] -> HOST (lnlike [W], gradient [W, ndim], Gauss-Newton matrix [W, ndim, ndim]), in
        chunks of rows whose workspace stays below ``fisher_chunk_bytes`` (every row is reduced in an order of its
        own, so the chunking does not change any result)."""
        torch = _torch()
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        if theta.ndim != 2:
            raise ValueError("theta must be [W, ndim]")
        W, n = theta.shape[0], self.ndim
        value, grad, fisher = np.empty(W), np.empty((W, n)), np.empty((W, n, n))
        step = self._fisher_rows_per_chunk()
        for i in range(0, W, step):
            th = torch.as_tensor(theta[i:i + step], device=self.tdev)
            v, g, f = self.lnlike_fisher_device(th)
            value[i:i + step], grad[i:i + step], fisher[i:i + step] = v.cpu().numpy(), g.cpu().numpy(), f.cpu().numpy()
        return value, grad, fisher

    def model_jacobian(self, inst: int, theta: np.ndarray) -> np.ndarray:
        """HOST theta [W, ndim] -> HOST d(model flux)/d theta [W, ndim, P] of instrument ``inst``
        (``rbv_model_jacobian_batch``: the LSF-convolved model of ``model_flux``), in chunks as
        ``lnlike_fisher_host``."""
        torch = _torch()
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        if theta.ndim != 2 or theta.shape[1] != self.ndim:
            raise ValueError(f"theta must be [W, {self.ndim}]")
        if not 0 <= inst < len(self.pixels):
            raise ValueError("bad instrument index")
        W, n, P = theta.shape[0], self.ndim, self.pixels[inst]
        out = np.empty((W, n, P))
        step = self._fisher_rows_per_chunk()
        for i in range(0, W, step):
            th = torch.as_tensor(theta[i:i + step], device=self.tdev)
            w = th.shape[0]
            jac = torch.empty((w, n, P), dtype=torch.float64, device=self.tdev)
            ws = self._fisher_ws(w)
            check(self.lib.rbv_model_jacobian_batch(self._h, inst, th.data_ptr(), w, jac.data_ptr(), ws.data_ptr(),
                                                    ws.numel(), self._stream()), "rbv_model_jacobian_batch")
            out[i:i + step] = jac.cpu().numpy()
        return out

    def _sl_bytes(self, fn, n: int, what: str) -> int:
        nbytes = C.c_size_t(0)
        check(fn(self._h, max(int(n), 1), C.byref(nbytes)), what)
        return int(nbytes.value)

    def _sl_ws(self, nbytes: int):
        torch = _torch()
        if getattr(self, "_sl_ws_t", None) is None or self._sl_ws_t.numel() < nbytes:
            self._sl_ws_t = None
            self._sl_ws_t = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=self.tdev)
        return self._sl_ws_t

    def lnlike_fisher_sightlines_device(self, theta_t, wps: int):
        """Survey mode (``rbv_lnlike_fisher_batch_sightlines``): DEVICE theta [S * wps, ndim], ``wps`` consecutive rows
        per sightline -> DEVICE (lnlike [S * wps], gradient [S * wps, ndim], Gauss-Newton matrix [S * wps, ndim,
        ndim]); each row bit for bit what a one-sightline context gives.  Asynchronous."""
        torch = _torch()
        self._dev_tensor(theta_t, torch.float64, "theta")
        if theta_t.dim() != 2 or theta_t.shape[1] != self.ndim:
            raise ValueError(f"theta must be [W, {self.ndim}]")
        W, n = int(theta_t.shape[0]), self.ndim
        value_t = torch.empty(W, dtype=torch.float64, device=self.tdev)
        grad_t = torch.empty((W, n), dtype=torch.float64, device=self.tdev)
        fisher_t = torch.empty((W, n, n), dtype=torch.float64, device=self.tdev)
        ws = self._sl_ws(self._sl_bytes(self.lib.rbv_fisher_workspace_bytes_sightlines, W,
                                        "rbv_fisher_workspace_bytes_sightlines"))
        check(self.lib.rbv_lnlike_fisher_batch_sightlines(self._h, theta_t.data_ptr(), W, int(wps), value_t.data_ptr(),
                                                          grad_t.data_ptr(), fisher_t.data_ptr(), ws.data_ptr(),
                                                          ws.numel(), self._stream()),
              "rbv_lnlike_fisher_batch_sightlines")
        return value_t, grad_t, fisher_t

    def lnlike_fisher_sightlines_host(self, theta: np.ndarray, wps: int):
        """HOST theta [S * wps, ndim] (``wps`` consecutive rows per sightline) -> HOST (lnlike, gradient, Gauss-Newton
        matrix).  The launch always covers every sightline, so a batch whose workspace would pass
        ``fisher_chunk_bytes`` is split into blocks of walkers of every sightline (down to one row per sightline);
        each row's results do not depend on the batch."""
        torch = _torch()
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        S, wps = len(self.pixels), int(wps)
        if theta.ndim != 2 or theta.shape != (S * wps, self.ndim) or wps <= 0:
            raise ValueError(f"theta must be [{S} * walkers_per_sightline, {self.ndim}]")
        n = self.ndim
        one = self._sl_bytes(self.lib.rbv_fisher_workspace_bytes_sightlines, S, "rbv_fisher_workspace_bytes_sightlines")
        step = max(1, int(self.fisher_chunk_bytes // max(one, 1)))
        th3 = theta.reshape(S, wps, n)
        value, grad, fisher = np.empty((S, wps)), np.empty((S, wps, n)), np.empty((S, wps, n, n))
        for j in range(0, wps, step):
            c = min(step, wps - j)
            th = torch.as_tensor(np.ascontiguousarray(th3[:, j:j + c]).reshape(S * c, n), device=self.tdev)
            v, g, f = self.lnlike_fisher_sightlines_device(th, c)
            value[:, j:j + c] = v.cpu().numpy().reshape(S, c)
            grad[:, j:j + c] = g.cpu().numpy().reshape(S, c, n)
            fisher[:, j:j + c] = f.cpu().numpy().reshape(S, c, n, n)
        return value.reshape(S * wps), grad.reshape(S * wps, n), fisher.reshape(S * wps, n, n)

    def lm_sightlines(self, theta0: np.ndarray, first: int, n: int, max_evals: int = 200, ftol: float = 1e-10,
                      xtol: float = 1e-10):
        """Levenberg-Marquardt fits of sightlines [first, first + n) on the device (``rbv_lm_run_sightlines``):
        HOST theta0 [n, ndim] -> HOST (x [n, ndim], chi2 [n], cov [n, ndim, ndim], n_evals [n], status [n],
        flags [n]).  Runs in blocks of whole sightlines whose workspace stays below ``fisher_chunk_bytes``: the
        sightlines are independent, so the blocks do not change any result."""
        torch = _torch()
        theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
        nd, first, n = self.ndim, int(first), int(n)
        if theta0.shape != (n, nd):
            raise ValueError(f"theta0 must be [{n}, {nd}]")
        ctl = _lib.RbvLMControl(int(max_evals), float(ftol), float(xtol))
        one = self._sl_bytes(self.lib.rbv_lm_workspace_bytes_sightlines, 1, "rbv_lm_workspace_bytes_sightlines")
        step = max(1, int(self.fisher_chunk_bytes // max(one, 1)))
        x, chi2, cov = theta0.copy(), np.empty(n), np.empty((n, nd, nd))
        n_evals, status, flags = (np.empty(n, dtype=np.int32) for _ in range(3))
        for b in range(0, n, step):
            c = min(step, n - b)
            th = torch.as_tensor(theta0[b:b + c], device=self.tdev)
            ch = torch.empty(c, dtype=torch.float64, device=self.tdev)
            cv = torch.empty((c, nd, nd), dtype=torch.float64, device=self.tdev)
            ne, st, fl = (torch.empty(c, dtype=torch.int32, device=self.tdev) for _ in range(3))
            ws = self._sl_ws(self._sl_bytes(self.lib.rbv_lm_workspace_bytes_sightlines, c,
                                            "rbv_lm_workspace_bytes_sightlines"))
            check(self.lib.rbv_lm_run_sightlines(self._h, first + b, c, th.data_ptr(), C.byref(ctl), ch.data_ptr(),
                                                 cv.data_ptr(), ne.data_ptr(), st.data_ptr(), fl.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), self._stream()), "rbv_lm_run_sightlines")
            x[b:b + c], chi2[b:b + c], cov[b:b + c] = th.cpu().numpy(), ch.cpu().numpy(), cv.cpu().numpy()
            n_evals[b:b + c], status[b:b + c], flags[b:b + c] = ne.cpu().numpy(), st.cpu().numpy(), fl.cpu().numpy()
        return x, chi2, cov, n_evals, status, flags

    def voigt_h_grad(self, x: np.ndarray, a: np.ndarray):
        """H, dH/dx, dH/da on a lattice (``rbv_voigt_h_grad``, test hook)."""
        torch = _torch()
        xs = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64).ravel(), device=self.tdev)
        as_ = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64).ravel(), device=self.tdev)
        H, Hx, Ha = (torch.empty_like(xs) for _ in range(3))
        check(self.lib.rbv_voigt_h_grad(self._h, xs.data_ptr(), as_.data_ptr(), H.data_ptr(), Hx.data_ptr(),
                                        Ha.data_ptr(), xs.numel(), self._stream()), "rbv_voigt_h_grad")
        return tuple(t.cpu().numpy().reshape(np.shape(x)) for t in (H, Hx, Ha))

    def lnlike_host(self, theta: np.ndarray) -> np.ndarray:
        """HOST theta [W, ndim] -> HOST lnlike [W] (``rbv_lnlike_batch``: the same launch without the prior)."""
        torch = _torch()
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        W, ndim = theta.shape
        if ndim != self.ndim:
            raise ValueError(f"theta has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._reserve(W, ndim, sightlines=False)
        th = torch.as_tensor(theta, device=self.tdev)
        out = torch.empty(W, dtype=torch.float64, device=self.tdev)
        check(self.lib.rbv_lnlike_batch(self._h, th.data_ptr(), W, out.data_ptr(), self._ws.data_ptr(), self._ws_bytes,
                                        self._stream()), "rbv_lnlike_batch")
        return out.cpu().numpy()

    def lnprob_sightlines_host(self, theta: np.ndarray, wps: int) -> np.ndarray:
        """HOST theta [S * wps, ndim] (wps consecutive rows per sightline) -> HOST lnprob [S * wps]."""
        torch = _torch()
        th = torch.from_numpy(np.ascontiguousarray(theta, dtype=np.float64))
        # a page-locked array (pinned_theta) is read in place by the copy engine; a pageable one is staged by the driver
        out = self.lnprob_sightlines_device(th.to(self.tdev, non_blocking=True), wps)
        W = out.shape[0]
        if getattr(self, "_sl_out_pin", None) is None or self._sl_out_pin.shape[0] < W:
            self._sl_out_pin = torch.empty(W, dtype=torch.float64, pin_memory=True)
        host = self._sl_out_pin[:W]
        host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(self.tdev).synchronize()
        return host.numpy().copy()

    def lnprob_sightlines_device(self, theta_t, wps: int, out_t=None):
        torch = _torch()
        self._dev_tensor(theta_t, torch.float64, "theta")
        W, ndim = theta_t.shape
        if ndim != self.ndim:
            raise ValueError(f"theta has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._reserve(W, ndim, sightlines=True)
        if out_t is None:
            out_t = torch.empty(W, dtype=torch.float64, device=self.tdev)
        self._dev_tensor(out_t, torch.float64, "out", (W,))
        check(self.lib.rbv_lnprob_batch_sightlines(self._h, theta_t.data_ptr(), W, int(wps), out_t.data_ptr(),
                                                   self._ws.data_ptr(), self._ws_bytes, self._stream()),
              "rbv_lnprob_batch_sightlines")
        return out_t

    def stretch_run(self, coords_t, lnp_t, n_steps: int, a: float, seed: int, first_step: int, chain_t, lnp_chain_t,
                    n_accepted_t, flag_t, use_graph: bool = True):
        """Device-resident stretch-move sampling (rbv_stretch_run): every tensor stays on the device; runs on the
        current torch stream (a CUDA graph needs a non-default one)."""
        torch = _torch()
        W, ndim = coords_t.shape
        if ndim != self.ndim:
            raise ValueError(f"coords has {ndim} columns, bounds were set for ndim={self.ndim}")
        for t, dt in ((coords_t, torch.float64), (lnp_t, torch.float64), (n_accepted_t, torch.int32),
                      (flag_t, torch.int32)):
            if t.dtype != dt or not t.is_contiguous() or t.device != self.tdev:
                raise ValueError("sampler state tensors must be contiguous, on the engine's device, f64 / i32")
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), W))
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_stretch_workspace_bytes(self._h, W, C.byref(nbytes)), "rbv_stretch_workspace_bytes")
        if self._stretch_ws is None or self._stretch_ws.numel() < nbytes.value:
            self._stretch_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        check(self.lib.rbv_stretch_run(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), W, int(n_steps), float(a),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step),
            chain_t.data_ptr() if chain_t is not None else None,
            lnp_chain_t.data_ptr() if lnp_chain_t is not None else None,
            n_accepted_t.data_ptr(), flag_t.data_ptr(), self._stretch_ws.data_ptr(), self._stretch_ws.numel(),
            int(bool(use_graph)), self._stream()), "rbv_stretch_run")

    def _stretch_workspace(self, W: int):
        torch = _torch()
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_stretch_workspace_bytes(self._h, W, C.byref(nbytes)), "rbv_stretch_workspace_bytes")
        if self._stretch_ws is None or self._stretch_ws.numel() < nbytes.value:
            self._stretch_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        return self._stretch_ws

    def stretch_propose_eval(self, coords_t, a: float, seed: int, step: int, split: int, row_lo: int, row_hi: int,
                             lnp_rows_t):
        """Multi-GPU half-step, first part (rbv_stretch_propose_eval): all proposals of the half, lnprob of rows
        [row_lo, row_hi) into ``lnp_rows_t``; asynchronous on the current stream."""
        torch = _torch()
        self._dev_tensor(coords_t, torch.float64, "coords")
        self._dev_tensor(lnp_rows_t, torch.float64, "lnprob rows")
        ws = self._stretch_workspace(coords_t.shape[0])
        check(self.lib.rbv_stretch_propose_eval(self._h, coords_t.data_ptr(), coords_t.shape[0], float(a),
                                                int(seed) & 0xFFFFFFFFFFFFFFFF, int(step), int(split), int(row_lo),
                                                int(row_hi), lnp_rows_t.data_ptr(), ws.data_ptr(), ws.numel(),
                                                self._stream()), "rbv_stretch_propose_eval")

    def stretch_accept(self, coords_t, lnp_t, a: float, seed: int, step: int, split: int, lnp_rows_t, chain_row_t,
                       lnp_chain_row_t, n_accepted_t, flag_t):
        """Multi-GPU half-step, second part (rbv_stretch_accept), after the all-gather of ``lnp_rows_t``."""
        torch = _torch()
        W = coords_t.shape[0]
        self._dev_tensor(coords_t, torch.float64, "coords")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (W,))
        self._dev_tensor(lnp_rows_t, torch.float64, "lnprob rows")
        self._dev_tensor(chain_row_t, torch.float64, "chain row", (W, coords_t.shape[1]))
        self._dev_tensor(lnp_chain_row_t, torch.float64, "lnprob chain row", (W,))
        self._dev_tensor(n_accepted_t, torch.int32, "n_accepted", (W,))
        self._dev_tensor(flag_t, torch.int32, "flag")
        ws = self._stretch_workspace(coords_t.shape[0])
        check(self.lib.rbv_stretch_accept(self._h, coords_t.data_ptr(), lnp_t.data_ptr(), coords_t.shape[0], float(a),
                                          int(seed) & 0xFFFFFFFFFFFFFFFF, int(step), int(split),
                                          lnp_rows_t.data_ptr(),
                                          chain_row_t.data_ptr() if chain_row_t is not None else None,
                                          lnp_chain_row_t.data_ptr() if lnp_chain_row_t is not None else None,
                                          n_accepted_t.data_ptr(), flag_t.data_ptr(), ws.data_ptr(), ws.numel(),
                                          self._stream()), "rbv_stretch_accept")

    # ------------------------------------------------------------------ multi-GPU (collective inside the library)
    def comm_init(self, group=None):
        """Collective over the ranks of ``group`` (default: the world group): attach this context to an NCCL
        communicator of its own (``rbv_comm_init``).  Rank 0 creates the unique id; it travels through
        ``torch.distributed.broadcast``.  Afterwards ``lnprob_allgather_device`` / ``stretch_run_dist`` /
        ``slice_run`` split their rows over the ranks and all-gather inside the library."""
        torch = _torch()
        import torch.distributed as dist
        if not dist.is_initialized() or dist.get_world_size(group) == 1:
            return False
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        ident = (C.c_ubyte * 128)()
        if rank == 0:
            check(self.lib.rbv_comm_unique_id(ident), "rbv_comm_unique_id")
        t = torch.tensor(list(ident), dtype=torch.uint8)
        on_gpu = dist.get_backend(group) == "nccl"
        if on_gpu:
            t = t.to(self.tdev)
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        ident = (C.c_ubyte * 128)(*t.cpu().tolist())
        check(self.lib.rbv_comm_init(self._h, ident, rank, world), "rbv_comm_init")
        self.comm_rank, self.comm_world = rank, world
        self._peer_attach(group, rank, world, on_gpu)
        return True

    def _peer_attach(self, group, rank, world, on_gpu):
        """The all-gather as one kernel over NVLink peer memory (``rbv_peer_export`` / ``rbv_peer_attach``): every
        rank's exchange block is mapped into every other rank through CUDA IPC; the 64-byte handles travel through
        ``torch.distributed.all_gather``.  Every rank takes the same decision (the outcome of the attach is reduced
        over the group): peer memory on all ranks or NCCL on all ranks.  ``RBVFIT_B200_PEER=0`` keeps NCCL."""
        torch = _torch()
        import torch.distributed as dist
        self.peer_attached = False
        if os.environ.get("RBVFIT_B200_PEER", "1") == "0" or not on_gpu or world > 16:
            return
        handle = (C.c_ubyte * 64)()
        ok = self.lib.rbv_peer_export(self._h, handle) == 0
        mine = torch.tensor(list(handle) + [1 if ok else 0], dtype=torch.uint8, device=self.tdev)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine, group=group)
        rows = [g.cpu().tolist() for g in gathered]
        if not all(r[64] for r in rows):
            return
        flat = (C.c_ubyte * (64 * world))(*[b for r in rows for b in r[:64]])
        ok = self.lib.rbv_peer_attach(self._h, flat, rank, world) == 0
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.tdev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 1:
            self.peer_attached = True
        elif ok:
            raise RbvError("rbv_peer_attach succeeded on this rank but failed on another: set RBVFIT_B200_PEER=0")

    def peer_error(self) -> int:
        """1 after a peer-memory all-gather gave up waiting for a rank (30 s without progress)."""
        att, err = C.c_int(0), C.c_int(0)
        check(self.lib.rbv_peer_info(self._h, C.byref(att), C.byref(err)), "rbv_peer_info")
        return int(err.value)

    @property
    def has_comm(self) -> bool:
        return self.comm_world > 1

    def lnprob_allgather_device(self, theta_t):
        """Replicated DEVICE theta [W, ndim] -> DEVICE lnprob [W], complete on every rank: this rank evaluates its
        rows, NCCL all-gather in place inside the library (``rbv_lnprob_batch_allgather``); asynchronous."""
        torch = _torch()
        self._dev_tensor(theta_t, torch.float64, "theta")
        W, ndim = theta_t.shape
        if ndim != self.ndim:
            raise ValueError(f"theta has {ndim} columns, bounds were set for ndim={self.ndim}")
        chunk = -(-W // self.comm_world)
        self._reserve(chunk, ndim, sightlines=False)
        out_t = torch.empty(chunk * self.comm_world, dtype=torch.float64, device=self.tdev)
        check(self.lib.rbv_lnprob_batch_allgather(self._h, theta_t.data_ptr(), W, out_t.data_ptr(), self._ws.data_ptr(),
                                                  self._ws_bytes, self._stream()), "rbv_lnprob_batch_allgather")
        return out_t[:W]

    def stretch_run_dist(self, coords_t, lnp_t, n_steps: int, a: float, seed: int, first_step: int, chain_t,
                         lnp_chain_t, n_accepted_t, flag_t, use_graph: bool = True):
        """``stretch_run`` over all ranks of the communicator (``rbv_stretch_run_dist``): replicated state, rows of
        every half-step split over the ranks, the lnprob all-gather inside the captured step."""
        torch = _torch()
        W, ndim = coords_t.shape
        if ndim != self.ndim:
            raise ValueError(f"coords has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._dev_tensor(coords_t, torch.float64, "coords")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (W,))
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), W))
        self._dev_tensor(n_accepted_t, torch.int32, "n_accepted", (W,))
        self._dev_tensor(flag_t, torch.int32, "flag")
        ws = self._stretch_workspace(W)
        check(self.lib.rbv_stretch_run_dist(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), W, int(n_steps), float(a),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step),
            chain_t.data_ptr() if chain_t is not None else None,
            lnp_chain_t.data_ptr() if lnp_chain_t is not None else None,
            n_accepted_t.data_ptr(), flag_t.data_ptr(), ws.data_ptr(), ws.numel(), int(bool(use_graph)),
            self._stream()), "rbv_stretch_run_dist")

    def stretch_run_to_host(self, coords_t, lnp_t, n_steps: int, a: float, seed: int, first_step: int,
                            n_accepted_t, flag_t, distributed: bool = False):
        """``stretch_run`` / ``stretch_run_dist`` with the chain delivered to the HOST while the run goes on
        (``rbv_stretch_run_sink``): returns (chain [n_steps, W, ndim], lnprob chain [n_steps, W]) as numpy arrays.
        The device only holds a ring of two blocks of steps; its halves travel through page-locked staging on a copy
        stream and are unpacked by this thread under the next block's kernels -- no pageable device-to-host copy
        (2 GB/s, measured) and no device time."""
        torch = _torch()
        W, ndim = coords_t.shape
        if ndim != self.ndim:
            raise ValueError(f"coords has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._dev_tensor(coords_t, torch.float64, "coords")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (W,))
        self._dev_tensor(n_accepted_t, torch.int32, "n_accepted", (W,))
        self._dev_tensor(flag_t, torch.int32, "flag")
        row = W * (ndim + 1)
        K = int(min(256, max(1, (6 << 20) // (row * 8)), max(1, (int(n_steps) + 1) // 2)))   # ~6 MB blocks
        need = 2 * K * row
        if self._sink_ring is None or self._sink_ring[0] != K or self._sink_ring[1].numel() < need:
            self._sink_ring = (K, torch.empty(need, dtype=torch.float64, device=self.tdev),
                               torch.empty(need, dtype=torch.float64, pin_memory=True))
        _k, ring_dev, ring_pin = self._sink_ring
        chain = np.empty((int(n_steps), W, ndim), dtype=np.float64)
        lps = np.empty((int(n_steps), W), dtype=np.float64)
        sink = RbvChainSink(chain.ctypes.data, lps.ctypes.data, ring_dev.data_ptr(), ring_pin.data_ptr(), K)
        ws = self._stretch_workspace(W)
        check(self.lib.rbv_stretch_run_sink(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), W, int(n_steps), float(a),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step), C.byref(sink), n_accepted_t.data_ptr(),
            flag_t.data_ptr(), ws.data_ptr(), ws.numel(), int(bool(distributed)), self._stream()),
            "rbv_stretch_run_sink")
        return chain, lps

    def stretch_run_sightlines(self, coords_t, lnp_t, n_steps: int, a: float, seed: int, first_step: int, chain_t,
                               lnp_chain_t, n_accepted_t, flag_t):
        """Survey-mode stretch move (rbv_stretch_run_sightlines): ``coords_t`` [S, W, ndim], one ensemble per
        sightline of this context, all advancing in lockstep on the current torch stream; asynchronous."""
        torch = _torch()
        S, W, ndim = coords_t.shape
        if ndim != self.ndim or S != len(self.pixels):
            raise ValueError(f"coords must be [{len(self.pixels)}, walkers_per_sightline, {self.ndim}]")
        for t, dt in ((coords_t, torch.float64), (lnp_t, torch.float64), (n_accepted_t, torch.int32),
                      (flag_t, torch.int32)):
            if t.dtype != dt or not t.is_contiguous() or t.device != self.tdev:
                raise ValueError("sampler state tensors must be contiguous, on the engine's device, f64 / i32")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (S, W))
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), S, W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), S, W))
        self._dev_tensor(n_accepted_t, torch.int32, "n_accepted", (S, W))
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_stretch_workspace_bytes_sightlines(self._h, W, C.byref(nbytes)),
              "rbv_stretch_workspace_bytes_sightlines")
        if self._stretch_ws is None or self._stretch_ws.numel() < nbytes.value:
            self._stretch_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        check(self.lib.rbv_stretch_run_sightlines(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), W, int(n_steps), float(a),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step),
            chain_t.data_ptr() if chain_t is not None else None,
            lnp_chain_t.data_ptr() if lnp_chain_t is not None else None,
            n_accepted_t.data_ptr(), flag_t.data_ptr(), self._stretch_ws.data_ptr(), self._stretch_ws.numel(),
            self._stream()), "rbv_stretch_run_sightlines")

    def _pt_checks(self, coords_t, lnp_t, betas_t, n_steps, beta_hist_t, n_accepted_t, n_swaps_t, flag_t):
        torch = _torch()
        if coords_t.dim() != 3:
            raise ValueError("coords must be [n_temps, n_walkers, ndim]")
        T, W, ndim = coords_t.shape
        if ndim != self.ndim:
            raise ValueError(f"coords has {ndim} columns, bounds were set for ndim={self.ndim}")
        self._dev_tensor(coords_t, torch.float64, "coords")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (T, W))
        self._dev_tensor(betas_t, torch.float64, "betas", (T,))
        self._dev_tensor(beta_hist_t, torch.float64, "beta history", (int(n_steps), T))
        self._dev_tensor(n_accepted_t, torch.int32, "n_accepted", (T, W))
        self._dev_tensor(n_swaps_t, torch.int64, "n_swaps_accepted", (max(T - 1, 1),))
        self._dev_tensor(flag_t, torch.int32, "flag")
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_pt_workspace_bytes(self._h, T, W, C.byref(nbytes)), "rbv_pt_workspace_bytes")
        if self._stretch_ws is None or self._stretch_ws.numel() < nbytes.value:
            self._stretch_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        return T, W, ndim

    def _pt_call(self, coords_t, lnp_t, betas_t, T, W, n_steps, a, seed, first_step, chain_p, lnp_chain_p, sink,
                 beta_hist_t, n_accepted_t, n_swaps_t, flag_t, use_graph, adapt, adaptation_lag, adaptation_time,
                 adapt_steps_done, n_record):
        ctl = RbvPtControl(float(a), int(bool(adapt)), float(adaptation_lag), float(adaptation_time),
                           int(adapt_steps_done), int(n_record))
        check(self.lib.rbv_pt_run(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), betas_t.data_ptr(), T, W, int(n_steps), C.byref(ctl),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step), chain_p, lnp_chain_p, sink,
            beta_hist_t.data_ptr() if beta_hist_t is not None else None, n_accepted_t.data_ptr(),
            n_swaps_t.data_ptr(), flag_t.data_ptr(), self._stretch_ws.data_ptr(), self._stretch_ws.numel(),
            int(bool(use_graph)), self._stream()), "rbv_pt_run")

    def pt_run(self, coords_t, lnp_t, betas_t, n_steps: int, a: float, seed: int, first_step: int, chain_t,
               lnp_chain_t, beta_hist_t, n_accepted_t, n_swaps_t, flag_t, use_graph: bool = True, adapt: bool = False,
               adaptation_lag: float = 10000.0, adaptation_time: float = 100.0, adapt_steps_done: int = 0,
               n_record: int = 1):
        """Parallel tempering on the device (rbv_pt_run): ``coords_t`` [T, W, ndim], ``lnp_t`` [T, W] (untempered),
        ``betas_t`` [T] (in/out); ``chain_t`` [n_steps, n_record, W, ndim], ``lnp_chain_t`` [n_steps, T, W] and
        ``beta_hist_t`` [n_steps, T] may be None; ``n_swaps_t`` int64 [max(T - 1, 1)] (the library's uint64
        counters).  Every tensor stays on the device; runs on the current torch stream."""
        torch = _torch()
        T, W, ndim = self._pt_checks(coords_t, lnp_t, betas_t, n_steps, beta_hist_t, n_accepted_t, n_swaps_t, flag_t)
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), int(n_record), W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), T, W))
        self._pt_call(coords_t, lnp_t, betas_t, T, W, n_steps, a, seed, first_step,
                      chain_t.data_ptr() if chain_t is not None else None,
                      lnp_chain_t.data_ptr() if lnp_chain_t is not None else None, None, beta_hist_t, n_accepted_t,
                      n_swaps_t, flag_t, use_graph, adapt, adaptation_lag, adaptation_time, adapt_steps_done,
                      n_record)

    def pt_run_to_host(self, coords_t, lnp_t, betas_t, n_steps: int, a: float, seed: int, first_step: int,
                       beta_hist_t, n_accepted_t, n_swaps_t, flag_t, adapt: bool = False,
                       adaptation_lag: float = 10000.0, adaptation_time: float = 100.0, adapt_steps_done: int = 0,
                       n_record: int = 1):
        """``pt_run`` with the chain delivered to the HOST while the run goes on (the chain sink of
        ``stretch_run_to_host``): returns (chain [n_steps, n_record, W, ndim], lnprob chain [n_steps, T, W])."""
        torch = _torch()
        T, W, ndim = self._pt_checks(coords_t, lnp_t, betas_t, n_steps, beta_hist_t, n_accepted_t, n_swaps_t, flag_t)
        row = int(n_record) * W * ndim + T * W
        K = int(min(256, max(1, (6 << 20) // (row * 8)), max(1, (int(n_steps) + 1) // 2)))   # ~6 MB blocks
        need = 2 * K * row
        if self._sink_ring is None or self._sink_ring[0] != K or self._sink_ring[1].numel() < need:
            self._sink_ring = (K, torch.empty(need, dtype=torch.float64, device=self.tdev),
                               torch.empty(need, dtype=torch.float64, pin_memory=True))
        _k, ring_dev, ring_pin = self._sink_ring
        chain = np.empty((int(n_steps), int(n_record), W, ndim), dtype=np.float64)
        lps = np.empty((int(n_steps), T, W), dtype=np.float64)
        sink = RbvChainSink(chain.ctypes.data, lps.ctypes.data, ring_dev.data_ptr(), ring_pin.data_ptr(), K)
        self._pt_call(coords_t, lnp_t, betas_t, T, W, n_steps, a, seed, first_step, None, None, C.byref(sink),
                      beta_hist_t, n_accepted_t, n_swaps_t, flag_t, True, adapt, adaptation_lag, adaptation_time,
                      adapt_steps_done, n_record)
        return chain, lps

    def _pt_sl_checks(self, coords_t, lnp_t, betas_t, n_steps, beta_hist_t, ti_t, n_accepted_t, n_swaps_t, flag_t):
        torch = _torch()
        if coords_t.dim() != 4 or coords_t.shape[0] != len(self.pixels) or coords_t.shape[3] != self.ndim:
            raise ValueError(f"coords must be [{len(self.pixels)}, n_temps, walkers_per_sightline, {self.ndim}]")
        S, T, W, ndim = coords_t.shape
        self._dev_tensor(coords_t, torch.float64, "coords")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (S, T, W))
        self._dev_tensor(betas_t, torch.float64, "betas", (S, T))
        self._dev_tensor(beta_hist_t, torch.float64, "beta history", (int(n_steps), S, T))
        self._dev_tensor(ti_t, torch.float64, "ti_moments", (S, T, 3))
        self._dev_tensor(n_accepted_t, torch.int32, "n_accepted", (S, T, W))
        self._dev_tensor(n_swaps_t, torch.int64, "n_swaps_accepted", (S, max(T - 1, 1)))
        self._dev_tensor(flag_t, torch.int32, "flag")
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_pt_workspace_bytes_sightlines(self._h, T, W, C.byref(nbytes)),
              "rbv_pt_workspace_bytes_sightlines")
        if self._stretch_ws is None or self._stretch_ws.numel() < nbytes.value:
            self._stretch_ws = None
            self._stretch_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        return S, T, W, ndim

    def _pt_sl_call(self, coords_t, lnp_t, betas_t, T, W, n_steps, a, seed, first_step, chain_p, lnp_chain_p, sink,
                    beta_hist_t, ti_t, n_accepted_t, n_swaps_t, flag_t, use_graph, adapt, adaptation_lag,
                    adaptation_time, adapt_steps_done, n_record):
        ctl = RbvPtControl(float(a), int(bool(adapt)), float(adaptation_lag), float(adaptation_time),
                           int(adapt_steps_done), int(n_record))
        check(self.lib.rbv_pt_run_sightlines(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), betas_t.data_ptr(), T, W, int(n_steps), C.byref(ctl),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step), chain_p, lnp_chain_p, sink,
            beta_hist_t.data_ptr() if beta_hist_t is not None else None,
            ti_t.data_ptr() if ti_t is not None else None, n_accepted_t.data_ptr(), n_swaps_t.data_ptr(),
            flag_t.data_ptr(), self._stretch_ws.data_ptr(), self._stretch_ws.numel(), int(bool(use_graph)),
            self._stream()), "rbv_pt_run_sightlines")

    def pt_run_sightlines(self, coords_t, lnp_t, betas_t, n_steps: int, a: float, seed: int, first_step: int,
                          chain_t, lnp_chain_t, beta_hist_t, ti_t, n_accepted_t, n_swaps_t, flag_t,
                          use_graph: bool = True, adapt: bool = False, adaptation_lag: float = 10000.0,
                          adaptation_time: float = 100.0, adapt_steps_done: int = 0, n_record: int = 1):
        """Survey-mode parallel tempering (rbv_pt_run_sightlines): ``coords_t`` [S, T, W, ndim], one tempered
        ladder of ensembles per sightline of this context, all advancing in lockstep; ``lnp_t`` [S, T, W]
        (untempered), ``betas_t`` [S, T] (in/out); ``chain_t`` [n_steps, S, n_record, W, ndim], ``lnp_chain_t``
        [n_steps, S, T, W], ``beta_hist_t`` [n_steps, S, T] and ``ti_t`` [S, T, 3] (the accumulated (n, mean, M2)
        of ln L; refused with ``adapt``) may be None; ``n_accepted_t`` int32 [S, T, W], ``n_swaps_t`` int64
        [S, max(T - 1, 1)].  Every tensor stays on the device; runs on the current torch stream."""
        torch = _torch()
        S, T, W, ndim = self._pt_sl_checks(coords_t, lnp_t, betas_t, n_steps, beta_hist_t, ti_t, n_accepted_t,
                                           n_swaps_t, flag_t)
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), S, int(n_record), W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), S, T, W))
        self._pt_sl_call(coords_t, lnp_t, betas_t, T, W, n_steps, a, seed, first_step,
                         chain_t.data_ptr() if chain_t is not None else None,
                         lnp_chain_t.data_ptr() if lnp_chain_t is not None else None, None, beta_hist_t, ti_t,
                         n_accepted_t, n_swaps_t, flag_t, use_graph, adapt, adaptation_lag, adaptation_time,
                         adapt_steps_done, n_record)

    def pt_run_sightlines_to_host(self, coords_t, lnp_t, betas_t, n_steps: int, a: float, seed: int,
                                  first_step: int, beta_hist_t, ti_t, n_accepted_t, n_swaps_t, flag_t,
                                  adapt: bool = False, adaptation_lag: float = 10000.0, adaptation_time: float = 100.0,
                                  adapt_steps_done: int = 0, n_record: int = 1, record_chain: bool = True,
                                  record_log_like: bool = True):
        """``pt_run_sightlines`` with the chain delivered to the HOST while the run goes on (the chain sink of
        ``pt_run_to_host``): returns (chain [n_steps, S, n_record, W, ndim] or None, lnprob chain [n_steps, S, T, W]
        or None).  Without ``record_log_like`` no lnprob row is recorded or copied."""
        torch = _torch()
        S, T, W, ndim = self._pt_sl_checks(coords_t, lnp_t, betas_t, n_steps, beta_hist_t, ti_t, n_accepted_t,
                                           n_swaps_t, flag_t)
        row = S * int(n_record) * W * ndim + (S * T * W if record_log_like else 0)
        K = int(min(256, max(1, (6 << 20) // (row * 8)), max(1, (int(n_steps) + 1) // 2)))   # ~6 MB blocks
        need = 2 * K * row
        if self._sink_ring is None or self._sink_ring[0] != K or self._sink_ring[1].numel() < need:
            self._sink_ring = None
            self._sink_ring = (K, torch.empty(need, dtype=torch.float64, device=self.tdev),
                               torch.empty(need, dtype=torch.float64, pin_memory=True))
        _k, ring_dev, ring_pin = self._sink_ring
        chain = np.empty((int(n_steps), S, int(n_record), W, ndim), dtype=np.float64) if record_chain else None
        lps = np.empty((int(n_steps), S, T, W), dtype=np.float64) if record_log_like else None
        sink = RbvChainSink(chain.ctypes.data if chain is not None else None,
                            lps.ctypes.data if lps is not None else None, ring_dev.data_ptr(), ring_pin.data_ptr(), K)
        self._pt_sl_call(coords_t, lnp_t, betas_t, T, W, n_steps, a, seed, first_step, None, None, C.byref(sink),
                         beta_hist_t, ti_t, n_accepted_t, n_swaps_t, flag_t, True, adapt, adaptation_lag,
                         adaptation_time, adapt_steps_done, n_record)
        return chain, lps

    def slice_run(self, coords_t, lnp_t, n_steps: int, tuning, seed: int, first_step: int, chain_t, lnp_chain_t,
                  flag_t, use_graph: bool = True) -> np.ndarray:
        """Device-resident ensemble slice sampling (rbv_slice_run) on the current torch stream; ``tuning`` is an
        ``RbvSliceTuning`` updated in place.  ``use_graph``: the per-half-step loop is a CUDA-graph WHILE node (needs
        a non-default stream), otherwise the host polls the device counters.  Returns mu after each step; the call
        returns when the run is done."""
        torch = _torch()
        W, ndim = coords_t.shape
        if ndim != self.ndim:
            raise ValueError(f"coords has {ndim} columns, bounds were set for ndim={self.ndim}")
        for t, dt in ((coords_t, torch.float64), (lnp_t, torch.float64), (flag_t, torch.int32)):
            if t.dtype != dt or not t.is_contiguous() or t.device != self.tdev:
                raise ValueError("sampler state tensors must be contiguous, on the engine's device, f64 / i32")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (W,))
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), W))
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_slice_workspace_bytes(self._h, W, C.byref(nbytes)), "rbv_slice_workspace_bytes")
        if self._slice_ws is None or self._slice_ws.numel() < nbytes.value:
            self._slice_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        mus_t = torch.zeros(max(int(n_steps), 1), dtype=torch.float64, device=self.tdev)
        check(self.lib.rbv_slice_run(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), W, int(n_steps), C.byref(tuning),
            int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step),
            chain_t.data_ptr() if chain_t is not None else None,
            lnp_chain_t.data_ptr() if lnp_chain_t is not None else None,
            mus_t.data_ptr(), flag_t.data_ptr(), self._slice_ws.data_ptr(), self._slice_ws.numel(),
            int(bool(use_graph)), self._stream()), "rbv_slice_run")
        return mus_t.cpu().numpy()[:int(n_steps)]

    def slice_run_sightlines(self, coords_t, lnp_t, n_steps: int, tuning, mu_t, tune_good_t, totals_t, seed: int,
                             first_step: int, chain_t, lnp_chain_t, mu_history_t, flag_t, use_graph: bool = True):
        """Survey-mode ensemble slice sampling (rbv_slice_run_sightlines) on the current torch stream: ``coords_t``
        [S, W, ndim], one ensemble per sightline of this context, all advancing in lockstep.  ``tuning`` is an
        ``RbvSliceTuning`` carrying the settings every sightline shares (its ``n_batches`` is written); each
        sightline's state is on the device and updated in place: ``mu_t`` [S] f64, ``tune_good_t`` [S, 2] i32,
        ``totals_t`` [S, 3] i64 (expansions, contractions, likelihood rows; accumulated).  ``mu_history_t``
        [n_steps, S] or None.  The call returns when the run is done."""
        torch = _torch()
        S, W, ndim = coords_t.shape
        if ndim != self.ndim or S != len(self.pixels):
            raise ValueError(f"coords must be [{len(self.pixels)}, walkers_per_sightline, {self.ndim}]")
        for t, dt in ((coords_t, torch.float64), (lnp_t, torch.float64), (flag_t, torch.int32)):
            if t.dtype != dt or not t.is_contiguous() or t.device != self.tdev:
                raise ValueError("sampler state tensors must be contiguous, on the engine's device, f64 / i32")
        self._dev_tensor(lnp_t, torch.float64, "lnprob", (S, W))
        self._dev_tensor(mu_t, torch.float64, "mu", (S,))
        self._dev_tensor(tune_good_t, torch.int32, "tune / good", (S, 2))
        self._dev_tensor(totals_t, torch.int64, "totals", (S, 3))
        self._dev_tensor(chain_t, torch.float64, "chain", (int(n_steps), S, W, ndim))
        self._dev_tensor(lnp_chain_t, torch.float64, "lnprob chain", (int(n_steps), S, W))
        self._dev_tensor(mu_history_t, torch.float64, "mu history", (int(n_steps), S))
        nbytes = C.c_size_t(0)
        check(self.lib.rbv_slice_workspace_bytes_sightlines(self._h, W, C.byref(nbytes)),
              "rbv_slice_workspace_bytes_sightlines")
        if self._slice_ws is None or self._slice_ws.numel() < nbytes.value:
            self._slice_ws = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.tdev)
        check(self.lib.rbv_slice_run_sightlines(
            self._h, coords_t.data_ptr(), lnp_t.data_ptr(), W, int(n_steps), C.byref(tuning), mu_t.data_ptr(),
            tune_good_t.data_ptr(), totals_t.data_ptr(), int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_step),
            chain_t.data_ptr() if chain_t is not None else None,
            lnp_chain_t.data_ptr() if lnp_chain_t is not None else None,
            mu_history_t.data_ptr() if mu_history_t is not None else None,
            flag_t.data_ptr(), self._slice_ws.data_ptr(), self._slice_ws.numel(), int(bool(use_graph)),
            self._stream()), "rbv_slice_run_sightlines")

    def model_flux(self, inst: int, theta: np.ndarray, convolve: bool = True) -> np.ndarray:
        """HOST theta [W, ndim] -> HOST model flux [W, P] of instrument ``inst``; ``convolve=False`` skips the LSF
        (``VoigtModel.evaluate(return_unconvolved=True)``)."""
        torch = _torch()
        cols = self.ndim if self.ndim else 3 * self.components[inst]
        theta = np.asarray(theta, dtype=np.float64)
        if theta.ndim != 2 or theta.shape[1] < cols:
            raise ValueError(f"theta must be [W, >= {cols}]")
        th = torch.as_tensor(np.ascontiguousarray(theta[:, :cols]), device=self.tdev)
        W = th.shape[0]
        out = torch.empty((W, self.pixels[inst]), dtype=torch.float64, device=self.tdev)
        ws, ws_bytes = None, 0
        if W >= 4:      # line constants once per walker instead of once per CTA
            nbytes = C.c_size_t(0)
            check(self.lib.rbv_flux_workspace_bytes(self._h, inst, W, C.byref(nbytes)), "rbv_flux_workspace_bytes")
            ws = torch.empty(max(int(nbytes.value), 8), dtype=torch.uint8, device=self.tdev)
            ws_bytes = int(nbytes.value)
        check(self.lib.rbv_model_flux_batch(self._h, inst, th.data_ptr(), W, int(bool(convolve)), out.data_ptr(),
                                            ws.data_ptr() if ws is not None else None, ws_bytes, self._stream()),
              "rbv_model_flux_batch")
        return out.cpu().numpy()

    def voigt_h(self, x: np.ndarray, a: np.ndarray, method: str = "wofz") -> np.ndarray:
        torch = _torch()
        xs = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64).ravel(), device=self.tdev)
        as_ = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64).ravel(), device=self.tdev)
        out = torch.empty_like(xs)
        check(self.lib.rbv_voigt_h(self._h, xs.data_ptr(), as_.data_ptr(), out.data_ptr(), xs.numel(),
                                   VOIGT_METHODS[method], self._stream()), "rbv_voigt_h")
        return out.cpu().numpy().reshape(np.shape(x))

    # ------------------------------------------------------------------ introspection
    @property
    def n_tiles(self) -> int:
        return self.lib.rbv_num_tiles(self._h)

    @property
    def launch_count(self) -> int:
        return int(self.lib.rbv_launch_count(self._h))

    @property
    def last_kernel(self):
        """'tile' / 'stream': the kernel the most recent lnprob launch used (None before the first)."""
        return {0: "tile", 1: "stream"}.get(self.lib.rbv_last_kernel(self._h))

    def measure_fp64_peak(self, millis: float = 200.0) -> float:
        out = C.c_double(0.0)
        check(self.lib.rbv_measure_fp64_peak(self._h, float(millis), C.byref(out)), "rbv_measure_fp64_peak")
        return out.value

    def selftest_rcp(self) -> float:
        out = C.c_double(0.0)
        check(self.lib.rbv_selftest_rcp(self._h, C.byref(out)), "rbv_selftest_rcp")
        return out.value
