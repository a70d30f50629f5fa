"""ctypes binding of include/rbvfit_b200.h.  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

_lib = None


class RbvError(RuntimeError):
    pass


class RbvLineTable(C.Structure):
    _fields_ = [("n_lines", C.c_int), ("n_components", C.c_int),
                ("lambda0", C.POINTER(C.c_double)), ("gamma", C.POINTER(C.c_double)),
                ("f", C.POINTER(C.c_double)), ("zfac", C.POINTER(C.c_double)),
                ("comp", C.POINTER(C.c_int)), ("voigt_method", C.c_int)]


class RbvSpectrum(C.Structure):
    _fields_ = [("n_pixels", C.c_int), ("wave", C.c_void_p), ("flux", C.c_void_p),
                ("inv_sigma2", C.c_void_p), ("log_inv_sigma2", C.c_void_p), ("inv_wave", C.c_void_p),
                ("taps", C.POINTER(C.c_double)), ("n_taps", C.c_int), ("normalize_taps", C.c_int)]


class RbvSliceTuning(C.Structure):
    _fields_ = [("mu", C.c_double), ("tolerance", C.c_double), ("tune", C.c_int), ("good", C.c_int),
                ("patience", C.c_int), ("maxsteps", C.c_int), ("maxiter", C.c_int), ("depth", C.c_int),
                ("n_expansions", C.c_ulonglong), ("n_contractions", C.c_ulonglong), ("n_calls", C.c_ulonglong),
                ("n_batches", C.c_ulonglong)]


class RbvLMControl(C.Structure):
    _fields_ = [("max_evals", C.c_int), ("ftol", C.c_double), ("xtol", C.c_double)]


class RbvChainSink(C.Structure):
    _fields_ = [("chain_host", C.c_void_p), ("lnprob_chain_host", C.c_void_p), ("ring_dev", C.c_void_p),
                ("ring_pinned", C.c_void_p), ("block_steps", C.c_int)]


class RbvPtControl(C.Structure):
    _fields_ = [("a", C.c_double), ("adapt", C.c_int), ("adaptation_lag", C.c_double),
                ("adaptation_time", C.c_double), ("adapt_steps_done", C.c_ulonglong), ("n_record", C.c_int)]


EXPORTS = {
    # name: (restype, argtypes)
    "rbv_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "rbv_destroy": (None, [C.c_void_p]),
    "rbv_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "rbv_set_farfield": (C.c_int, [C.c_void_p, C.c_int]),
    "rbv_add_instrument": (C.c_int, [C.c_void_p, C.POINTER(RbvLineTable), C.POINTER(RbvSpectrum),
                                     C.POINTER(C.c_int)]),
    "rbv_set_bounds": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int]),
    "rbv_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_lnprob_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                   C.c_void_p]),
    "rbv_lnlike_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                   C.c_void_p]),
    "rbv_workspace_bytes_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_lnprob_batch_sightlines": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                              C.c_size_t, C.c_void_p]),
    "rbv_lnprob_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_stretch_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_stretch_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_ulonglong,
                                  C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_stretch_propose_eval": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_ulonglong, C.c_ulonglong,
                                           C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_stretch_accept": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_ulonglong,
                                     C.c_ulonglong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_comm_unique_id": (C.c_int, [C.c_void_p]),
    "rbv_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "rbv_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "rbv_host_pinned": (C.c_int, [C.c_void_p]),
    "rbv_peer_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rbv_peer_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "rbv_peer_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "rbv_lnprob_batch_allgather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                             C.c_void_p]),
    "rbv_stretch_run_dist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double,
                                       C.c_ulonglong, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_stretch_run_sink": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double,
                                       C.c_ulonglong, C.c_ulonglong, C.POINTER(RbvChainSink), C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_stretch_workspace_bytes_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_stretch_run_sightlines": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double,
                                             C.c_ulonglong, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_pt_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_pt_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                             C.POINTER(RbvPtControl), C.c_ulonglong, C.c_ulonglong, C.c_void_p, C.c_void_p,
                             C.POINTER(RbvChainSink), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_pt_workspace_bytes_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_pt_run_sightlines": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(RbvPtControl), C.c_ulonglong, C.c_ulonglong, C.c_void_p,
                                        C.c_void_p, C.POINTER(RbvChainSink), C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_slice_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_slice_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(RbvSliceTuning),
                                C.c_ulonglong, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_slice_workspace_bytes_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_slice_run_sightlines": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                           C.POINTER(RbvSliceTuning), C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_ulonglong, C.c_ulonglong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "rbv_flux_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_model_flux_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_num_instruments": (C.c_int, [C.c_void_p]),
    "rbv_num_tiles": (C.c_int, [C.c_void_p]),
    "rbv_ndim": (C.c_int, [C.c_void_p]),
    "rbv_launch_count": (C.c_longlong, [C.c_void_p]),
    "rbv_last_kernel": (C.c_int, [C.c_void_p]),
    "rbv_voigt_h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "rbv_voigt_h_grad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                   C.c_void_p]),
    "rbv_grad_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_lnprob_grad_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p]),
    "rbv_fisher_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_lnlike_fisher_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_model_jacobian_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_size_t, C.c_void_p]),
    "rbv_fisher_workspace_bytes_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_lnlike_fisher_batch_sightlines": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rbv_lm_workspace_bytes_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]),
    "rbv_lm_run_sightlines": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(RbvLMControl),
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p]),
    "rbv_measure_fp64_peak": (C.c_int, [C.c_void_p, C.c_double, C.POINTER(C.c_double)]),
    "rbv_selftest_rcp": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "rbv_last_error": (C.c_char_p, []),
    "rbv_version": (C.c_char_p, []),
}


def load():
    """Load the in-tree CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("RBVFIT_B200_LIB", LIB_PATH)    # override = tuning experiments only
    if not os.path.exists(path):
        raise RbvError(
            f"{path} is missing: build it with `python -m rbvfit_b200.build` "
            "(or __graft_entry__.build()).  rbvfit_b200 has no CPU fallback.")
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in EXPORTS.items():
        if path != LIB_PATH and not hasattr(lib, name):
            continue                # an experiment's build of an older source tree: newer entry points are absent
        fn = getattr(lib, name)     # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str = ""):
    if status != 0:
        msg = load().rbv_last_error().decode("utf-8", "replace")
        raise RbvError(f"{what or 'rbvfit_b200'} failed (status {status}): {msg}")
