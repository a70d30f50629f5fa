"""CPU: the scalar restatement of the survey-mode LM update (oracle/lm_replay.py) against the host driver
rbvfit_b200.lm.levenberg_marquardt, both driven by the Fisher oracle."""
import numpy as np
import pytest

from oracle import lm_replay
from oracle import voigt_fisher_oracle as vf
from oracle import voigt_oracle as vo
from rbvfit_b200 import lm
from rbvfit_b200 import workloads as wl


def _problem(w, theta_data=None):
    """(fisher_fn, lb, ub) of workload w's first instrument, data made at theta_data (default theta_true)."""
    ocfg = vo.OracleConfig()
    for (z, ion, trans, comps) in w["systems"]:
        ocfg.add_system(z, ion, trans, comps)
    (name, spec), = w["instruments"].items()
    om = vo.lower(ocfg, FWHM=spec["FWHM"])
    t = w["theta_true"] if theta_data is None else theta_data
    rng = np.random.default_rng(w["seed"])
    flux = vo.model_flux(om, t, spec["wave"]) + wl.SIGMA * rng.standard_normal(spec["wave"].size)
    comp = vo.compile_instruments({name: dict(model=om, wave=spec["wave"], flux=flux,
                                              error=np.full(spec["wave"].size, wl.SIGMA))})
    return (lambda x: vf.lnlike_fisher(comp, x)), w["lb"].astype(float), w["ub"].astype(float)


def _offset(w):
    C = w["theta_true"].size // 3
    return w["theta_true"] + np.concatenate([np.full(C, 0.15), np.full(C, -3.0), np.full(C, 4.0)])


def _compare(rep, ref):
    assert (rep.status > 0) == (ref.status > 0), (rep.status, ref.status)
    assert abs(rep.chi2 - ref.chi2) <= 1e-10 * abs(ref.chi2)
    sig = np.sqrt(np.diag(ref.cov))
    ok = np.isfinite(sig)
    assert np.array_equal(ok, np.isfinite(np.diag(rep.cov)))
    assert np.all(np.abs(rep.x - ref.x)[ok] <= 1e-4 * sig[ok])
    assert np.array_equal(rep.x[~ok], ref.x[~ok])
    d = np.sqrt(np.outer(sig, sig))
    both = np.isfinite(d)
    assert np.max(np.abs(rep.cov - ref.cov)[both] / d[both]) <= 1e-6   # the two x differ in the last digits


@pytest.mark.parametrize("case", ["C1", "C4", "C5b0", "C5b1", "C5b2", "C5b3"])
def test_replay_vs_host_driver(case):
    w = wl.c5b_sightline(int(case[3:])) if case.startswith("C5b") else wl.get_workload(case)
    fn, lb, ub = _problem(w)
    x0 = _offset(w)
    rep = lm_replay.run(fn, x0, lb, ub)
    ref = lm.levenberg_marquardt(fn, x0, lb, ub)
    print(case, "replay", rep.chi2, rep.n_evals, rep.status, "| lm", ref.chi2, ref.n_evals, ref.status)
    assert rep.flags == 0 and rep.status > 0
    _compare(rep, ref)


def test_replay_parameter_pinned_on_bound():
    """Data made with log N of component 0 above its upper bound, start on that bound: the gradient points out of the
    box, the parameter leaves the free set, stays on the bound, and its covariance row and column are NaN."""
    w = wl.get_workload("C1")
    t = w["theta_true"].copy()
    t[0] = w["ub"][0] + 0.5
    fn, lb, ub = _problem(w, t)
    x0 = _offset(w)
    x0[0] = ub[0]
    _ll, g, F = fn(x0)
    assert g[0] > 0 and 0 not in lm_replay.free_set(list(x0), list(g), F.tolist(), lb, ub)
    assert not lm.free_set(x0, g, F, lb, ub)[0]
    rep = lm_replay.run(fn, x0, lb, ub)
    ref = lm.levenberg_marquardt(fn, x0, lb, ub)
    assert rep.x[0] == ub[0] and ref.x[0] == ub[0]
    assert np.all(np.isnan(rep.cov[0])) and np.all(np.isnan(rep.cov[:, 0]))
    assert np.isfinite(rep.cov[1, 1])
    _compare(rep, ref)


def test_replay_stops_on_max_evals():
    w = wl.get_workload("C1")
    fn, lb, ub = _problem(w)
    x0 = _offset(w)
    rep = lm_replay.run(fn, x0, lb, ub, max_evals=3)
    ref = lm.levenberg_marquardt(fn, x0, lb, ub, max_evals=3)
    assert rep.status == ref.status == lm.STATUS_MAX_EVALS
    assert rep.n_evals == ref.n_evals == 3
    _compare(rep, ref)
