"""Parallel tempering on the device (DESIGN.md section 18), timed on one GPU.

  * steps/s of DeviceParallelTemperingSampler for T in {1, 4, 8, default ladder} on C1 (W = 50), C2 (W = 80) and
    C3 (W = 50), against DeviceEnsembleSampler on the same problem: wall clock around run_mcmc after a warm-up run
    (both end in a synchronise and include the chain's hand-off to the host); launches per step from the library's
    counter
  * the swap stage's device time per step (copy + plan kernel + gather/record kernel) from torch.profiler over a
    run without the graph, and the whole step's kernel time for comparison
  * the wall time of the C1 one- versus two-component comparison (LM fit + PT run + evidence, both models)
  * --parent-lib: bench.py with that library and with this one, alternated

Writes one JSON document to stdout (and to --out).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # pragma: no cover
        return f"unavailable ({e})"


def _problem(name):
    from rbvfit_b200 import FitConfiguration, lsf, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    w = wl.get_workload(name)

    def models(c):
        cfg = FitConfiguration()
        for (z, ion, trans, k) in w["systems"]:
            cfg.add_system(z=z, ion=ion, transitions=trans, components=k if c is None else c)
        return {n: GpuVoigtModel(cfg, FWHM=i["FWHM"],
                                 lsf_taps=lsf.cos_like_taps(321) if i.get("lsf") == "cos_like" else None)
                for n, i in w["instruments"].items()}

    compiled = {n: m.compile() for n, m in models(None).items()}
    spectra = wl.make_spectra(w, lambda n, th, wave: compiled[n].model_flux(th, wave))
    return w, spectra, models


def _like(w, spectra, models):
    from rbvfit_b200.likelihood import GpuLikelihood
    return GpuLikelihood({n: dict(model=m, **spectra[n]) for n, m in models(None).items()}, w["lb"], w["ub"])


def _p0(w, T, W, seed=1):
    rng = np.random.default_rng(seed)
    sc = np.concatenate([np.full(len(w["lb"]) // 3, 0.02), np.full(len(w["lb"]) // 3, 0.5),
                         np.full(len(w["lb"]) // 3, 0.5)])
    return np.clip(w["theta_true"] + sc * rng.standard_normal((T, W, len(w["lb"]))), w["lb"], w["ub"])


def speed(names, walkers, warm, timed):
    import torch
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler, default_betas
    from rbvfit_b200.sampler import DeviceEnsembleSampler
    out = {}
    for name, W in zip(names, walkers):
        w, spectra, models = _problem(name)
        like = _like(w, spectra, models)
        nd = len(w["lb"])
        eng = like.engine
        rows = {}
        st = DeviceEnsembleSampler(W, nd, like, seed=1)
        p0 = _p0(w, 1, W)[0]
        st.run_mcmc(p0, warm)
        torch.cuda.synchronize()
        l0, t0 = eng.launch_count, time.perf_counter()
        st.run_mcmc(None, timed)
        dt = time.perf_counter() - t0
        rows["stretch"] = dict(steps_per_s=timed / dt, launches_per_step=(eng.launch_count - l0) / timed)
        ladders = {"T1": [1.0], "T4": [1.0, 0.3, 0.1, 0.0], "T8": list(np.append(2.0 ** -np.arange(7.0), 0.0)),
                   "default": list(default_betas(nd))}
        for key, betas in ladders.items():
            T = len(betas)
            smp = DeviceParallelTemperingSampler(W, nd, like, betas=betas, seed=1)
            smp.run_mcmc(_p0(w, T, W), warm)
            torch.cuda.synchronize()
            l0, t0 = eng.launch_count, time.perf_counter()
            smp.run_mcmc(None, timed)
            dt = time.perf_counter() - t0
            rows[key] = dict(T=T, steps_per_s=timed / dt, launches_per_step=(eng.launch_count - l0) / timed,
                             cost_vs_stretch=rows["stretch"]["steps_per_s"] * dt / timed,
                             swap_acceptance=[round(float(x), 3) for x in smp.tswap_acceptance_fraction])
        rows["swap_stage"] = swap_stage(like, w, W, list(default_betas(nd)))
        out[name] = dict(W=W, ndim=nd, **rows)
        like.close()
    return out


def swap_stage(like, w, W, betas, n=20):
    """Device time per step of the swap stage and of the whole step (torch.profiler, run without the graph)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler
    smp = DeviceParallelTemperingSampler(W, len(w["lb"]), like, betas=betas, seed=2, use_graph=False)
    smp.run_mcmc(_p0(w, len(betas), W), 3)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        smp.run_mcmc(None, n)
        torch.cuda.synchronize()
    swap = total = 0.0
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        total += us
        if "pt_swap_plan" in e.name or "pt_gather_record" in e.name or "Memcpy DtoD" in e.name:
            swap += us
    return dict(T=len(betas), swap_stage_us_per_step=swap / n, step_kernels_us_per_step=total / n)


def comparison(nsteps):
    """C1 one- versus two-component evidence, wall clock of the whole comparison."""
    import torch
    from rbvfit_b200 import workloads as wl
    from rbvfit_b200.pt_sampler import default_betas
    from rbvfit_b200.vfit_mcmc import vfit
    w, spectra, models = _problem("C1")
    lb1, ub1 = wl.default_bounds([14.6], [40.0], [0.0])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = {}
    for comps, theta0, lb, ub in ((1, np.array([14.6, 40.0, 0.0]), lb1, ub1),
                                  (2, np.clip(w["theta_true"] + [0.05, -0.05, 2, -2, 3, -3.0], w["lb"], w["ub"]),
                                   w["lb"], w["ub"])):
        f = vfit({n: dict(model=m, **spectra[n]) for n, m in models(comps).items()}, theta0, lb, ub,
                 no_of_Chain=50, no_of_steps=nsteps, seed=3, sampler="pt", betas=default_betas(3 * comps))
        f.fit_quick(verbose=False, method="lm")
        f.theta = f.theta_best
        f.runmcmc(optimize=False, verbose=False, progress=False)
        res[f"lnZ_{comps}"] = f.log_evidence()
    res["seconds"] = time.perf_counter() - t0
    res["steps"] = nsteps
    return res


def _bench_line(env, args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.steps),
                        "--warmup", str(args.warmup), "--no-cpu"], capture_output=True, text=True, env=env, cwd=ROOT)
    for line in reversed(r.stdout.splitlines()):
        if line.startswith("{"):
            d = json.loads(line)
            return dict(value=d["value"], ms_per_step=d["ms_per_step"])
    return dict(error=r.stderr[-2000:])


def regression(args):
    new_env = dict(os.environ)
    new_env.pop("RBVFIT_B200_LIB", None)
    old_env = dict(new_env, RBVFIT_B200_LIB=os.path.abspath(args.parent_lib))
    runs = []
    for i in range(args.bench_pairs):
        order = (("parent", old_env), ("this", new_env)) if i % 2 == 0 else (("this", new_env), ("parent", old_env))
        for name, env in order:
            runs.append(dict(lib=name, **_bench_line(env, args)))
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["C1", "C2", "C3"])
    ap.add_argument("--walkers", type=int, nargs="+", default=[50, 80, 50])
    ap.add_argument("--warm", type=int, default=20)
    ap.add_argument("--timed", type=int, default=200)
    ap.add_argument("--compare-steps", type=int, default=2000)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--bench-pairs", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20, help="bench.py --steps")
    ap.add_argument("--warmup", type=int, default=3, help="bench.py --warmup")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = dict(gpu=_gpu_info(), speed=speed(args.workloads, args.walkers, args.warm, args.timed))
    if args.compare_steps:
        res["one_vs_two_components"] = comparison(args.compare_steps)
    if args.parent_lib:
        res["bench_alternated"] = regression(args)
    res["gpu_after"] = _gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
