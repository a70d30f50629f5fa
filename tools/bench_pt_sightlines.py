"""Survey-mode parallel tempering (DESIGN.md section 19), timed on one GPU.

  * survey PT: SightlineParallelTemperingSampler over S C5b sightlines x W walkers for T in {4, 8, default ladder}:
    steps/s of a continued run (accumulating the evidence moments, cold chain streamed to the host) after a warm-up
    run; wall clock around run_mcmc, which ends in a synchronise.  Launches per step from the library's counter
  * sequential baseline: the same work as back-to-back DeviceParallelTemperingSampler runs on one-sightline contexts,
    measured at the smallest S and scaled linearly above it (labelled as scaled)
  * --profile: the swap stage's device time per step (copy + plan kernel + gather/record kernel) at S = 1 and at the
    largest S, from torch.profiler over a run without the graph (run this separately from the timings)
  * --compare-steps: only the wall time of the 1- versus 2-component comparison over the largest S (two
    SightlineBatches, fit_quick each, PT seeded around each fit, burn-in without accumulation, then lnZ(2) - lnZ(1)
    per sightline)
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


def _c5b(S, components=(2,)):
    """C5b's first S sightlines: {components: sightline dicts with that many MgII components per model}, spectra
    drawn from the two-component truth."""
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    out = {c: [] for c in components}
    for s in range(S):
        w = wl.c5b_sightline(s)
        z = w["systems"][0][0]
        models = {}
        for c in set(components) | {2}:
            cfg = FitConfiguration()
            cfg.add_system(z=z, ion="MgII", transitions=[2796.3, 2803.5], components=c)
            models[c] = GpuVoigtModel(cfg, FWHM="6.5")
        c2 = models[2].compile(verbose=False)
        sp = wl.make_spectra(w, lambda n, th, wave: c2.model_flux(th, wave))["COS"]
        for c in components:
            out[c].append(dict(model=models[c], **sp))
    return out, wl.c5b_sightline(0)


def _start(w0, shape, seed=1):
    rng = np.random.default_rng(seed)
    nd = len(w0["theta_true"])
    return np.clip(w0["theta_true"] + 1e-3 * rng.standard_normal(tuple(shape) + (nd,)), w0["lb"], w0["ub"])


def _timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def _ladders(nd):
    from rbvfit_b200.pt_sampler import default_betas
    return {"T4": [1.0, 0.3, 0.1, 0.0], "T8": list(np.append(2.0 ** -np.arange(7.0), 0.0)),
            "default": list(default_betas(nd))}


def survey(sight, w0, Ss, W, warm, timed, seq_steps):
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.pt_sampler import DeviceParallelTemperingSampler, SightlineParallelTemperingSampler
    nd = len(w0["theta_true"])
    ladders = _ladders(nd)
    out = dict(W=W, warmup_steps=warm, timed_steps=timed, sequential={}, per_S={})
    S0 = min(Ss)
    singles = [GpuLikelihood({"COS": sight[e]}, w0["lb"], w0["ub"]) for e in range(S0)]
    for key, betas in ladders.items():
        T = len(betas)
        p0 = _start(w0, (S0, T, W))
        samplers = [DeviceParallelTemperingSampler(W, nd, singles[e], betas=betas, seed=1) for e in range(S0)]
        for e, smp in enumerate(samplers):
            smp.run_mcmc(p0[e], warm)
        t = _timed(lambda: [smp.run_mcmc(None, seq_steps) for smp in samplers])
        out["sequential"][key] = dict(S=S0, T=T, steps=seq_steps, steps_per_s=seq_steps / t, seconds=t)
        del samplers
    for like in singles:
        like.close()
    for S in Ss:
        batch = SightlineBatch(sight[:S], w0["lb"], w0["ub"])
        eng = batch.engine
        rows = {}
        for key, betas in ladders.items():
            T = len(betas)
            smp = SightlineParallelTemperingSampler(W, nd, batch, betas=betas, seed=1)
            tw = _timed(lambda: smp.run_mcmc(_start(w0, (S, W)), warm, accumulate=False))
            l0 = eng.launch_count
            t = _timed(lambda: smp.run_mcmc(None, timed))
            seq = out["sequential"][key]["steps_per_s"] * S0 / S
            rows[key] = dict(T=T, rows_per_half_step=S * T * ((W + 1) // 2), steps_per_s=timed / t, seconds=t,
                             warmup_seconds=tw, launches_per_step=(eng.launch_count - l0) / timed,
                             sequential_steps_per_s=seq, sequential_scaled=S != S0,
                             speedup_vs_sequential=(timed / t) / seq,
                             lnZ_finite=int(np.isfinite(smp.log_evidence_estimate()[0]).sum()))
            del smp
        out["per_S"][S] = rows
        batch.close()
    return out


def swap_stage(sight, w0, Ss, W, n=10):
    """Device time per step of the swap stage and of all the step's kernels (torch.profiler, no graph)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from rbvfit_b200.likelihood import SightlineBatch
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler, default_betas
    nd = len(w0["theta_true"])
    betas = default_betas(nd)
    out = {}
    for S in Ss:
        batch = SightlineBatch(sight[:S], w0["lb"], w0["ub"])
        smp = SightlineParallelTemperingSampler(W, nd, batch, betas=betas, seed=2, use_graph=False,
                                                record_chain=False)
        smp.run_mcmc(_start(w0, (S, W)), 3)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            smp.run_mcmc(None, n)
            torch.cuda.synchronize()
        swap = total = 0.0
        parts = {}
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            total += us
            for key in ("pt_swap_plan", "pt_gather_record", "Memcpy DtoD"):
                if key in e.name:
                    swap += us
                    parts[key] = parts.get(key, 0.0) + us / n
        out[S] = dict(T=len(betas), swap_stage_us_per_step=swap / n, step_kernels_us_per_step=total / n,
                      parts_us_per_step=parts)
        batch.close()
    return out


def comparison(sights, w0, W, burn, nsteps):
    """1- versus 2-component evidence of every sightline, wall clock of the whole comparison (the batches exist)."""
    import torch
    from rbvfit_b200 import workloads as wl
    from rbvfit_b200.likelihood import SightlineBatch
    from rbvfit_b200.pt_sampler import SightlineParallelTemperingSampler, default_betas
    lb1, ub1 = wl.default_bounds([14.6], [40.0], [0.0])
    setups = ((1, sights[1], np.array([14.6, 40.0, 0.0]), lb1, ub1),
              (2, sights[2], np.clip(w0["theta_true"] + [0.05, -0.05, 2, -2, 3, -3.0], w0["lb"], w0["ub"]),
               w0["lb"], w0["ub"]))
    batches = {c: SightlineBatch(sl, lb, ub) for c, sl, _t, lb, ub in setups}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lnz, dlnz, parts = {}, {}, {}
    for c, _sl, theta0, lb, ub in setups:
        b = batches[c]
        t1 = time.perf_counter()
        fit = b.fit_quick(theta0)
        t_fit = time.perf_counter() - t1
        rng = np.random.default_rng(c)
        p0 = np.clip(fit.x[:, None, :] + 1e-4 * rng.standard_normal((b.n_sightlines, W, b.ndim)), lb + 1e-10,
                     ub - 1e-10)
        smp = SightlineParallelTemperingSampler(W, b.ndim, b, betas=default_betas(b.ndim), seed=c)
        smp.run_mcmc(p0, burn, accumulate=False)
        smp.run_mcmc(None, nsteps)
        lnz[c], dlnz[c] = smp.log_evidence_estimate()
        parts[c] = dict(fit_seconds=t_fit, pt_seconds=time.perf_counter() - t1 - t_fit, T=smp.ntemps)
    seconds = time.perf_counter() - t0
    d = lnz[2] - lnz[1]
    res = dict(S=len(sights[2]), W=W, burn_steps=burn, steps=nsteps, seconds=seconds, parts=parts,
               dlnZ21_median=float(np.nanmedian(d)), dlnZ21_min=float(np.nanmin(d)),
               sightlines_preferring_two=int(np.sum(d > 0)), dlnZ_median=[float(np.nanmedian(dlnz[1])),
                                                                        float(np.nanmedian(dlnz[2]))])
    for b in batches.values():
        b.close()
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
    ap.add_argument("--sightlines", type=int, nargs="+", default=[64, 256, 1024])
    ap.add_argument("--walkers", type=int, default=32)
    ap.add_argument("--warmup-steps", type=int, default=10)
    ap.add_argument("--timed-steps", type=int, default=30)
    ap.add_argument("--seq-steps", type=int, default=30)
    ap.add_argument("--profile", action="store_true", help="only the swap-stage profile at S = 1 and the largest S")
    ap.add_argument("--compare-burn", type=int, default=100)
    ap.add_argument("--compare-steps", type=int, default=0)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--bench-pairs", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20, help="bench.py --steps")
    ap.add_argument("--warmup", type=int, default=3, help="bench.py --warmup")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = dict(gpu=_gpu_info())
    Smax = max(args.sightlines)
    sights, w0 = _c5b(Smax, components=(1, 2) if args.compare_steps else (2,))
    if args.profile:
        res["swap_stage"] = swap_stage(sights[2], w0, [1, Smax], args.walkers)
    elif args.compare_steps:
        res["one_vs_two_components"] = comparison(sights, w0, args.walkers, args.compare_burn, args.compare_steps)
    else:
        res["survey"] = survey(sights[2], w0, args.sightlines, args.walkers, args.warmup_steps, args.timed_steps,
                               args.seq_steps)
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
