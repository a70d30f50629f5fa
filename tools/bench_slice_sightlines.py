"""Survey-mode ensemble slice sampling (DESIGN.md section 17), timed on one GPU.

  * survey zeus: SightlineEnsembleSliceSampler over S C5b sightlines x W walkers, steps/s of a continued run after a
    warm-up run that ends mu tuning (wall clock around run_mcmc, which ends in a synchronise and includes the copy of
    the chain to the host); launches per half-step
  * sequential baseline: the same sightlines as back-to-back DeviceEnsembleSliceSampler runs on one-sightline
    contexts, measured at the smallest S and scaled linearly above it (labelled as scaled).  Its launches per
    half-step, averaged over sightlines, is what one sightline needs alone; the survey's launches per half-step over
    that mean is the lockstep tail cost (same depth on both sides)
  * context: SightlineEnsembleSampler (stretch move) steps/s at the same S and W
  * effective samples: at the smallest S and --ess-steps steps, the median integrated autocorrelation time of both
    survey samplers and effective samples per second
  * --parent-lib: DeviceEnsembleSliceSampler chains, mu history and counters on C1 and C2 (graph / polled, depth 1 / 2)
    with that library and with this one (bitwise), and bench.py with the two libraries alternated

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


def _c5b(S):
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    sight = []
    for s in range(S):
        w = wl.c5b_sightline(s)
        cfg = FitConfiguration()
        for (z, ion, trans, comps) in w["systems"]:
            cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        m = GpuVoigtModel(cfg, FWHM="6.5")
        c = m.compile(verbose=False)
        sp = wl.make_spectra(w, lambda n, th, wave: c.model_flux(th, wave))["COS"]
        sight.append(dict(model=m, **sp))
    return sight, wl.c5b_sightline(0)


def _start(w0, S, W, seed=1):
    rng = np.random.default_rng(seed)
    return np.clip(w0["theta_true"] + 1e-3 * rng.standard_normal((S, W, len(w0["theta_true"]))), w0["lb"], w0["ub"])


def _timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def _median_tau(chains, discard):
    """chains [steps, S, W, ndim] -> median over sightlines of the median over parameters of tau"""
    from rbvfit_b200.sampler import integrated_time
    taus = [np.median(integrated_time(chains[discard:, e], quiet=True)) for e in range(chains.shape[1])]
    return float(np.median(taus)), np.array(taus)


def survey(Ss, W, warm, steps, seq_steps, ess_steps, ess_discard):
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    from rbvfit_b200.sampler import SightlineEnsembleSampler
    from rbvfit_b200.slice_sampler import DeviceEnsembleSliceSampler, SightlineEnsembleSliceSampler
    sight, w0 = _c5b(max(Ss))
    nd = len(w0["theta_true"])
    out = dict(W=W, warmup_steps=warm, timed_steps=steps, per_S={})
    # sequential baseline at the smallest S
    S0 = min(Ss)
    p0 = _start(w0, S0, W)
    singles = [GpuLikelihood({"COS": sight[e]}, w0["lb"], w0["ub"]) for e in range(S0)]
    samplers = [DeviceEnsembleSliceSampler(W, nd, singles[e], seed=1) for e in range(S0)]
    for e, smp in enumerate(samplers):
        smp.run_mcmc(p0[e], warm)
    before = [smp.nbatches for smp in samplers]
    t = _timed(lambda: [smp.run_mcmc(None, seq_steps) for smp in samplers])
    alone = np.array([(smp.nbatches - b) / (2 * seq_steps) for smp, b in zip(samplers, before)])
    seq_sps = seq_steps / t
    out["sequential"] = dict(S=S0, steps=seq_steps, steps_per_s=seq_sps, seconds=t,
                             launches_per_half_step_alone_mean=float(alone.mean()),
                             launches_per_half_step_alone_max=float(alone.max()))
    for like in singles:
        like.close()
    del samplers
    for S in Ss:
        batch = SightlineBatch(sight[:S], w0["lb"], w0["ub"])
        p0 = _start(w0, S, W)
        zeus = SightlineEnsembleSliceSampler(W, nd, batch, seed=1)
        tw = _timed(lambda: zeus.run_mcmc(p0, warm))
        still_tuning = int(zeus.tune.sum())
        b0 = zeus.nbatches
        t = _timed(lambda: zeus.run_mcmc(None, steps))
        lph = (zeus.nbatches - b0) / (2 * steps)
        row = dict(zeus_steps_per_s=steps / t, zeus_seconds=t, zeus_warmup_seconds=tw,
                   sightlines_still_tuning_after_warmup=still_tuning, launches_per_half_step=lph,
                   lockstep_tail_ratio=lph / out["sequential"]["launches_per_half_step_alone_mean"],
                   sequential_steps_per_s=seq_sps * S0 / S, sequential_scaled=S != S0)
        row["speedup_vs_sequential"] = row["zeus_steps_per_s"] / row["sequential_steps_per_s"]
        stretch = SightlineEnsembleSampler(W, nd, batch, seed=1)
        stretch.run_mcmc(p0, 5)
        t = _timed(lambda: stretch.run_mcmc(None, steps))
        row["stretch_steps_per_s"] = steps / t
        if S == S0 and ess_steps > 0:
            t = _timed(lambda: zeus.run_mcmc(None, ess_steps))
            tau, taus = _median_tau(zeus.get_chain()[-ess_steps:], ess_discard)
            n = (ess_steps - ess_discard) * W
            row["zeus_ess"] = dict(steps=ess_steps, discard=ess_discard, median_tau=tau, seconds=t,
                                   ess_per_s=float(np.sum(n / taus) / t))
            t = _timed(lambda: stretch.run_mcmc(None, ess_steps))
            tau, taus = _median_tau(stretch.get_chain()[-ess_steps:], ess_discard)
            row["stretch_ess"] = dict(steps=ess_steps, discard=ess_discard, median_tau=tau, seconds=t,
                                      ess_per_s=float(np.sum(n / taus) / t))
        out["per_S"][S] = row
        del zeus, stretch
        batch.close()
    return out


def dump_single(path, c2_steps):
    """DeviceEnsembleSliceSampler on C1 and C2, graph / polled x depth 1 / 2 -> npz (run once per library)."""
    sys.path.insert(0, ROOT)
    from bench import build_problem
    from rbvfit_b200.slice_sampler import DeviceEnsembleSliceSampler
    out = {}
    for name, nsteps in (("C1", 40), ("C2", c2_steps)):
        w, models, like, thetas, spectra = build_problem(name, 0)
        nd = like.ndim
        W = max(16, 2 * nd + (2 * nd) % 2)
        p0 = np.clip(w["theta_true"] + 1e-3 * np.random.default_rng(2).standard_normal((W, nd)), w["lb"], w["ub"])
        for graph in (True, False):
            for depth in (1, 2):
                s = DeviceEnsembleSliceSampler(W, nd, like, seed=11, use_graph=graph, depth=depth)
                s.run_mcmc(p0, nsteps)
                k = f"{name}_{'graph' if graph else 'poll'}_d{depth}"
                out[k + "__chain"], out[k + "__lnp"] = s.get_chain(), s.get_log_prob()
                out[k + "__mus"] = np.asarray(s.mus)
                out[k + "__counters"] = np.array([s.ncall, s.nexp, s.ncon, s.nbatches, int(s.tune), s.good])
                out[k + "__mu"] = np.array([s.mu])
        like.close()
    np.savez(path, **out)


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
    tmp = os.environ.get("TMPDIR", "/tmp")
    paths = {}
    for name, env in (("parent", old_env), ("this", new_env)):
        paths[name] = os.path.join(tmp, f"slice_single_{name}_{os.getpid()}.npz")
        subprocess.run([sys.executable, os.path.abspath(__file__), "--dump-single", paths[name],
                        "--c2-steps", str(args.c2_steps)], env=env, check=True, cwd=ROOT)
    a, b = np.load(paths["parent"]), np.load(paths["this"])
    same = {k: bool(np.array_equal(a[k], b[k], equal_nan=True)) for k in a.files}
    runs = []
    for i in range(args.bench_pairs):
        for name, env in (("parent", old_env), ("this", new_env)) if i % 2 == 0 else (("this", new_env),
                                                                                       ("parent", old_env)):
            runs.append(dict(lib=name, **_bench_line(env, args)))
    return dict(single_slice_bit_identical=all(same.values()), single_slice_arrays_compared=len(same),
                single_slice_mismatches=[k for k, v in same.items() if not v], bench_runs=runs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sightlines", type=int, nargs="+", default=[64, 256, 1024])
    ap.add_argument("--walkers", type=int, default=64)
    ap.add_argument("--warmup-steps", type=int, default=30)
    ap.add_argument("--timed-steps", type=int, default=20)
    ap.add_argument("--seq-steps", type=int, default=20)
    ap.add_argument("--ess-steps", type=int, default=2000)
    ap.add_argument("--ess-discard", type=int, default=500)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--bench-pairs", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20, help="bench.py --steps")
    ap.add_argument("--warmup", type=int, default=3, help="bench.py --warmup")
    ap.add_argument("--c2-steps", type=int, default=15)
    ap.add_argument("--dump-single", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.dump_single:
        dump_single(args.dump_single, args.c2_steps)
        return
    res = dict(gpu=_gpu_info(), survey=survey(args.sightlines, args.walkers, args.warmup_steps, args.timed_steps,
                                               args.seq_steps, args.ess_steps, args.ess_discard))
    if args.parent_lib:
        res["regression"] = regression(args)
    res["gpu_after"] = _gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
