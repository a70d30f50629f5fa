"""Survey-mode Fisher matrix and device Levenberg-Marquardt loop over sightlines (DESIGN.md section 16), timed on one GPU.

  * Fisher launch: rbv_lnlike_fisher_batch_sightlines over S C5b sightlines (one row each) against S back-to-back
    one-row rbv_lnlike_fisher_batch launches on a one-sightline context (CUDA events, median of repeats)
  * whole fit: SightlineBatch.fit_quick on S = 1024 C5b sightlines against per-sightline
    vfit.fit_quick(method="lm") timed on 32 sightlines and scaled by S / 32 (wall clock; both end in a synchronise)
  * behaviour: iterations, device launches, status histogram
  * --parent-lib: bench.py with that library and with this one, alternated; and rbv_lnlike_fisher_batch outputs of both
    libraries on every golden case (bitwise)

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
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # pragma: no cover
        return f"unavailable ({e})"


def _c5b(S, first=0):
    from rbvfit_b200 import FitConfiguration, workloads as wl
    from rbvfit_b200.model import GpuVoigtModel
    sight, thetas = [], []
    for s in range(first, first + S):
        w = wl.c5b_sightline(s)
        cfg = FitConfiguration()
        for (z, ion, trans, comps) in w["systems"]:
            cfg.add_system(z=z, ion=ion, transitions=trans, components=comps)
        m = GpuVoigtModel(cfg, FWHM="6.5")
        c = m.compile(verbose=False)
        sp = wl.make_spectra(w, lambda n, th, wave: c.model_flux(th, wave))["COS"]
        sight.append(dict(model=m, **sp))
        rng = np.random.default_rng(s)
        C = w["theta_true"].size // 3
        off = np.concatenate([np.full(C, 0.1), np.full(C, 3.0), np.full(C, 4.0)]) * rng.standard_normal(3 * C)
        thetas.append(np.clip(w["theta_true"] + off, w["lb"], w["ub"]))
    return sight, np.array(thetas), wl.c5b_sightline(0)


def _events(fn, reps=20):
    import torch
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def fisher_launch(Ss):
    import torch
    from rbvfit_b200.likelihood import GpuLikelihood, SightlineBatch
    sight, thetas, w0 = _c5b(max(Ss))
    out = {}
    single = GpuLikelihood({"COS": sight[0]}, w0["lb"], w0["ub"])
    eng1 = single.engine
    th1 = torch.as_tensor(thetas[:1], device=eng1.tdev)
    eng1.lnlike_fisher_device(th1)
    for S in Ss:
        batch = SightlineBatch(sight[:S], w0["lb"], w0["ub"])
        eng = batch.engine
        th = torch.as_tensor(thetas[:S], device=eng.tdev)
        t_batch = _events(lambda: eng.lnlike_fisher_sightlines_device(th, 1))

        def singles():
            for _ in range(S):
                eng1.lnlike_fisher_device(th1)
        t_single = _events(singles, reps=5)
        out[S] = dict(sightline_launch_ms=t_batch, S_single_launches_ms=t_single, speedup=t_single / t_batch)
        batch.close()
    single.close()
    return out


def whole_fit(S, n_host):
    import warnings
    import torch
    from rbvfit_b200.likelihood import SightlineBatch
    from rbvfit_b200.vfit_mcmc import vfit
    sight, thetas, w0 = _c5b(S)
    batch = SightlineBatch(sight, w0["lb"], w0["ub"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        batch.fit_quick(thetas)     # warm-up (module load, workspace)
        torch.cuda.synchronize()
        n0 = batch.engine.launch_count
        t0 = time.perf_counter()
        res = batch.fit_quick(thetas)
        t_dev = time.perf_counter() - t0
    launches = batch.engine.launch_count - n0
    hist = {int(k): int(v) for k, v in zip(*np.unique(res.status, return_counts=True))}
    batch.close()
    t_host = 0.0
    for s in range(n_host):
        f = vfit({"COS": sight[s]}, thetas[s], w0["lb"], w0["ub"], no_of_Chain=8, no_of_steps=2)
        if s == 0:
            f.fit_quick(verbose=False, method="lm")
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            f.fit_quick(verbose=False, method="lm")
        t_host += time.perf_counter() - t0
        f._like.close()
    return dict(S=S, device_fit_s=t_dev, iterations=int(res.n_evals.max()), device_launches=launches,
                mean_n_evals=float(res.n_evals.mean()), status_histogram=hist,
                host_fit_s_measured=t_host, host_sightlines_measured=n_host,
                host_fit_s_scaled=t_host * S / n_host, speedup=t_host * S / n_host / t_dev)


def dump_joint(path):
    """rbv_lnlike_fisher_batch on every golden case's fixture rows (no prior: every row)."""
    from golden_util import CASES, Golden
    from test_gpu_gradient import _like
    out = {}
    for case in [c for c in CASES if c != "C1_fast"] + ["C5a"]:
        g = Golden(case)
        like = _like(g)
        rows = g.thetas[:4] if case == "C5a" else g.thetas
        v, gr, F = like.lnlike_and_fisher(rows)
        out[f"{case}__v"], out[f"{case}__g"], out[f"{case}__F"] = v, gr, F
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
    runs = []
    for i in range(args.bench_pairs):
        for name, env in (("parent", old_env), ("this", new_env)) if i % 2 == 0 else (("this", new_env),
                                                                                       ("parent", old_env)):
            runs.append(dict(lib=name, **_bench_line(env, args)))
    tmp = os.environ.get("TMPDIR", "/tmp")
    paths = {}
    for name, env in (("parent", old_env), ("this", new_env)):
        paths[name] = os.path.join(tmp, f"joint_fisher_{name}_{os.getpid()}.npz")
        subprocess.run([sys.executable, os.path.abspath(__file__), "--dump-joint", paths[name]], env=env, check=True,
                       cwd=ROOT)
    a, b = np.load(paths["parent"]), np.load(paths["this"])
    same = {k: bool(np.array_equal(a[k], b[k], equal_nan=True)) for k in a.files}
    return dict(bench_runs=runs, joint_fisher_bit_identical=all(same.values()),
                joint_fisher_arrays_compared=len(same), joint_fisher_mismatches=[k for k, v in same.items() if not v])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sightlines", type=int, nargs="+", default=[64, 256, 1024])
    ap.add_argument("--fit-sightlines", type=int, default=1024)
    ap.add_argument("--host-sightlines", type=int, default=32)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--bench-pairs", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-joint", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.dump_joint:
        dump_joint(args.dump_joint)
        return
    res = dict(gpu=_gpu_info(), fisher_launch=fisher_launch(args.sightlines),
               whole_fit=whole_fit(args.fit_sightlines, args.host_sightlines))
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
