"""Gradient launch vs lnprob launch, and optimize_guess with finite differences vs the device gradient.

    python tools/bench_grad.py [--reps 20] [--out DIR]

Times rbv_lnprob_grad_batch and rbv_lnprob_batch with CUDA events (warm-up, then --reps launches per timed window,
best of 5 windows) at C1 (W = 1, 50), C2 (W = 1, 80), C3 (W = 1) and the C5a geometry (W = 256), and runs
vfit.optimize_guess from the first in-bounds fixture row with gradient="fd" and gradient="device" at C1, C2 and C3
(wall time, objective calls, device rows).  Prints one JSON document (and writes it to DIR/bench_grad.json with
--out), with the card's name and power limit read in the same process.
"""
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


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:       # pragma: no cover
        return f"unknown ({e})"


def build_like(case):
    from golden_util import Golden
    from test_gpu_parity import _gpu_models
    from rbvfit_b200.likelihood import GpuLikelihood
    g = Golden(case)
    models = _gpu_models(g)
    inst = {n: dict(model=models[n], wave=g.inst(n, "wave"), flux=g.inst(n, "flux"), error=g.inst(n, "error"))
            for n in g.instruments}
    ok = [i for i in range(len(g.thetas)) if np.all(g.thetas[i] >= g.lb) and np.all(g.thetas[i] <= g.ub)]
    return g, inst, GpuLikelihood(inst, g.lb, g.ub), g.thetas[ok]


def time_launch(fn, reps, windows=5):
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    return best * 1e3        # us per launch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from rbvfit_b200.vfit_mcmc import vfit
    res = {"card": card(), "reps": args.reps, "launch": [], "optimize_guess": []}
    for case, walkers in (("C1", (1, 50)), ("C2", (1, 80)), ("C3", (1,)), ("C5a", (256,))):
        g, inst, like, rows = build_like(case)
        px = like.total_pixels
        for W in walkers:
            th = torch.tensor(rows[np.arange(W) % len(rows)], dtype=torch.float64, device=like.engine.tdev)
            out = torch.empty(W, dtype=torch.float64, device=like.engine.tdev)
            val = torch.empty(W, dtype=torch.float64, device=like.engine.tdev)
            grad = torch.empty((W, like.ndim), dtype=torch.float64, device=like.engine.tdev)
            t_lnp = time_launch(lambda: like.engine.lnprob_device(th, out), args.reps)
            t_grad = time_launch(lambda: like.engine.lnprob_grad_device(th, True, val, grad), args.reps)
            rel = float(torch.max(torch.abs(val - out) / torch.abs(out)))
            row = dict(case=case, W=W, pixels=px, lnprob_us=t_lnp, grad_us=t_grad, ratio=t_grad / t_lnp,
                       lnprob_walker_px_per_s=W * px / (t_lnp * 1e-6), grad_walker_px_per_s=W * px / (t_grad * 1e-6),
                       value_vs_lnprob_max_rel=rel)
            print(json.dumps(row), flush=True)
            res["launch"].append(row)
        if case in ("C1", "C2", "C3"):
            fitter = vfit(inst, rows[0], g.lb, g.ub, no_of_Chain=8, no_of_steps=2)
            for mode in ("fd", "device"):
                calls, nrows = [0], [0]
                f_lnp, f_grad = fitter._like.lnprob, fitter._like.lnprob_and_grad

                def spy_lnp(theta, f=f_lnp):
                    calls[0] += 1
                    nrows[0] += np.atleast_2d(theta).shape[0]
                    return f(theta)

                def spy_grad(theta, f=f_grad):
                    calls[0] += 1
                    nrows[0] += np.atleast_2d(theta).shape[0]
                    return f(theta)

                fitter._like.lnprob, fitter._like.lnprob_and_grad = spy_lnp, spy_grad
                fitter.optimize_guess(rows[0], gradient=mode)          # warm-up (workspaces, module load)
                calls[0] = nrows[0] = 0
                t0 = time.perf_counter()
                best = fitter.optimize_guess(rows[0], gradient=mode)
                wall = time.perf_counter() - t0
                fitter._like.lnprob, fitter._like.lnprob_and_grad = f_lnp, f_grad
                row = dict(case=case, gradient=mode, wall_s=wall, objective_calls=calls[0], device_rows=nrows[0],
                           final_lnprob=float(fitter.lnprob(best)))
                print(json.dumps(row), flush=True)
                res["optimize_guess"].append(row)
        like.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_grad.json"), "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
