"""Fisher launch vs gradient launch, and fit_quick with L-BFGS-B (finite differences / device gradient) vs
Levenberg-Marquardt on the device's Gauss-Newton matrix.

    python tools/bench_fisher.py [--reps 20] [--out DIR]

Times rbv_lnlike_fisher_batch and rbv_lnprob_grad_batch (without the prior) with CUDA events (warm-up, then --reps
launches per timed window, best of 5 windows) at C1 (W = 1, 50), C2 (W = 1), C3 (W = 1) and the C5a geometry
(W = 1, 8), and runs vfit.fit_quick from the first in-bounds fixture row at C1, C2, C3 and C4 with
method="lbfgsb" (gradient="fd" and "device") and method="lm" (wall time after one warm-up fit, objective calls,
device launches, final chi^2).  Prints one JSON document (and writes it to DIR/bench_fisher.json with --out), with
the card's name and power limit read in the same process.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_grad import build_like, card, time_launch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from rbvfit_b200.vfit_mcmc import vfit
    res = {"card": card(), "reps": args.reps, "launch": [], "fit_quick": []}
    for case, walkers in (("C1", (1, 50)), ("C2", (1,)), ("C3", (1,)), ("C4", ()), ("C5a", (1, 8))):
        g, inst, like, rows = build_like(case)
        eng, px, n = like.engine, like.total_pixels, like.ndim
        for W in walkers:
            th = torch.tensor(rows[np.arange(W) % len(rows)], dtype=torch.float64, device=eng.tdev)
            val = torch.empty(W, dtype=torch.float64, device=eng.tdev)
            grad = torch.empty((W, n), dtype=torch.float64, device=eng.tdev)
            fval = torch.empty(W, dtype=torch.float64, device=eng.tdev)
            fgrad = torch.empty((W, n), dtype=torch.float64, device=eng.tdev)
            fisher = torch.empty((W, n, n), dtype=torch.float64, device=eng.tdev)
            t_grad = time_launch(lambda: eng.lnprob_grad_device(th, False, val, grad), args.reps)
            c0 = eng.launch_count
            t_fish = time_launch(lambda: eng.lnlike_fisher_device(th, fval, fgrad, fisher), args.reps)
            launches = (eng.launch_count - c0) // (3 + 5 * args.reps)
            row = dict(case=case, W=W, pixels=px, ndim=n, grad_us=t_grad, fisher_us=t_fish, ratio=t_fish / t_grad,
                       fisher_launches_per_call=launches,
                       value_identical=bool(torch.equal(val, fval)),
                       grad_max_abs_diff=float(torch.max(torch.abs(grad - fgrad))))
            print(json.dumps(row), flush=True)
            res["launch"].append(row)
        if case != "C5a":
            fitter = vfit(inst, rows[0], g.lb, g.ub, no_of_Chain=8, no_of_steps=2)
            L = fitter._like
            for method, mode in (("lbfgsb", "fd"), ("lbfgsb", "device"), ("lm", "fd")):
                calls = [0]
                orig = {k: getattr(L, k) for k in ("lnlike", "lnlike_and_grad", "lnlike_and_fisher")}

                def spy(f):
                    def wrapped(theta):
                        calls[0] += 1
                        return f(theta)
                    return wrapped

                for k, f in orig.items():
                    setattr(L, k, spy(f))
                fitter.fit_quick(verbose=False, gradient=mode, method=method)      # warm-up
                calls[0] = 0
                c0 = eng_launches = L.engine.launch_count
                t0 = time.perf_counter()
                best, _err = fitter.fit_quick(verbose=False, gradient=mode, method=method)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                eng_launches = L.engine.launch_count - c0
                for k, f in orig.items():
                    setattr(L, k, f)
                row = dict(case=case, method=method, gradient=mode if method == "lbfgsb" else None, wall_s=wall,
                           objective_calls=calls[0], device_launches=eng_launches,
                           chi2=float(fitter._chi2_batch(best)[0]))
                print(json.dumps(row), flush=True)
                res["fit_quick"].append(row)
            L.close()
        like.close()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_fisher.json"), "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
