"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the survey-mode ensemble slice sampler
(rbvfit_b200/csrc/rbv_slice.cuh, C ABI rbv_slice_run_sightlines), one sightline's ensemble at a time.

rbv_slice_run_sightlines advances S ensembles of W walkers in lockstep.  Ensemble e is the single-ensemble algorithm
that ``oracle/slice_replay.py`` restates, with two survey-specific facts added here:

  * its random streams are those of a single ensemble with the walker counter offset by e W (``walker_offset``):
    purposes 8 + s, 10 + s and 16 + 2 it + s; the step's split is shared by all ensembles;
  * a half-step of the survey launches as many batches as its slowest ensemble needs, so ``run`` also returns the
    batches of every half-step (``batches_per_half``): device launches of a half-step = the maximum over sightlines
    of that sightline's replay batches.

With ``walker_offset=0`` ``run`` is ``slice_replay.run`` (tests/test_slice_replay_sightlines.py checks that bit for
bit); driven by a sightline's own one-sightline GPU lnprob it reproduces that sightline of the device run
(tests/test_gpu_slice_sightlines.py).
"""
from __future__ import annotations

import numpy as np

from .slice_replay import DONE, LEFT, RIGHT, SHRINK
from .stretch_replay import _rand, split_geometry, step_perm, u01


def run(lnprob_fn, coords, lnp, nsteps, seed, mu=1.0, tune=True, tolerance=0.05, patience=5, maxsteps=10000,
        maxiter=10000, first_step=0, good=0, depth=1, walker_offset=0):
    """Returns a dict: chain [nsteps, W, ndim], lnp_chain [nsteps, W], mus [nsteps], mu, tune, good, nexp, ncon,
    ncall, nbatches, batches_per_half [2 nsteps] (batches of every half-step, summing to nbatches).
    ``lnprob_fn`` maps (n, ndim) -> (n,) and is called once per batch with the candidates of the walkers that are
    still unfinished.  ``walker_offset`` shifts the walker counter of every random stream (e W for ensemble e of a
    survey run).  ``depth`` = logical iterations served per batch (1: the sequential
    algorithm; 2: the second iteration's candidates are evaluated speculatively in the same batch -- chain, mu,
    nexp, ncon and ncall are those of depth 1, nbatches is what the device launches)."""
    X = np.array(coords, dtype=np.float64, copy=True)
    Z = np.array(lnp, dtype=np.float64, copy=True)
    W, ndim = X.shape
    chain = np.empty((nsteps, W, ndim))
    lps = np.empty((nsteps, W))
    mus = np.empty(nsteps)
    tot_exp = tot_con = ncall = nbatches = 0
    per_half = []
    for s in range(nsteps):
        step = first_step + s
        pa, pb = step_perm(seed, step, W)
        walker = [(pa * pos + pb) % W for pos in range(W)]
        nexp = ncon = 0
        for split in (0, 1):
            offS, nS, offC, nC = split_geometry(W, split)
            idx = np.array([walker[offS + k] for k in range(nS)])
            direction = np.empty((nS, ndim))
            z0, lo, hi = np.empty(nS), np.empty(nS), np.empty(nS)
            jb, kb = np.empty(nS, dtype=np.int64), np.empty(nS, dtype=np.int64)
            for k, i in enumerate(idx):
                r = _rand(seed, step, walker_offset + i, 8 + split)
                j = r[0] % nC
                l = (j + 1 + r[1] % (nC - 1)) % nC
                direction[k] = (2.0 * mu) * (X[walker[offC + j]] - X[walker[offC + l]])
                J = int(np.floor(maxsteps * u01(r[2], r[3])))
                q = _rand(seed, step, walker_offset + i, 10 + split)
                z0[k] = Z[i] + np.log(u01(q[0], q[1]))
                lo[k] = -u01(q[2], q[3])
                hi[k] = lo[k] + 1.0
                jb[k], kb[k] = J, maxsteps - 1 - J
            state = np.full(nS, LEFT | RIGHT, dtype=np.int64)
            lit = np.zeros(nS, dtype=np.int64)               # logical iterations consumed per walker
            batches_before = nbatches
            while np.any(state != DONE):
                if np.any(lit[state != DONE] > maxiter):
                    raise RuntimeError("Number of contractions exceeded maximum limit!")
                rows, cand, draws = [], [], {}               # rows: (walker row k, which end / draw, logical iteration)
                for k in np.flatnonzero(state != DONE):
                    i = idx[k]
                    if state[k] == SHRINK:
                        r = _rand(seed, step, walker_offset + i, 16 + 2 * int(lit[k]) + split)
                        t1 = lo[k] + u01(r[0], r[1]) * (hi[k] - lo[k])
                        rows.append((k, SHRINK, 0))
                        cand.append(X[i] + t1 * direction[k])
                        t2 = None
                        if depth > 1:                        # the draw that follows if t1 is rejected
                            lo2, hi2 = (t1, hi[k]) if t1 < 0.0 else (lo[k], t1)
                            r2 = _rand(seed, step, walker_offset + i, 16 + 2 * (int(lit[k]) + 1) + split)
                            t2 = lo2 + u01(r2[0], r2[1]) * (hi2 - lo2)
                            rows.append((k, SHRINK, 1))
                            cand.append(X[i] + t2 * direction[k])
                        draws[k] = (t1, t2)
                        continue
                    if state[k] & LEFT:
                        rows.append((k, LEFT, 0))
                        cand.append(X[i] + lo[k] * direction[k])
                        if depth > 1 and jb[k] >= 1:         # the next test point, if this one succeeds
                            rows.append((k, LEFT, 1))
                            cand.append(X[i] + (lo[k] - 1.0) * direction[k])
                    if state[k] & RIGHT:
                        rows.append((k, RIGHT, 0))
                        cand.append(X[i] + hi[k] * direction[k])
                        if depth > 1 and kb[k] >= 1:
                            rows.append((k, RIGHT, 1))
                            cand.append(X[i] + (hi[k] + 1.0) * direction[k])
                cand = np.array(cand)
                zs = np.asarray(lnprob_fn(cand), dtype=np.float64)
                nbatches += 1
                got = {key: n for n, key in enumerate(rows)}

                def look(k, what, d):
                    n = got[(k, what, d)]
                    if np.isnan(zs[n]):
                        raise ValueError("Probability function returned NaN")
                    return n

                # replay of up to `depth` logical iterations per walker, in order, with the sequential rules; rows
                # the replay does not reach are dropped (not counted)
                for k in np.flatnonzero(state != DONE):
                    if state[k] == SHRINK:
                        for d in range(depth):
                            n = look(k, SHRINK, d)
                            ncall += 1
                            lit[k] += 1
                            if zs[n] >= z0[k]:
                                X[idx[k]] = cand[n]
                                Z[idx[k]] = zs[n]
                                state[k] = DONE
                                break
                            t = draws[k][d]
                            if t < 0.0:
                                lo[k] = t
                            else:
                                hi[k] = t
                            ncon += 1
                        continue
                    for d in range(depth):
                        if state[k] & LEFT:
                            n = look(k, LEFT, d)
                            ncall += 1
                            if zs[n] >= z0[k] and jb[k] >= 1:
                                lo[k] -= 1.0
                                jb[k] -= 1
                                nexp += 1
                            else:
                                state[k] &= ~LEFT
                        if state[k] & RIGHT:
                            n = look(k, RIGHT, d)
                            ncall += 1
                            if zs[n] >= z0[k] and kb[k] >= 1:
                                hi[k] += 1.0
                                kb[k] -= 1
                                nexp += 1
                            else:
                                state[k] &= ~RIGHT
                        lit[k] += 1
                        if state[k] == 0:
                            state[k] = SHRINK               # both ends closed: shrink from the next iteration on
                            break
            per_half.append(nbatches - batches_before)
        chain[s], lps[s] = X, Z
        tot_exp += nexp
        tot_con += ncon
        if tune:
            ne = max(nexp, 1)
            mu = mu * (2.0 * ne / (ne + ncon))
            if abs(ne / (ne + ncon) - 0.5) < tolerance:
                good += 1
            if good > patience:
                tune = False
        mus[s] = mu
    return dict(chain=chain, lnp_chain=lps, mus=mus, mu=mu, tune=tune, good=good, nexp=tot_exp, ncon=tot_con,
                ncall=ncall, nbatches=nbatches, batches_per_half=np.array(per_half, dtype=np.int64))
