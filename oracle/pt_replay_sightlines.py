"""TEST INFRASTRUCTURE ONLY -- numpy restatement of ONE sightline of the device's survey-mode parallel tempering
(rbvfit_b200/csrc/rbv_pt.cuh, C ABI rbv_pt_run_sightlines), random streams and evidence moments included.

Sightline s of a survey run is the one-sightline run of oracle/pt_replay.py with every walker counter of purposes 1-6
offset by s T W (``walker_offset``); the step-split permutation (purpose 0) is shared.  With ``walker_offset=0`` this
replay equals oracle/pt_replay.run, which is unchanged, bit for bit.  It also returns the thermodynamic-integration
moments the survey run accumulates on the device: every step's post-swap lnprob of each temperature merged by
``merge_moments``.  The Philox, permutation, tempered-accept and ladder-adaptation primitives are pt_replay's.
"""
from __future__ import annotations

import numpy as np

from oracle.pt_replay import adapt_ladder, affine_perm_vec, philox_vec, tempered_accept, u01_vec
from oracle.stretch_replay import split_geometry


def merge_moments(moments, x):
    """The device's accumulator step (rbv_pt.cuh): ``moments`` [..., 3] = (n, mean, M2), ``x`` [..., W] one step's
    values -> the merged moments.  x is reduced in walker order to m = (sum x) / W and q = sum (x - m)^2, then
    n' = n + W, d = m - mean, mean' = mean + d (W / n'), M2' = M2 + q + d^2 (n W / n') (Chan et al.)."""
    moments = np.asarray(moments, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    W = x.shape[-1]
    with np.errstate(invalid="ignore", over="ignore"):
        total = np.zeros(x.shape[:-1])
        for k in range(W):
            total = total + x[..., k]
        m = total / float(W)
        q = np.zeros(x.shape[:-1])
        for k in range(W):
            d = x[..., k] - m
            q = q + d * d
        n, mean, M2 = moments[..., 0], moments[..., 1], moments[..., 2]
        n1 = n + float(W)
        d = m - mean
        return np.stack([n1, mean + d * (float(W) / n1), (M2 + q) + (d * d) * ((n * float(W)) / n1)], axis=-1)


def _draws(seed, steps, T, W, walker_offset):
    """Every random number of the steps ``steps`` (they do not depend on the state); every walker counter of
    purposes 1-6 offset by ``walker_offset``."""
    st = np.asarray(steps, dtype=np.uint64)
    r = philox_vec(seed, st, 0xFFFFFFFF, 0)
    pa, pb = affine_perm_vec(r[0], r[1], W)
    walker = (pa[:, None] * np.arange(W)[None, :] + pb[:, None]) % W          # [n, W]: position -> walker
    tt = np.arange(T)[None, :, None]
    halves = []
    for split in (0, 1):
        offS, nS, offC, nC = split_geometry(W, split)
        idx = walker[:, offS:offS + nS]                                          # [n, nS]
        ctr = walker_offset + tt * W + idx[:, None, :]                           # [n, T, nS]
        rp = philox_vec(seed, st[:, None, None], ctr, 1 + split)
        u = u01_vec(rp[0], rp[1])
        j = np.take_along_axis(walker[:, None, :].repeat(T, axis=1), offC + (rp[2] % np.uint64(nC)).astype(np.int64),
                               axis=2)
        ra = philox_vec(seed, st[:, None, None], ctr, 3 + split)
        halves.append((idx, j, u, np.log(u01_vec(ra[0], ra[1]))))
    swaps = None
    if T > 1:
        lv = np.arange(1, T)                                                     # level i at index i - 1
        rp = philox_vec(seed, st[:, None], walker_offset + 2 * lv[None, :], 5)
        rq = philox_vec(seed, st[:, None], walker_offset + 2 * lv[None, :] + 1, 5)
        pa, pb = affine_perm_vec(rp[0], rp[1], W)
        qa, qb = affine_perm_vec(rq[0], rq[1], W)
        k = np.arange(W)
        p = (pa[..., None] * k + pb[..., None]) % W                              # [n, T - 1, W]
        q = (qa[..., None] * k + qb[..., None]) % W
        ru = philox_vec(seed, st[:, None, None], walker_offset + lv[None, :, None] * W + k, 6)
        swaps = (p, q, np.log(u01_vec(ru[0], ru[1])))
    return halves, swaps


def run(lnprob_fn, coords, lnp, betas, nsteps, seed, a_scale=2.0, first_step=0, n_record=1, adapt=False,
        adapt_t0=0, lag=10000.0, tau=100.0, beta_history_device=None, block=64, walker_offset=0, ti=None):
    """One sightline: coords [T, W, ndim], lnp [T, W] (untempered), betas [T]; ``walker_offset`` = s T W for
    sightline s of a survey run.  ``lnprob_fn`` maps (n, ndim) -> (n,).  Returns pt_replay.run's dict plus ti [T, 3]:
    the moments of every step's post-swap lnprob merged into ``ti`` (zeros by default)."""
    coords = np.array(coords, dtype=np.float64, copy=True)
    lnp = np.array(lnp, dtype=np.float64, copy=True)
    b = np.array(betas, dtype=np.float64, copy=True)
    T, W, ndim = coords.shape
    chain = np.empty((nsteps, n_record, W, ndim))
    lps = np.empty((nsteps, T, W))
    bh = np.empty((nsteps, T))
    pred = np.empty((nsteps, T))
    nacc = np.zeros((T, W), dtype=np.int64)
    nswap = np.zeros(max(T - 1, 0), dtype=np.int64)
    mom = np.zeros((T, 3)) if ti is None else np.array(ti, dtype=np.float64, copy=True)
    tt = np.arange(T)[:, None]
    for s0 in range(0, nsteps, block):
        n = min(block, nsteps - s0)
        halves, swaps = _draws(seed, np.arange(first_step + s0, first_step + s0 + n), T, W, walker_offset)
        for ds in range(n):
            s = s0 + ds
            pred[s] = b
            if beta_history_device is not None:
                b = np.array(beta_history_device[s], dtype=np.float64, copy=True)
            bh[s] = b
            for split in (0, 1):
                idx, j, u, lnu = (h[ds] for h in halves[split])
                i = np.broadcast_to(idx[None, :], j.shape)
                t_ = (a_scale - 1.0) * u + 1.0
                zz = t_ * t_ / a_scale
                fac = (ndim - 1.0) * np.log(zz)
                cj = coords[tt, j]
                q = cj - (cj - coords[tt, i]) * zz[..., None]                    # [T, nS, ndim]
                new = np.asarray(lnprob_fn(q.reshape(-1, ndim)), dtype=np.float64).reshape(j.shape)
                acc = tempered_accept(b[:, None], fac, new, lnp[tt, i], lnu)
                ta, ia = np.nonzero(acc)
                wa = i[ta, ia]
                coords[ta, wa] = q[ta, ia]
                lnp[ta, wa] = new[ta, ia]
                nacc[ta, wa] += 1
            n_step = np.zeros(max(T - 1, 0), dtype=np.int64)
            for lvl in range(T - 1, 0, -1):
                p, qq, lu = swaps[0][ds, lvl - 1], swaps[1][ds, lvl - 1], swaps[2][ds, lvl - 1]
                lx, ly = lnp[lvl, p], lnp[lvl - 1, qq]
                with np.errstate(invalid="ignore"):
                    sw = lu < (b[lvl - 1] - b[lvl]) * (lx - ly)
                xs, ys = p[sw], qq[sw]
                cx = coords[lvl, xs].copy()
                coords[lvl, xs] = coords[lvl - 1, ys]
                coords[lvl - 1, ys] = cx
                lnp[lvl, xs], lnp[lvl - 1, ys] = ly[sw], lx[sw]
                n_step[lvl - 1] = int(sw.sum())
            nswap += n_step
            if adapt:
                b = adapt_ladder(b, n_step, W, adapt_t0 + s, lag, tau)
            chain[s] = coords[:n_record]
            lps[s] = lnp
            mom = merge_moments(mom, lnp)
    out = dict(chain=chain, lnp_chain=lps, n_accepted=nacc, n_swaps=nswap, beta_history=bh, betas=b, coords=coords,
               lnp=lnp, ti=mom)
    if beta_history_device is not None:
        out["beta_pred"] = pred
    return out
