"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the device's parallel tempering (rbvfit_b200/csrc/rbv_pt.cuh,
C ABI rbv_pt_run), random streams included.

Built on oracle/stretch_replay.py (Philox4x32-10, uniforms, the step's split): the stretch move of every temperature
is that replay's with the walker counter offset by t W, accepted against prior x L^beta_t; then ptemcee's swap stage
(Vousden, Farr & Mandel 2016), hottest pair first, and optionally its ladder adaptation.  What the device adds and is
restated here bit for bit:

  * tempered accept: a -inf (or NaN) proposal is rejected; a walker at -inf accepts; else
    ln u < ((ndim - 1) ln z + beta new) - beta old;
  * swap level i = T-1 .. 1: p_i / q_i = affine permutations from purpose 5, walker counter 2 i / 2 i + 1 (a advanced
    until gcd(a, W) = 1); pair k = (walker p_i(k) of temperature i, walker q_i(k) of i - 1), its u from purpose 6,
    walker counter i W + k; swap when ln u < (beta_{i-1} - beta_i)(lnL_i - lnL_{i-1});
  * the record is the state after the swaps; beta_history[s] is the ladder step s ran with.

Philox is vectorised over walkers and blocks of steps with numpy uint64 arithmetic (the scalar version of
stretch_replay.py is too slow for thousands of steps over tens of temperatures); with T = 1 the chain equals
stretch_replay.run's exactly.  Driven by the GPU's lnprob this reproduces the device chain; with adaptation on,
exp / log may differ in the last bit, so ``beta_history_device`` lets the replay continue from the device's ladder
and return its own prediction of every step's ladder for comparison.
"""
from __future__ import annotations

import numpy as np

from oracle.stretch_replay import M0, M1, MASK, W0, W1, split_geometry

_M0, _M1, _MASK = np.uint64(M0), np.uint64(M1), np.uint64(MASK)


def philox_vec(seed, step, walker, purpose):
    """philox4x32_10 of stretch_replay over broadcast arrays: counter (step lo, step hi, walker, purpose),
    key = seed -> four uint64 arrays holding 32-bit words."""
    step = np.asarray(step, dtype=np.uint64)
    walker, purpose = np.asarray(walker, dtype=np.uint64), np.asarray(purpose, dtype=np.uint64)
    step, walker, purpose = np.broadcast_arrays(step, walker, purpose)
    c0, c1 = step & _MASK, step >> np.uint64(32)
    c2, c3 = walker & _MASK, purpose & _MASK
    k0, k1 = int(seed) & MASK, (int(seed) >> 32) & MASK
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> s32) ^ c1 ^ np.uint64(k0)) & _MASK, p1 & _MASK, \
                         ((p0 >> s32) ^ c3 ^ np.uint64(k1)) & _MASK, p0 & _MASK
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return c0, c1, c2, c3


def u01_vec(hi, lo):
    m = ((hi << np.uint64(32)) | lo) >> np.uint64(11)
    return (m.astype(np.float64) + 0.5) * 1.1102230246251565e-16


def affine_perm_vec(rx, ry, W):
    """(a, b) of the affine permutations pos -> (a pos + b) mod W drawn as (rx, ry); a advanced until gcd(a, W) = 1."""
    a, b = (rx % np.uint64(W)).astype(np.int64), (ry % np.uint64(W)).astype(np.int64)
    if W == 1:
        return a, b
    while True:
        bad = np.gcd(a, W) != 1
        if not bad.any():
            return a, b
        a[bad] = (a[bad] + 1) % W


def _draws(seed, steps, T, W):
    """Every random number of the steps ``steps`` (they do not depend on the state)."""
    n = len(steps)
    st = np.asarray(steps, dtype=np.uint64)
    r = philox_vec(seed, st, 0xFFFFFFFF, 0)
    pa, pb = affine_perm_vec(r[0], r[1], W)
    walker = (pa[:, None] * np.arange(W)[None, :] + pb[:, None]) % W          # [n, W]: position -> walker
    tt = np.arange(T)[None, :, None]
    halves = []
    for split in (0, 1):
        offS, nS, offC, nC = split_geometry(W, split)
        idx = walker[:, offS:offS + nS]                                          # [n, nS]
        ctr = tt * W + idx[:, None, :]                                           # [n, T, nS]
        rp = philox_vec(seed, st[:, None, None], ctr, 1 + split)
        u = u01_vec(rp[0], rp[1])
        j = np.take_along_axis(walker[:, None, :].repeat(T, axis=1), offC + (rp[2] % np.uint64(nC)).astype(np.int64),
                               axis=2)
        ra = philox_vec(seed, st[:, None, None], ctr, 3 + split)
        halves.append((idx, j, u, np.log(u01_vec(ra[0], ra[1]))))
    swaps = None
    if T > 1:
        lv = np.arange(1, T)                                                     # level i at index i - 1
        rp = philox_vec(seed, st[:, None], 2 * lv[None, :], 5)
        rq = philox_vec(seed, st[:, None], 2 * lv[None, :] + 1, 5)
        pa, pb = affine_perm_vec(rp[0], rp[1], W)
        qa, qb = affine_perm_vec(rq[0], rq[1], W)
        k = np.arange(W)
        p = (pa[..., None] * k + pb[..., None]) % W                              # [n, T - 1, W]
        q = (qa[..., None] * k + qb[..., None]) % W
        ru = philox_vec(seed, st[:, None, None], lv[None, :, None] * W + k, 6)
        swaps = (p, q, np.log(u01_vec(ru[0], ru[1])))
    return halves, swaps


def tempered_accept(beta, fac, new, old, lnu):
    with np.errstate(invalid="ignore"):
        lnq = (fac + beta * new) - beta * old
        return np.where(~(new > -np.inf), False, np.where(old == -np.inf, True, lnu < lnq))


def adapt_ladder(betas, n_acc, W, t, lag=10000.0, tau=100.0):
    """ptemcee's ladder adjustment after a step with n_acc [T - 1] accepted swaps; t = adaptation steps before it."""
    b = np.array(betas, dtype=np.float64, copy=True)
    if len(b) < 3:
        return b
    A = n_acc / float(W)
    kappa = (lag / (float(t) + lag)) / tau
    dS = kappa * (A[:-1] - A[1:])
    inv = 1.0 / b[:-1]
    dT = np.diff(inv) * np.exp(dS)
    b[1:-1] = 1.0 / (np.cumsum(dT) + inv[0])
    return b


def run(lnprob_fn, coords, lnp, betas, nsteps, seed, a_scale=2.0, first_step=0, n_record=1, adapt=False,
        adapt_t0=0, lag=10000.0, tau=100.0, beta_history_device=None, block=64):
    """coords [T, W, ndim], lnp [T, W] (untempered), betas [T].  ``lnprob_fn`` maps (n, ndim) -> (n,).
    Returns a dict: chain [n, n_record, W, ndim], lnp_chain [n, T, W], n_accepted [T, W], n_swaps [T - 1],
    beta_history [n, T] (the ladder each step ran with), betas (after the run), coords, lnp; with
    ``beta_history_device`` the ladder of step s is the device's row s and beta_pred [n, T] is the replay's own."""
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
    tt = np.arange(T)[:, None]
    for s0 in range(0, nsteps, block):
        n = min(block, nsteps - s0)
        halves, swaps = _draws(seed, np.arange(first_step + s0, first_step + s0 + n), T, W)
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
    out = dict(chain=chain, lnp_chain=lps, n_accepted=nacc, n_swaps=nswap, beta_history=bh, betas=b, coords=coords,
               lnp=lnp)
    if beta_history_device is not None:
        out["beta_pred"] = pred
    return out
