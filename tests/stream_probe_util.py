"""Per-pixel probes of the lnprob kernels.

The streaming kernel writes no flux, only chi^2, so a lnprob tolerance is all a direct test of it can assert -- and
one pixel's error hides easily in a sum over 10^4 pixels.  The probe recovers single model-flux values from lnprob
instead: a ``SightlineBatch`` whose sightlines all share one instrument (model, wave, taps), where sightline j has
error 1, data 2 everywhere and a ``weight_mask`` that is True only at pixel p_j.  Masked pixels add exact zeros and
sum(log w) = 0, so lnprob_j = -(2 - M_{p_j})^2 / 2, and since 0 <= M <= 1 the residual lies in [1, 2] and
M_{p_j} = 2 - sqrt(-2 lnprob_j) to a few 1e-16 for every theta row.

``oracle_flux_at`` evaluates the CPU oracle only on the pixels an LSF needs around the probed ones, so long spectra
cost the oracle a few thousand pixels per row, not all of them."""
import numpy as np

SUPER = 1024     # super-chunk: the unit of the streaming kernel's range schedule
ROW = 256        # pixels of one row of the streaming kernel


def n_taps(om) -> int:
    return 1 if om.kernel_taps is None else int(np.asarray(om.kernel_taps).size)


def line_x_a(om, theta, wave):
    """x [L, P] and a [L] of every line at every pixel, with the oracle's own lowering (oracle.voigt_tau)."""
    theta, wave = np.asarray(theta, dtype=np.float64), np.asarray(wave, dtype=np.float64)
    c = 299792.458
    z_total = om.z_factors * (1 + theta[om.v_indices] / c) - 1
    lam0 = om.atomic_lambda0[:, None]
    b_f = theta[om.b_indices][:, None] / lam0 * 1e13
    freq0 = 2.99792458e18 / lam0
    freq = 2.99792458e18 / (wave[None, :] / (1 + z_total[:, None]))
    return (freq - freq0) / b_f, (np.asarray(om.atomic_gamma, dtype=np.float64)[:, None] / (4 * np.pi * b_f))[:, 0]


def probe_pixels(P, K, om=None, theta=None, wave=None, n_random=24, seed=0, targets=(64.0, 576.0, 4e4)):
    """Sorted unique pixel indices where a lnprob kernel can go wrong:
    - every pixel within K + 1 of a multiple of 1024 (any range boundary of any schedule);
    - the first and the last K + 2 pixels (edge replication of the LSF);
    - +-1 around each multiple of 256 (row starts) in the first two super-chunks;
    - per line (with ``om``, ``theta``, ``wave``): the pixels nearest to |z|^2 = x^2 + a^2 = each of ``targets``
      (default 64, 576 and 4e4, the kernels' Voigt tier switches) on either side of the line, and the one nearest to
      its centre;
    - ``n_random`` seeded random pixels."""
    sel = [np.arange(min(P, K + 2)), np.arange(max(0, P - K - 2), P)]
    for m in range(SUPER, P, SUPER):
        sel.append(np.arange(m - K - 1, m + K + 2))
    for m in range(ROW, 2 * SUPER + 1, ROW):
        sel.append(np.arange(m - 1, m + 2))
    if om is not None:
        x, a = line_x_a(om, theta, wave)
        for xl, al in zip(x, a):
            z2 = xl * xl + al * al
            sel.append([int(np.argmin(np.abs(xl)))])
            for target in targets:
                for side in (xl < 0, xl >= 0):
                    if side.any():
                        d = np.where(side, np.abs(z2 - target), np.inf)
                        sel.append([int(np.argmin(d))])
    sel.append(np.random.default_rng(seed).integers(0, P, n_random))
    px = np.unique(np.concatenate([np.asarray(s, dtype=np.int64).ravel() for s in sel]))
    return px[(px >= 0) & (px < P)]


def boundary_windows(P, K):
    """Pixels within K + 2 of each multiple of 1024: the outputs behind every possible range boundary."""
    sel = [np.arange(m - K - 2, m + K + 2) for m in range(SUPER, P, SUPER)]
    if not sel:
        return np.zeros(0, dtype=np.int64)
    px = np.unique(np.concatenate(sel))
    return px[(px >= 0) & (px < P)]


def oracle_flux_at(om, theta, wave, px):
    """The oracle's LSF-convolved model flux (oracle.voigt_oracle.model_flux) at pixels ``px`` only: the unconvolved
    flux on the pixels the kernel reaches, then out[i] = sum_m k[m] f[clip(i + h - m)] with k the normalised taps --
    what both ndimage.convolve1d(mode='nearest') and convolve_extend compute for an odd kernel."""
    from oracle import voigt_oracle as vo
    wave = np.asarray(wave, dtype=np.float64)
    px = np.asarray(px, dtype=np.int64)
    P, K = wave.size, n_taps(om)
    if K == 1:
        return vo.model_flux(om, theta, wave[px], convolve=False)
    h = K // 2
    taps = np.asarray(om.kernel_taps, dtype=np.float64)
    k = taps / taps.sum()
    src = np.clip(px[:, None] + h - np.arange(K)[None, :], 0, P - 1)
    need = np.unique(src)
    raw = vo.model_flux(om, theta, wave[need], convolve=False)
    return (raw[np.searchsorted(need, src)] * k[None, :]).sum(axis=1)


def probe_sightlines(compiled, wave, px):
    """One sightline per probed pixel: error 1, data 2, weight 1 at that pixel only."""
    wave = np.asarray(wave, dtype=np.float64)
    P = wave.size
    flux, error = np.full(P, 2.0), np.ones(P)
    out = []
    for p in px:
        mask = np.zeros(P, dtype=bool)
        mask[p] = True
        out.append(dict(model=compiled, wave=wave, flux=flux, error=error, weight_mask=mask))
    return out


def flux_from_lnprob(lnp):
    """M = 2 - sqrt(-2 lnprob) (data 2, error 1, one unmasked pixel)."""
    return 2.0 - np.sqrt(-2.0 * np.asarray(lnp, dtype=np.float64))


def probe_lnprob_numpy(om, thetas, wave, px):
    """The probe's lnprob [S, Ws] restated in numpy on the oracle flux (vfit.lnlike with weight 1 at p_j only): the
    CPU self-check of the harness."""
    from oracle import voigt_oracle as vo
    wave = np.asarray(wave, dtype=np.float64)
    out = np.empty((len(px), len(thetas)))
    for j, s in enumerate(probe_sightlines(None, wave, px)):
        err, mask = s["error"], s["weight_mask"]
        w = np.where(mask, 1.0 / err ** 2, 0.0)                  # likelihood._weights, then the mask
        lw = np.where(mask, np.log(1.0 / err ** 2), 0.0)
        for r, th in enumerate(thetas):
            M = vo.model_flux(om, th, wave)
            out[j, r] = -0.5 * np.sum((s["flux"] - M) ** 2 * w - lw)
    return out


def probe_model_flux(model, wave, thetas, px, lb, ub, far_field=None):
    """GPU model flux [Ws, S] at pixels ``px`` for theta rows ``thetas`` [Ws, ndim], recovered from one sightline-mode
    lnprob launch, and the kernel that launch took ('stream' / 'tile')."""
    from rbvfit_b200.likelihood import SightlineBatch
    from rbvfit_b200.model import GpuVoigtModel
    compiled = model.compile() if isinstance(model, GpuVoigtModel) else model
    thetas = np.atleast_2d(np.asarray(thetas, dtype=np.float64))
    batch = SightlineBatch(probe_sightlines(compiled, wave, px), lb, ub)
    try:
        if far_field is not None:
            batch.engine.set_farfield(far_field)
        lnp = batch.lnprob(np.ascontiguousarray(np.broadcast_to(thetas, (len(px),) + thetas.shape)))
        kernel = batch.engine.last_kernel
    finally:
        batch.close()
    return flux_from_lnprob(lnp.T), kernel
