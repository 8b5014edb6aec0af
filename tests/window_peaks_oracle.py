"""NumPy float64 restatement of the windowed seed descent of BigFieldStrip.find_peaks / srhmc_big_find_peaks -- TEST
INFRASTRUCTURE ONLY.  It is the checker of the device descent on images too large for the reference's whole-image
evaluation; it uses the windows of stellar_oracle.patch_eval, and the merge stays stellar_oracle.merge_peaks.  On an
image no larger than rad + 1 pixels per side it is stellar_oracle.ls_find_peaks' descent (checked in
test_bigfield_peaks.py)."""
from __future__ import annotations

import numpy as np

import stellar_oracle as so


def window_find_peaks(L: so.LightSetup, q_seed, rad, f_lim, Nstep=1000, dt_f_coeff=1e-1, dt_xy_coeff=1e-1,
                      whole_image_stop=False, chunk=4096):
    """The descent of find_peaks (samplers.py:196-226) with every potential and gradient of a seed taken over its
    window: the (2 rad + 1)^2 patch centred on the pixel holding it, clipped to the image (the windows of patch_eval),
    on the pure-background model B_count.  The stop test |dV/V| < 1e-9 compares V at the new position with V at the
    old one, both on the window of the new position (the old one is re-evaluated when the step changed the pixel).
    With a window covering the image (num_rows, num_cols <= rad + 1) this is ls_find_peaks' descent.
    whole_image_stop: the stop test uses V summed over the whole image (the reference's rule taken literally: the
    pixels outside the window hold the background alone), which on a large image stops every seed at once.
    q_seed [n,3]; returns (q [n,3], alive [n], steps [n]).  Seeds are processed together, `chunk` at a time."""
    q_seed = np.asarray(q_seed, dtype=float).reshape(-1, 3)
    D = np.asarray(L.D, dtype=float)
    R, C = D.shape
    W = 2 * rad + 1
    sig2 = (L.PSF_FWHM_pix / so.FWHM_TO_SIGMA) ** 2
    norm = 1.0 / (2.0 * np.pi * sig2)
    B = L.B_count
    bg = -(D * np.log(B) - B)   # potential of a background-only pixel
    bg_total = float(np.sum(bg))
    off = np.arange(W) - rad

    def window(x, y):
        mi = np.clip(np.floor(x), 0, R - 1).astype(np.int64)
        mj = np.clip(np.floor(y), 0, C - 1).astype(np.int64)
        return mi, mj

    def evaluate(f, x, y, mi, mj):
        ri, cj = mi[:, None] + off, mj[:, None] + off                     # [m, W]
        mr, mc = (ri >= 0) & (ri < R), (cj >= 0) & (cj < C)
        dx = ri + 0.5 - x[:, None]
        dy = cj + 0.5 - y[:, None]
        ex = np.where(mr, np.exp(-(dx * dx) / (2.0 * sig2)), 0.0)
        ey = np.where(mc, np.exp(-(dy * dy) / (2.0 * sig2)) * norm, 0.0)
        mask = mr[:, :, None] & mc[:, None, :]
        d = np.where(mask, D[np.clip(ri, 0, R - 1)[:, :, None], np.clip(cj, 0, C - 1)[:, None, :]], 0.0)
        psf = ex[:, :, None] * ey[:, None, :]
        lam = B + f[:, None, None] * psf
        V = -np.sum(np.where(mask, d * np.log(lam) - lam, 0.0), axis=(1, 2))
        if whole_image_stop:
            V = V + bg_total - np.sum(np.where(mask, bg[np.clip(ri, 0, R - 1)[:, :, None], np.clip(cj, 0, C - 1)[:, None, :]],
                                               0.0), axis=(1, 2))
        w = np.where(mask, d / lam - 1.0, 0.0) * psf
        g = np.stack([-np.sum(w, axis=(1, 2)),
                      -np.sum(w * dx[:, :, None], axis=(1, 2)) * f / sig2,
                      -np.sum(w * dy[:, None, :], axis=(1, 2)) * f / sig2], axis=1)
        return V, g

    q = q_seed.copy()
    alive = np.ones(len(q), dtype=bool)
    steps = np.zeros(len(q), dtype=np.int64)
    for c0 in range(0, len(q), chunk):
        sel = np.arange(c0, min(len(q), c0 + chunk))
        f, x, y = (q[sel, k].copy() for k in range(3))
        mi, mj = window(x, y)
        V_prev, g = evaluate(f, x, y, mi, mj)
        act = np.arange(len(sel))
        for i in range(Nstep):
            if act.size == 0:
                break
            fo, xo, yo = f[act], x[act], y[act]
            dt_f, dt_xy = fo * dt_f_coeff, dt_xy_coeff / fo
            f[act] = fo - g[act, 0] * dt_f
            x[act] = xo - g[act, 1] * dt_xy
            y[act] = yo - g[act, 2] * dt_xy
            steps[sel[act]] = i + 1
            faint = f[act] < f_lim
            alive[sel[act[faint]]] = False
            keep = ~faint
            act, fo, xo, yo = act[keep], fo[keep], xo[keep], yo[keep]
            nmi, nmj = window(x[act], y[act])
            moved = (nmi != mi[act]) | (nmj != mj[act])
            mi[act], mj[act] = nmi, nmj
            if moved.any():
                V_prev[act[moved]] = evaluate(fo[moved], xo[moved], yo[moved], nmi[moved], nmj[moved])[0]
            V_cur, g_cur = evaluate(f[act], x[act], y[act], nmi, nmj)
            g[act] = g_cur
            stop = np.abs((V_cur - V_prev[act]) / V_prev[act]) < 1e-9
            V_prev[act] = V_cur
            act = act[~stop]
        q[sel, 0], q[sel, 1], q[sel, 2] = f, x, y
    return q, alive, steps
