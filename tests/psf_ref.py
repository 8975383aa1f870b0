"""TEST INFRASTRUCTURE: the numpy statement of the diffraction PSF contract (include/ort_b200.h, ort_wavefront_psf_dev).
It evaluates the explicit mirrored 2n-point sum -- every kept ray at (+x, y) and at (-x, y) with the same W -- as
matrix products over the pupil grid, not the device's cos form and not its column mirror."""
import numpy as np


def pixels(n, d):
    """pixel centres (i - (n - 1)/2) d, i = 0 .. n - 1"""
    return (np.arange(n) - (n - 1) / 2) * d


def phase(w, dtype=np.float64):
    """exp(2 pi i w), with the integer part of w removed exactly first (|w| may be ~1e6 waves)"""
    w = np.asarray(w, dtype=dtype)
    return np.exp((2j * np.pi) * (w - np.round(w)))


def set_psf(opd, mask, n_kept, ys, xs, n_u, n_v, du, dv, s, dtype=np.float64):
    """one set, opd and mask [ny * nx] (y outer): -> psf (n_v, n_u), strehl (2,) = (strehl_ref, max psf), peak, status.
    dtype np.longdouble carries the whole sum in extended precision (small sizes only)."""
    ys, xs = np.asarray(ys, dtype=dtype), np.asarray(xs, dtype=dtype)
    ny, nx = len(ys), len(xs)
    keep = np.asarray(mask).reshape(ny, nx) == 1
    W = np.asarray(opd, dtype=np.float64).reshape(ny, nx)
    nan = np.full((n_v, n_u), np.nan)
    if n_kept <= 0:
        return nan, np.array([np.nan, np.nan]), -1, 1
    if not np.all(np.isfinite(W[keep])):
        return nan, np.array([np.nan, np.nan]), -1, 3
    P = np.where(keep, phase(np.where(keep, W, 0.0), dtype), 0)                  # [ny][nx]
    P2 = np.concatenate([P, P], axis=1)                                          # the mirrored set: +x, then -x
    x2 = np.concatenate([xs, -xs])
    xi, eta = pixels(n_u, du).astype(dtype), pixels(n_v, dv).astype(dtype)
    s = dtype(s)
    X = np.exp((2j * np.pi) * (s * x2[:, None] * xi[None, :]))                    # [2 nx][n_u]
    Y = np.exp((2j * np.pi) * (s * eta[:, None] * ys[None, :]))                   # [n_v][ny]
    E = Y @ (P2 @ X)
    n = dtype(n_kept)
    psf = (np.abs(E) ** 2 / (2 * n) ** 2).astype(np.float64)
    ref = float(np.abs(P.sum()) ** 2 / n ** 2)
    peak = int(np.argmax(psf))
    return psf, np.array([ref, psf.ravel()[peak]]), peak, 0


def sets_psf(opd, mask, stats, ys, xs, n_u, n_v, du, dv, s, dtype=np.float64):
    """[n_sets][ny * nx] arrays, ys (ny,) or (n_sets, ny) -> psf (n_sets, n_v, n_u), strehl (n_sets, 2), peak, status"""
    ys = np.asarray(ys)
    out = [set_psf(opd[j], mask[j], int(stats[j]["n_kept"]), ys[j] if ys.ndim == 2 else ys, xs, n_u, n_v, du, dv, s,
                   dtype) for j in range(len(opd))]
    return (np.stack([o[0] for o in out]), np.stack([o[1] for o in out]), np.array([o[2] for o in out], dtype=np.int32),
            np.array([o[3] for o in out], dtype=np.int32))
