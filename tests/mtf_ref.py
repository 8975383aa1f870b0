"""TEST INFRASTRUCTURE: the numpy statement of the diffraction MTF contract (include/ort_b200.h, ort_wavefront_mtf_dev).

Two forms of the lag sums C(k):
- `brute`: the mirrored multiset built explicitly, as psf_ref does -- every kept ray at (+ix, iy) and at (-ix, iy) with
  the same P, the x = 0 column twice -- and every pair of points whose lattice indices differ by the lag summed, with no
  use of the mirror symmetry.  Small sizes only; dtype np.longdouble carries the sums in extended precision.
- `fast`: the mirrored amplitude A (column 0 doubled, width 2 nx - 1) and one shifted product per lag, in row chunks:
  float64, for grids up to the bench size at a handful of frequencies.
Both share the lag selection and the interpolation, which follow the contract's expressions operation for operation."""
import numpy as np

from psf_ref import phase


def steps(ys, xs):
    """the lattice steps by index: dx = xs[-1] / (nx - 1), dy = (ys[-1] - ys[0]) / (ny - 1) (signed)"""
    return xs[-1] / (len(xs) - 1), (ys[-1] - ys[0]) / (len(ys) - 1)


def lattice_ok(ys, xs):
    dx, dy = steps(np.asarray(ys, dtype=np.float64), np.asarray(xs, dtype=np.float64))
    return bool(xs[0] == 0.0 and np.isfinite(dx) and dx > 0 and np.isfinite(dy) and dy != 0)


def lags_brute(P, kmax_s, kmax_t):
    """C_sag(0 .. kmax_s), C_tan(0 .. kmax_t) of the explicit mirrored multiset: P2 = [P, P] at jx = [ix, -ix]"""
    ny, nx = P.shape
    jx = np.concatenate([np.arange(nx), -np.arange(nx)])
    P2 = np.concatenate([P, P], axis=1)                                  # [ny][2 nx]: the 2n-point set, row by row
    D = jx[:, None] - jx[None, :]                                        # jx_p - jx_q of every pair in a row
    cs = np.zeros(kmax_s + 1, dtype=P.dtype)
    for iy in range(ny):
        prod = P2[iy][:, None] * np.conj(P2[iy])[None, :]
        for k in range(kmax_s + 1):
            cs[k] += prod[D == k].sum()
    ct = np.zeros(kmax_t + 1, dtype=P.dtype)
    for k in range(kmax_t + 1):
        for iy in range(ny - k):
            prod = P2[iy + k][:, None] * np.conj(P2[iy])[None, :]
            ct[k] += prod[D == 0].sum()                                  # the two points at jx = 0 pair with each other too
    return cs, ct


def lag_fast(P, az, k, rows=512):
    """C(k) of one azimuth from the mirrored amplitude A (width 2 nx - 1, column 0 doubled), float64"""
    ny, nx = P.shape
    c = 0j
    if az == 0:
        for r0 in range(0, ny, rows):
            p = P[r0:r0 + rows]
            A = np.concatenate([p[:, :0:-1], 2 * p[:, :1], p[:, 1:]], axis=1)
            c += np.sum(A[:, k:] * np.conj(A[:, :A.shape[1] - k]))
        return c
    w = np.full(nx, 2.0)
    w[0] = 4.0
    for c0 in range(0, nx, rows):
        p = P[:, c0:c0 + rows]
        c += np.sum(w[c0:c0 + rows] * np.sum(p[k:] * np.conj(p[:ny - k]), axis=0))
    return c


def select(freqs, s, d, kmax):
    """per frequency: (k0, f) as the device takes them, k0 = -1 past the last lag"""
    out = []
    for nu in np.asarray(freqs, dtype=np.float64):
        q = 0.0 if nu == 0 else nu / (s * d)
        out.append((-1, 0.0) if not q < kmax + 1.0 else (int(np.floor(q)), q - np.floor(q)))
    return out


def set_otf(opd, mask, n_kept, ys, xs, freqs, s, form="fast", dtype=np.float64):
    """one set, opd and mask [ny * nx] (y outer): -> otf (2, n_freq) complex (sagittal, tangential), status"""
    ys, xs = np.asarray(ys, dtype=np.float64), np.asarray(xs, dtype=np.float64)
    ny, nx = len(ys), len(xs)
    keep = np.asarray(mask).reshape(ny, nx) == 1
    W = np.asarray(opd, dtype=np.float64).reshape(ny, nx)
    nan = np.full((2, len(freqs)), np.nan + 1j * np.nan)
    if n_kept <= 0:
        return nan, 1
    if not np.all(np.isfinite(W[keep])):
        return nan, 3
    if not lattice_ok(ys, xs):
        return nan, 4
    dx, dy = steps(ys, xs)
    P = np.where(keep, phase(np.where(keep, W, 0.0), dtype), 0)
    kmax = (2 * (nx - 1), ny - 1)
    sel = [select(freqs, s, dx, kmax[0]), select(freqs, s, abs(dy), kmax[1])]
    if form == "brute":
        cs, ct = lags_brute(P, *kmax)
        C = [lambda k, c=cs: c[k], lambda k, c=ct: c[k]]
    else:
        C = [lambda k: lag_fast(P, 0, k), lambda k: lag_fast(P, 1, k)]
    otf = np.zeros((2, len(freqs)), dtype=np.complex128)
    for az in range(2):
        c0 = C[az](0).real
        val = lambda k: 0j if k > kmax[az] else (1 + 0j if k == 0 else complex(C[az](k) / c0))
        for i, (k0, f) in enumerate(sel[az]):
            if k0 < 0:
                continue
            v = (1 - f) * val(k0) + f * val(k0 + 1)
            v = complex(v.real, 0.0) if az == 0 else (v.conjugate() if dy < 0 else v)
            otf[az, i] = v
    return otf, 0


def sets_otf(opd, mask, stats, ys, xs, freqs, s, form="fast", dtype=np.float64):
    """[n_sets][ny * nx] arrays, ys (ny,) or (n_sets, ny) -> otf (n_sets, 2, n_freq) complex, status (n_sets,)"""
    ys = np.asarray(ys)
    out = [set_otf(opd[j], mask[j], int(stats[j]["n_kept"]), ys[j] if ys.ndim == 2 else ys, xs, freqs, s, form, dtype)
           for j in range(len(opd))]
    return np.stack([o[0] for o in out]), np.array([o[1] for o in out], dtype=np.int32)
