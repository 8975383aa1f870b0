"""numpy statement of the Zernike-fit contract of include/ort_b200.h (ort_wavefront_zernike_dev): the ANSI Z80.28 / OSA
basis and index, the split into terms symmetric and antisymmetric under the mirror theta -> pi - theta, the full-basis
least-squares fit of the explicitly mirrored set, and a normal-equation fit accumulated in np.longdouble for large
sets -- what the device must equal within a tolerance derived from the conditioning of the normal matrix."""
from math import factorial

import numpy as np

EPS = np.finfo(np.float64).eps
PIVOT = 1e-10                  # status 2: a Cholesky pivot <= PIVOT x its diagonal entry of G


def n_terms(n_max):
    return (n_max + 1) * (n_max + 2) // 2


def ansi_index(n_max):
    """(n, m) of j = (n(n+2) + m)/2, j = 0 .. n_terms(n_max) - 1"""
    nm = [(n, m) for n in range(n_max + 1) for m in range(-n, n + 1, 2)]
    return np.array([a for a, _ in nm]), np.array([b for _, b in nm])


def symmetric(n_max):
    """True for the terms the mirror keeps: cos m theta with m even (m >= 0), sin |m| theta with |m| odd (m < 0)"""
    _, m = ansi_index(n_max)
    return np.where(np.abs(m) % 2 == 0, m >= 0, m < 0)


def norm(n, m):
    return np.sqrt(2.0 * (n + 1) / (1.0 + (m == 0)))


def basis(n_max, rho, theta, dtype=np.float64, cols=None):
    """[len(rho)][J] matrix of Z_j(rho, theta) in ANSI order (or only the columns `cols`), evaluated in dtype by the
    factorial sum of R_n^|m|"""
    rho, theta = np.asarray(rho, dtype=dtype), np.asarray(theta, dtype=dtype)
    n, m = ansi_index(n_max)
    js = range(len(n)) if cols is None else np.flatnonzero(cols)
    pw = [np.ones_like(rho)]
    for _ in range(n_max):
        pw.append(pw[-1] * rho)
    cs = {k: (np.cos(k * theta), np.sin(k * theta)) for k in range(1, n_max + 1)}
    out = np.empty((len(rho), len(js)), dtype=dtype)
    for c, j in enumerate(js):
        nn, am = int(n[j]), abs(int(m[j]))
        R = np.zeros_like(rho)
        for k in range((nn - am) // 2 + 1):
            R = R + dtype(radial_coef(nn, am, k)) * pw[nn - 2 * k]
        ang = cs[am][0] if m[j] > 0 else cs[am][1] if m[j] < 0 else 1
        out[:, c] = dtype(norm(nn, int(m[j]))) * R * ang
    return out


def radial_coef(n, am, k):
    """the coefficient of rho^(n - 2k) in R_n^|m|"""
    return (-1) ** k * factorial(n - k) // (factorial(k) * factorial((n + am) // 2 - k) * factorial((n - am) // 2 - k))


def lstsq_mirrored(opd, rho, theta, n_max):
    """full-basis least squares over the 2n points (rho, theta), (rho, pi - theta), both with opd"""
    r2 = np.concatenate([rho, rho])
    t2 = np.concatenate([theta, np.pi - theta])
    A = basis(n_max, r2, t2)
    return np.linalg.lstsq(A, np.concatenate([opd, opd]), rcond=None)[0]


def _cholesky_solve(G, b):
    """(c, ok) of G c = b by Cholesky in G's dtype; ok False when a pivot is <= PIVOT x its diagonal entry"""
    J = len(b)
    L = np.zeros_like(G)
    for k in range(J):
        d = G[k, k] - np.dot(L[k, :k], L[k, :k])
        if not d > PIVOT * G[k, k]:
            return None, False
        L[k, k] = np.sqrt(d)
        for i in range(k + 1, J):
            L[i, k] = (G[i, k] - np.dot(L[i, :k], L[k, :k])) / L[k, k]
    y = np.zeros_like(b)
    for k in range(J):
        y[k] = (b[k] - np.dot(L[k, :k], y[:k])) / L[k, k]
    c = np.zeros_like(b)
    for k in reversed(range(J)):
        c[k] = (y[k] - np.dot(L[k + 1:, k], c[k + 1:])) / L[k, k]
    return c, True


def normal_equations(opd, rho, theta, n_max, chunk=1 << 16, basis_dtype=np.longdouble):
    """(G, b) of the symmetric subset, accumulated chunk by chunk in np.longdouble (each chunk's products in float64 from
    a basis evaluated in basis_dtype; float64 loses ~1e-13 near rho = 1 at n = 12 and is ~10 x faster for bench-size
    sets).  The fitted terms of a lower order are the leading rows and columns."""
    sym = symmetric(n_max)
    Js = int(sym.sum())
    G = np.zeros((Js, Js), dtype=np.longdouble)
    b = np.zeros(Js, dtype=np.longdouble)
    for i0 in range(0, len(opd), chunk):
        Z = basis(n_max, np.asarray(rho[i0:i0 + chunk], dtype=basis_dtype),
                  np.asarray(theta[i0:i0 + chunk], dtype=basis_dtype), basis_dtype, sym).astype(np.float64)
        G += (Z.T @ Z).astype(np.longdouble)
        b += (Z.T @ np.asarray(opd[i0:i0 + chunk], dtype=np.float64)).astype(np.longdouble)
    return G, b


def solve_normal(G, b, n_max):
    """coef [J] float64 (antisymmetric terms exactly 0) of the normal equations of order n_max, or None when singular;
    G, b may be those of a higher order"""
    sym = symmetric(n_max)
    Js = int(sym.sum())
    c, ok = _cholesky_solve(G[:Js, :Js], b[:Js])
    if not ok:
        return None
    coef = np.zeros(n_terms(n_max))
    coef[sym] = c.astype(np.float64)
    return coef


def normal_fit(opd, rho, theta, n_max, chunk=1 << 16):
    """the longdouble normal-equation fit -> (coef or None when singular, G float64)"""
    G, b = normal_equations(opd, rho, theta, n_max, chunk)
    return solve_normal(G, b, n_max), G.astype(np.float64)


def residual(opd, rho, theta, n_max, coef, chunk=1 << 16, dtype=np.longdouble):
    """(RMS, PV) of opd - sum c_j Z_j over the rays, the fit evaluated in dtype and the squares summed in longdouble"""
    ssq, lo, hi = np.longdouble(0), np.inf, -np.inf
    sym = symmetric(n_max)
    for i0 in range(0, len(opd), chunk):
        Z = basis(n_max, np.asarray(rho[i0:i0 + chunk], dtype=dtype), np.asarray(theta[i0:i0 + chunk], dtype=dtype),
                  dtype, sym)
        e = np.asarray(opd[i0:i0 + chunk], dtype=dtype) - Z @ np.asarray(coef[sym], dtype=dtype)
        ssq += np.sum(np.asarray(e * e, dtype=np.longdouble))
        lo, hi = min(lo, float(e.min())), max(hi, float(e.max()))
    return float(np.sqrt(ssq / len(opd))), hi - lo


def kept(opd, r, theta, mask, n_kept):
    """the kept rays of one set: full grid with mask (uint8, kept == 1) or compacted (mask None: the first n_kept)"""
    if mask is None:
        return opd[:n_kept], r[:n_kept], theta[:n_kept]
    k = np.asarray(mask) == 1
    return opd[k], r[k], theta[k]


def set_fit(opd, r, theta, mask, n_kept, r_max, n_max, r_norm):
    """coef, (RMS, PV), status of one set as the header defines them; r_norm 0 means r_max"""
    o, rr, th = kept(opd, r, theta, mask, n_kept)
    J = n_terms(n_max)
    nan = (np.full(J, np.nan), (np.nan, np.nan))
    if len(o) < int(symmetric(n_max).sum()):
        return nan + (1,)
    if not np.all(np.isfinite(o)):
        return nan + (3,)
    rho = rr / (r_norm if r_norm > 0 else r_max)
    coef, _ = normal_fit(o, rho, th, n_max)
    if coef is None:
        return nan + (2,)
    return coef, residual(o, rho, th, n_max, coef), 0


def cond_tol(G, n):
    """error bound of a coefficient relative to the size of the data: the normal equations lose cond(G) times what
    summing n products loses, sqrt(n) rounding errors on a random walk; with a factor 8 for the evaluation of the
    terms and the solve"""
    return 8.0 * np.linalg.cond(G) * np.sqrt(max(n, 1)) * EPS
