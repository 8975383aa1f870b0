"""Plain op-for-op statement of the reference's 2-D meridional trace, raytrace(surfaces, y, U, RealRay)
(src/RayTracing.jl:145-173: transfer :152, sag :75-88 with sec^2 U + K, :158-161, tilt :98-101, Snell :163-164), in
Python floats, with the libm calls made through glibc's libm so that its roundings are the ones the CPU oracle gets.

`branch` names how the tilt angle of a surface is taken:
  "asin"         AbstractMatrix / Layout{Spherical}: K forced to 0, asin(tilt(y, R)) on every surface (:162, :101)
  "atan_always"  Layout{Aspheric}: K from the layout, atan(tilt(y, R, K, p)) on every surface -- its p holds
                 Polynomial(zero), which is not === zero, so iszero(Ks) && ps === zero never holds (src/Types.jl:27, 91)
  "per_surface"  K from the layout, asin where K == 0 and atan elsewhere: the rule the tracers used to follow

Near grazing incidence (|y / R| -> 1) asin(y / R) and atan(y / sqrt(R^2 - y^2)) round very differently, so a ray chosen
there tells which form a tracer took.  grazing_rays() finds such rays.
"""
import ctypes
import ctypes.util
import math

import numpy as np

LIBM_NAME = ctypes.util.find_library("m")
_m = ctypes.CDLL(LIBM_NAME)
for _f in ("tan", "cos", "sin", "asin", "atan"):
    getattr(_m, _f).restype = ctypes.c_double
    getattr(_m, _f).argtypes = [ctypes.c_double]
tan, cos, sin, asin, atan = _m.tan, _m.cos, _m.sin, _m.asin, _m.atan

F_MISS, F_TIR, F_DOMAIN = 1, 2, 4
BRANCHES = ("asin", "atan_always", "per_surface")


def _sign(x):
    return 1.0 if x > 0.0 else (-1.0 if x < 0.0 else x)


def _div(a, b):
    """a / b with IEEE semantics for b == 0 (Python raises)"""
    if b != 0.0:
        return a / b
    if a != a or a == 0.0:
        return math.nan
    return math.copysign(math.inf, a) * math.copysign(1.0, b)


def _sqrt(x):
    return math.sqrt(x) if x >= 0.0 else math.nan


def tilt(y, R, K, use_asin):
    """theta of the surface at height y and whether its argument left the domain (:98-101)"""
    if use_asin:
        q = _div(y, R)
        return (asin(q), abs(q) > 1.0) if not abs(q) > 1.0 else (math.nan, True)
    D = R * R - y * y * (1.0 + K)
    return atan(_div(_sign(R) * y, _sqrt(D))), D < 0.0


def refract(U, theta, n1, n2):
    """U after the surface (:163-164) and whether the ray was totally reflected"""
    sin_ip = _div(n1 * sin(U + theta), n2)
    if abs(sin_ip) <= 1.0:
        return asin(sin_ip) - theta, False
    return math.nan, abs(sin_ip) > 1.0


def trace(R, t, n, K, y, U, branch):
    """one ray -> (y at every row, U at every row, ts, flags), the layout of orc_trace2d"""
    rows = len(R)
    ts = [float(v) for v in t]
    ys, Us = [y], [U]
    flags = 0
    for i in range(rows - 1):
        tU = tan(U)
        y = y + tU * ts[i]                                   # :152
        Rs = R[i + 1]
        Ks = 0.0 if branch == "asin" else float(K[i + 1])
        if math.isfinite(Rs):                                # sag :75-88
            beta = Rs - y * tan(U)
            y2 = y * y
            sec = _div(1.0, cos(U))
            D = beta * beta - y2 * (sec * sec + Ks)
            if D >= 0.0:
                s = _div(y2, beta + _sign(Rs) * math.sqrt(D))
            else:
                s = math.nan
                if D < 0.0:
                    flags |= F_MISS
        else:
            s = 0.0
        y = y + s * tan(U)                                   # :158
        ts[i] += s                                           # :160
        ts[i + 1] -= s                                       # :161
        use_asin = branch == "asin" or (branch == "per_surface" and Ks == 0.0)
        theta, dom = tilt(y, Rs, Ks, use_asin)
        if dom:
            flags |= F_DOMAIN
        U, tir = refract(U, theta, n[i], n[i + 1])
        if tir:
            flags |= F_TIR
        ys.append(y)
        Us.append(U)
    return ys, Us, ts, flags


def batch(S, K, y0, U0, branch):
    """rays -> (y, U, ts) as (rows, N) arrays and flags (N,), the layout of orc.trace2d_batch"""
    S = np.asarray(S, dtype=np.float64)
    R, t, n = [float(v) for v in S[:, 0]], [float(v) for v in S[:, 1]], [float(v) for v in S[:, 2]]
    Kl = [0.0] * len(R) if K is None else [float(v) for v in K]
    N = len(y0)
    Y, UU, TS = (np.empty((len(R), N)) for _ in range(3))
    F = np.zeros(N, dtype=np.uint8)
    for j in range(N):
        ys, Us, ts, f = trace(R, t, n, Kl, float(y0[j]), float(U0[j]), branch)
        Y[:, j], UU[:, j], TS[:, j], F[j] = ys, Us, ts, f
    return Y, UU, TS, F


def ulp_diff(a, b):
    """distance in units in the last place between two finite doubles of the same sign"""
    ia = np.asarray(a, dtype=np.float64).view(np.int64).astype(object)
    ib = np.asarray(b, dtype=np.float64).view(np.int64).astype(object)
    return np.abs(np.asarray(ia - ib, dtype=np.float64))


def surface_step(R, K, n1, n2, y, U_in, use_asin):
    """U after one surface from the hit height y on it and the U that arrived (:162-164)"""
    theta, _ = tilt(y, R, K, use_asin)
    return refract(U_in, theta, n1, n2)[0]


def grazing_rays(S, K, surf, U0=0.0, n_targets=160, seed=0, min_ulp=32, lo=1e-7, hi=1e-5):
    """Entrance heights y0 (rays of slope angle U0) whose hit on surface `surf` lands at |y / R| = 1 - d, d drawn
    log-uniformly in [lo, hi], and for which the atan and asin forms of that surface's tilt give U after it at least
    `min_ulp` ulp apart (both forms taken from the same hit height and incoming U).  The height is bisected on the
    "atan_always" trace; the surface must be a K = 0 sphere.  Returns (y0 array, ulp distances)."""
    S = np.asarray(S, dtype=np.float64)
    R, t, n = [float(v) for v in S[:, 0]], [float(v) for v in S[:, 1]], [float(v) for v in S[:, 2]]
    Kl = [0.0] * len(R) if K is None else [float(v) for v in K]
    Rj = R[surf]
    assert Kl[surf] == 0.0 and math.isfinite(Rj)

    def q_at(y):                      # |y / R| on the surface, None once the ray has failed before it
        ys, Us, _, _ = trace(R[:surf + 1], t[:surf + 1], n[:surf + 1], Kl[:surf + 1], y, U0, "atan_always")
        v = abs(ys[surf] / Rj)
        return v if math.isfinite(v) and all(math.isfinite(u) for u in Us[:surf]) else None

    # bracket: scan outwards on both sides of the axis for the last height still short of 1 - lo
    brackets = []
    for side in (1.0, -1.0):
        grid = side * np.linspace(0.0, 4.0 * abs(Rj), 4001)
        prev = None
        for y in grid:
            q = q_at(float(y))
            if prev is not None and prev[1] is not None and prev[1] < 1.0 - hi and (q is None or q > 1.0 - lo):
                brackets.append((prev[0], float(y)))
                break
            prev = (float(y), q)
    assert brackets, "surface %d cannot be reached near grazing" % surf
    rng = np.random.default_rng(seed)
    out, dist = [], []
    for k in range(n_targets):
        a, b = brackets[k % len(brackets)]
        target = 1.0 - 10.0 ** rng.uniform(math.log10(lo), math.log10(hi))
        for _ in range(80):
            m = 0.5 * (a + b)
            if m == a or m == b:
                break
            q = q_at(m)
            if q is not None and q < target:
                a = m
            else:
                b = m
        ys, Us, _, _ = trace(R[:surf + 1], t[:surf + 1], n[:surf + 1], Kl[:surf + 1], a, U0, "atan_always")
        if not (q_at(a) is not None and 1.0 - 2 * hi < q_at(a) < 1.0 - lo / 2):
            continue
        ua = surface_step(Rj, 0.0, n[surf - 1], n[surf], ys[surf], Us[surf - 1], False)
        us = surface_step(Rj, 0.0, n[surf - 1], n[surf], ys[surf], Us[surf - 1], True)
        if math.isfinite(ua) and math.isfinite(us) and ulp_diff(ua, us) >= min_ulp:
            out.append(a)
            dist.append(float(ulp_diff(ua, us)))
    return np.array(out), np.array(dist)


# A purpose-built Layout{Aspheric} whose K = 0 sphere is the SECOND surface and can be reached near grazing.  Only a ray
# that meets a sphere parallel to the axis can come within 1e-5 of |y / R| = 1 (a ray of slope angle U leaves it at
# cos U), so the surface before it is a plane: a ray entering at U = 0 keeps U = 0 and its height.  The sphere takes the
# ray from glass into denser glass, so a grazing ray is refracted, not totally reflected.
DEEP = np.array([[np.inf, 0.0, 1.0, 0.0],
                 [np.inf, 4.0, 1.5, 0.0],
                 [-40.0, 6.0, 1.8, 0.0],
                 [np.inf, 0.0, 1.0, 0.0]])


def branch_cases(ort, pre):
    """name -> (surfaces [R t n], K, the K = 0 sphere the grazing rays are aimed at).  Each is traced as a Layout{Aspheric}:
    a K = 0 sphere first (COOKE_ASPHERIC), a K = 0 mirror first (REFLECTIVE with its K column), the reversed chief-ray
    layouts the preludes build for COOKE and DOUBLE_GAUSS, and a K = 0 sphere behind a plane (DEEP).  The deeper spheres
    of the real prescriptions cannot be reached near grazing: the ray meets them at a slope, or an earlier surface misses
    or reflects it."""
    P = ort.prescriptions
    CA = P.COOKE_ASPHERIC["surfaces"]
    cases = {"COOKE_ASPHERIC": (CA[:, :3], CA[:, 3], 1),
             "REFLECTIVE": (P.REFLECTIVE["surfaces"], P.REFLECTIVE["K"], 1),
             "DEEP": (DEEP[:, :3], DEEP[:, 3], 2)}
    for name in ("COOKE", "DOUBLE_GAUSS"):
        Q = getattr(P, name)
        s = pre.solve(Q["surfaces"], Q["a"], Q["h"])
        rev, Kr = P.reversed_chief_layout(Q["surfaces"], s.marginal.z[-1] - s.marginal.z[-2])
        cases["REVERSED_" + name] = (rev, Kr, 1)
    return cases


def case_rays(S, K, surf, n_random=400, seed=0):
    """(y0, U0, number of grazing rays first): the grazing rays of grazing_rays() and a random bundle over the surface"""
    yg, _ = grazing_rays(S, K, surf, seed=seed)
    rng = np.random.default_rng(seed + 1)
    amax = 0.9 * abs(float(S[surf, 0]))
    y0 = np.concatenate([yg, rng.uniform(-amax, amax, n_random)])
    U0 = np.concatenate([np.zeros(len(yg)), rng.uniform(-0.2, 0.2, n_random)])
    return y0, U0, len(yg)


# ---- independent 50-digit meridional check ----------------------------------------------------------------------------
MERIDIONAL_FIXTURES = ("COOKE", "DOUBLE_GAUSS", "DOUBLE_GAUSS_CONIC", "COOKE_ASPHERIC", "REFLECTIVE", "PARABOLA")


def meridional_fixture(ort, name):
    """(surfaces [R t n], K or None, aspheric, |y| range, |U| range) -- polynomial terms are left out: the reference's
    + p(y) at the vertex-plane height is not a geometric surface"""
    P = ort.prescriptions
    if name == "COOKE":
        return P.COOKE["surfaces"], None, False, 14.0, 0.25
    if name == "DOUBLE_GAUSS":
        return P.DOUBLE_GAUSS["surfaces"], None, False, 24.0, 0.2
    if name == "DOUBLE_GAUSS_CONIC":
        S = P.DOUBLE_GAUSS["surfaces"]
        return S, np.where(np.isfinite(S[:, 0]), -0.3, 0.0), True, 24.0, 0.2
    if name == "COOKE_ASPHERIC":
        S = P.COOKE_ASPHERIC["surfaces"]
        return S[:, :3], S[:, 3], True, 14.0, 0.25
    if name == "REFLECTIVE":
        return P.REFLECTIVE["surfaces"], P.REFLECTIVE["K"], True, 14.0, 0.1
    S = P.PARABOLA["surfaces"]
    return S[:, :3], S[:, 3], True, 30.0, 0.1


def meridional_rays(S, K, ymax, umax, n=2000, seed=0):
    """a random bundle plus rays bisected near grazing on the first surface (K = 0 or not) and rays near total internal
    reflection, when the layout has them: y0 with |y0 / R1| in [1 - 1e-5, 1 - 1e-7] at U0 = 0, and rays bisected to
    where the first failing surface turns from refracting to reflecting.  Returns (y0, U0, edge): `edge` marks the
    rays bisected to within ~1e-9 mm of a miss or TIR, whose status is checked but whose values are ill-conditioned"""
    rng = np.random.default_rng(seed)
    n_rand = n - n // 5
    y0 = list(rng.uniform(-ymax, ymax, n_rand))
    U0 = list(rng.uniform(-umax, umax, n_rand))
    R1 = abs(float(S[1, 0]))
    Kl = [0.0] * len(S) if K is None else [float(v) for v in K]
    if np.isfinite(R1):                                   # near grazing on surface 1: |y / R| = 1 - d at U = 0
        sq = math.sqrt(1.0 + Kl[1]) if 1.0 + Kl[1] > 0.0 else 1.0
        for d in 10.0 ** rng.uniform(-7, -5, n // 10):
            y0.append(float(rng.choice([-1.0, 1.0]) * R1 / sq * (1.0 - d)))
            U0.append(0.0)
    # near TIR / miss: bisect the entrance height between a ray that passes and one that fails
    R, t, nn = [float(v) for v in S[:, 0]], [float(v) for v in S[:, 1]], [float(v) for v in S[:, 2]]
    tries, n_edge = 0, len(y0)
    while len(y0) < n and tries < 50 * n:
        tries += 1
        U = float(rng.uniform(-umax, umax))
        a, b = 0.0, float(rng.choice([-1.0, 1.0])) * 3.0 * ymax
        if trace(R, t, nn, Kl, a, U, "atan_always")[3] != 0 or trace(R, t, nn, Kl, b, U, "atan_always")[3] == 0:
            continue
        for _ in range(36):                              # to ~1e-9 mm of the edge: near it, but not within rounding
            m = 0.5 * (a + b)
            if trace(R, t, nn, Kl, m, U, "atan_always")[3] == 0:
                a = m
            else:
                b = m
        y0 += [a, b]
        U0 += [U, U]
    y0, U0 = np.array(y0[:n]), np.array(U0[:n])
    return y0, U0, np.arange(len(y0)) >= n_edge


def meridional_compare(S, K, y0, U0, yt, Ut, flags, cond, edge):
    """tracer output (rows, N) tables against the independent 50-digit tracer at x = v = 0.  `cond` (N,) marks the
    well-conditioned rays, `edge` the rays next to a miss or TIR.  Returns a dict of worst errors and of the rays whose
    miss / TIR status differs (off the edge and on it)."""
    from oracle import independent_tracer as it
    worst_p = worst_u = 0.0
    n_cmp = status_off = status_edge = 0
    for i in range(len(y0)):
        dirs = []
        xs, ys, d, st = it.trace(S, y0[i], 0.0, math.tan(U0[i]), 0.0, K=K, dirs=dirs)
        if (st == "ok") != (flags[i] == 0):
            if edge[i]:
                status_edge += 1
            else:
                status_off += 1
            continue
        if st != "ok" or not cond[i]:
            continue
        py = np.array([float(a) for a in ys])
        tu = np.array([float(dd[1] / dd[2]) for dd in dirs])
        sc = max(np.max(np.abs(py)), 1.0)
        worst_p = max(worst_p, float(np.max(np.abs(py - yt[1:, i])) / sc))
        worst_u = max(worst_u, float(np.max(np.abs(tu - np.tan(Ut[1:, i])) / np.maximum(np.abs(tu), 1.0))))
        n_cmp += 1
    return dict(compared=n_cmp, max_position_err_rel=worst_p, max_tanU_err_rel=worst_u, status_differs=status_off,
                status_differs_at_edge=status_edge, edge_rays=int(np.sum(edge)))


def conditioning(trace_batch, y0, U0, rel=2.0 ** -40):
    """well-conditioned rays: moving y0 by `rel` relative moves every hit height and tan U by less than 10 x that,
    relative to the position scale (near grazing and near TIR the trace amplifies its own roundings far more)"""
    ya, Ua = trace_batch(y0, U0)[:2]
    yb, Ub = trace_batch(y0 * (1.0 + rel) + (y0 == 0.0) * rel, U0)[:2]
    with np.errstate(invalid="ignore"):
        sc = np.maximum(np.nanmax(np.abs(ya), axis=0), 1.0)
        dy = np.nanmax(np.abs(ya - yb), axis=0) / sc
        du = np.nanmax(np.abs(np.tan(Ua) - np.tan(Ub)) / np.maximum(np.abs(np.tan(Ua)), 1.0), axis=0)
    return np.isfinite(dy) & np.isfinite(du) & (dy < 10 * rel) & (du < 10 * rel)
