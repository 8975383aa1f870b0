"""An INDEPENDENT 50-digit skew-ray tracer -- test infrastructure, used only to pin oracle/ort_oracle.c off the meridional
plane (VERDICT r1: the reference's own tests pin the x != 0 arithmetic of src/PupilSampling.jl:1-65 only to +-0.07 RMS,
and orc_trace3d_ld is the same formulas in 80 bits).

Nothing here is derived from the reference's sag / tilt / refract! formulas.  It is textbook vector geometry in global
coordinates, evaluated with decimal.Decimal at 50 significant digits:

  ray        P + s d, d a unit vector (the reference parametrises by slopes u = dy/dz, v = dx/dz)
  surface    the conicoid  c (X^2 + Y^2 + (1 + K) Z^2) - 2 Z = 0  about its vertex (c = 1/R; a plane for c = 0)
  hit        the quadratic  A s^2 + 2 B s + C = 0,  A = c (dx^2 + dy^2 + (1+K) dz^2),  B = c (X dx + Y dy + (1+K) Z dz) - dz,
             C = c (X^2 + Y^2 + (1+K) Z^2) - 2 Z;  of its two roots the hit on the sheet through the vertex (smaller |Z|)
  normal     the gradient (c X, c Y, c (1+K) Z - 1), normalised, turned against the incoming ray
  Snell      d' = mu d + (mu cos I - sqrt(1 - mu^2 (1 - cos^2 I))) N,  mu = |n1| / |n2|        (vector form)
  mirror     d' = d + 2 cos I N          (the reference marks a mirror by n2 = -n1, test/runtests.jl:376-387)

trace() returns the (x, y) hit coordinates at every surface and the final unit direction, as Decimals; a missed surface or
total internal reflection ends the trace (status "miss" / "tir").

Optical path length (opl=[] asks for it; the OPL is appended to that list, NaN when the ray ends early or its line misses
the reference sphere):

  legs       sum over legs of |n_i| s_i, s_i the SIGNED parameter along the unit direction (a ray starting behind the sag of
             the first surface has a negative first leg)
  start      collimated (mode 0): n0 (x d_x + y d_y), the lead of the start point (x, y, 0) over the plane wavefront through
             the origin; finite object (mode 1): the path from the plane z = z0 to the start point along the ray,
             n0 (0 - z0) / d_z.  The caller's slopes define the ray, so it passes through the object point only as closely
             as tan((ybar - y) / z0) does.
  closure    rr != 0: the ray is continued from its last hit P to the point at distance |rr| from the centre
             C = (xc, yc, z_last), z_last the vertex of the last surface: |P + s d - C| = |rr|, of the roots
             s = -b -+ sqrt(b^2 - (|q|^2 - rr^2)),  q = P - C, b = q.d,  the one with sign  -sgn(rr) sgn(n_last)  on the root,
             and |n_last| s is added.  In a positive medium a positive rr closes on the sheet behind the ray (towards the
             exit pupil), a negative rr on the sheet ahead of it; a negative (reflected) medium reverses both.
             C lies on the last surface's vertex plane, so the closure is exact only when the last surface is a plane
             (the image plane every sweep appends): the ray's last hit is then in the plane of C.
"""
from decimal import Decimal, getcontext

getcontext().prec = 50
D = Decimal
ZERO, ONE, TWO = D(0), D(1), D(2)


def _dec(x):
    return D(repr(float(x))) if not isinstance(x, Decimal) else x          # exact: repr(float) round-trips


def trace(surfaces, y, x, u, v, K=None, dirs=None, opl=None, mode=0, z0=0.0, xc=0.0, yc=0.0, rr=0.0):
    """surfaces: rows x 3 [R t n] (row 0 = object space, as the reference's Layout); slopes u = tan U, v = tan V.
    -> (xs, ys, d, status): hit coordinates at surfaces 1 .. rows-1, final direction, "ok" | "miss" | "tir".
    dirs, if a list, receives the unit direction after every surface traced.  opl, if a list, receives the optical path
    length (module docstring): start term of `mode` (z0 for mode 1), legs, and the closure on the sphere of radius rr
    about (xc, yc, z_last) if rr != 0."""
    rows = len(surfaces)
    R = [float(r[0]) for r in surfaces]
    t = [float(r[1]) for r in surfaces]
    n = [float(r[2]) for r in surfaces]
    Kc = [0.0] * rows if K is None else [float(k) for k in K]
    u, v = _dec(u), _dec(v)
    nrm = (u * u + v * v + ONE).sqrt()
    d = [v / nrm, u / nrm, ONE / nrm]                    # (dx, dy, dz)
    P = [_dec(x), _dec(y), ZERO]                         # global; the reference starts on the object-space row's plane
    zv = ZERO                                            # vertex of the current row
    xs, ys = [], []
    n0 = _dec(abs(n[0]))
    path = n0 * (-_dec(z0)) / d[2] if mode == 1 else n0 * (P[0] * d[0] + P[1] * d[1])
    for i in range(rows - 1):
        t_i = t[i]
        zv = zv + (_dec(t_i) if t_i == t_i and abs(t_i) != float("inf") else ZERO)      # vertex of row i + 1
        Ri, Ki = R[i + 1], _dec(Kc[i + 1])
        X, Y, Z = P[0], P[1], P[2] - zv
        if abs(Ri) == float("inf"):                      # plane Z = 0
            s = -Z / d[2]
            grad = [ZERO, ZERO, -ONE]
        else:
            c = ONE / _dec(Ri)
            q = ONE + Ki
            A = c * (d[0] * d[0] + d[1] * d[1] + q * d[2] * d[2])
            B = c * (X * d[0] + Y * d[1] + q * Z * d[2]) - d[2]
            Cc = c * (X * X + Y * Y + q * Z * Z) - TWO * Z
            if A == 0:
                s = -Cc / (TWO * B)
            else:
                disc = B * B - A * Cc
                if disc < 0:
                    return _end(opl, xs, ys, d, "miss")
                sq = disc.sqrt()
                roots = [(-B + sq) / A, (-B - sq) / A]
                s = min(roots, key=lambda r: abs(Z + r * d[2]))          # the sheet through the vertex
            grad = None
        P = [P[0] + s * d[0], P[1] + s * d[1], P[2] + s * d[2]]
        path += _dec(abs(n[i])) * s
        xs.append(P[0]); ys.append(P[1])
        if grad is None:
            Zh = P[2] - zv
            grad = [c * P[0], c * P[1], c * (ONE + Ki) * Zh - ONE]
        g = (grad[0] * grad[0] + grad[1] * grad[1] + grad[2] * grad[2]).sqrt()
        N = [grad[0] / g, grad[1] / g, grad[2] / g]
        cosI = -(d[0] * N[0] + d[1] * N[1] + d[2] * N[2])
        if cosI < 0:
            N = [-a for a in N]; cosI = -cosI
        n1, n2 = n[i], n[i + 1]
        if (n1 < 0) != (n2 < 0):                          # mirror
            d = [d[j] + TWO * cosI * N[j] for j in range(3)]
        elif n1 != n2:
            mu = _dec(abs(n1)) / _dec(abs(n2))
            rad = ONE - mu * mu * (ONE - cosI * cosI)
            if rad < 0:
                return _end(opl, xs, ys, d, "tir")
            gco = mu * cosI - rad.sqrt()
            d = [mu * d[j] + gco * N[j] for j in range(3)]
        l = (d[0] * d[0] + d[1] * d[1] + d[2] * d[2]).sqrt()
        d = [a / l for a in d]
        if dirs is not None:
            dirs.append(d)
    if opl is not None:
        rr = _dec(rr)
        if rr != 0:
            q = [P[0] - _dec(xc), P[1] - _dec(yc), P[2] - zv]
            b = q[0] * d[0] + q[1] * d[1] + q[2] * d[2]
            disc = b * b - (q[0] * q[0] + q[1] * q[1] + q[2] * q[2] - rr * rr)
            if disc < 0:                                 # the line misses the sphere: no closed path
                opl.append(D("NaN"))
                return xs, ys, d, "ok"
            sgn = (1 if rr > 0 else -1) * (1 if n[-1] > 0 else -1)
            path += _dec(abs(n[-1])) * (-b - sgn * disc.sqrt())
        opl.append(path)
    return xs, ys, d, "ok"


def _end(opl, xs, ys, d, status):
    if opl is not None:
        opl.append(D("NaN"))
    return xs, ys, d, status
