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
"""
from decimal import Decimal, getcontext

getcontext().prec = 50
D = Decimal
ZERO, ONE, TWO = D(0), D(1), D(2)


def _dec(x):
    return D(repr(float(x))) if not isinstance(x, Decimal) else x          # exact: repr(float) round-trips


def trace(surfaces, y, x, u, v, K=None, dirs=None):
    """surfaces: rows x 3 [R t n] (row 0 = object space, as the reference's Layout); slopes u = tan U, v = tan V.
    -> (xs, ys, d, status): hit coordinates at surfaces 1 .. rows-1, final direction, "ok" | "miss" | "tir".
    dirs, if a list, receives the unit direction after every surface traced."""
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
                    return xs, ys, d, "miss"
                sq = disc.sqrt()
                roots = [(-B + sq) / A, (-B - sq) / A]
                s = min(roots, key=lambda r: abs(Z + r * d[2]))          # the sheet through the vertex
            grad = None
        P = [P[0] + s * d[0], P[1] + s * d[1], P[2] + s * d[2]]
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
                return xs, ys, d, "tir"
            gco = mu * cosI - rad.sqrt()
            d = [mu * d[j] + gco * N[j] for j in range(3)]
        l = (d[0] * d[0] + d[1] * d[1] + d[2] * d[2]).sqrt()
        d = [a / l for a in d]
        if dirs is not None:
            dirs.append(d)
    return xs, ys, d, "ok"
