"""Pins the oracle's optical path length and OPD (orc_trace3d_ext, orc_opl_start, orc_grid_trace_ext) off axis against the
INDEPENDENT 50-digit tracer (oracle/independent_tracer.py: sum of |n| s over the legs in direction cosines, the start term
as a distance to the plane wavefront or the object plane, the reference-sphere closure as a ray-sphere intersection), and
checks the reference-sphere convention itself with physics: the real-ray OPD of the Cooke triplet at small fields
reproduces its Seidel W131, W222 and W220.

Precondition of every closure here: the last surface is a plane (the image plane the sweeps append).  The closure puts the
sphere's centre on that plane and ignores the ray's z offset from it, so it is exact only there."""
import math

import numpy as np
import pytest

from oracle_backend import OracleBackend
from test_oracle_independent import fixture as _fixture5

FIXTURES = ("COOKE", "DOUBLE_GAUSS", "DOUBLE_GAUSS_CONIC", "REFLECTIVE", "PARABOLA", "COOKE_ASPHERIC", "TESSAR")
REL = 1e-13          # x path length: the 50-digit OPL is exact to far below it; the oracle's is a double sum of ~10 legs
LAM = 587.5618e-6


def fixture(ort, name):
    """[R t n] rows with an image plane appended, K (or None), ray-height and slope ranges of the random rays"""
    if name not in ("COOKE_ASPHERIC", "TESSAR"):
        return _fixture5(ort, name)
    P = getattr(ort.prescriptions, name)
    S = P["surfaces"]
    ext = np.vstack([S[:, :3], [np.inf, 0.0, S[-1, 2]]])
    ext[-2, 1] = 60.0 if name == "COOKE_ASPHERIC" else 40.0
    K = np.append(S[:, 3], 0.0) if S.shape[1] > 3 else None
    return ext, K, (12.0 if name == "COOKE_ASPHERIC" else 8.0), (0.25 if name == "COOKE_ASPHERIC" else 0.2)


def dec_opl(ext, K, y, x, u, v, **kw):
    from oracle import independent_tracer as it
    L = []
    _, _, _, st = it.trace(ext, y, x, u, v, K=K, opl=L, **kw)
    return float(L[0]) if st == "ok" else float("nan")


def system_layout(ort, name):
    """(Layout, a, h) of a fixture for the host API: conic columns travel in the Layout"""
    P = ort.prescriptions
    if name == "DOUBLE_GAUSS_CONIC":
        S = P.DOUBLE_GAUSS["surfaces"]
        return ort.Layout(S, K=np.where(np.isfinite(S[:, 0]), -0.3, 0.0)), P.DOUBLE_GAUSS["a"], P.DOUBLE_GAUSS["h"]
    Q = getattr(P, name)
    return ort.Layout(Q["surfaces"]), Q["a"], Q["h"]


@pytest.mark.parametrize("name", FIXTURES)
def test_oracle_opl_of_skew_rays(orc, ort, name):
    """orc_trace3d_ext with the collimated start term of orc_opl_start (v != 0), unclosed and closed on spheres of both
    signs of rr about off-axis centres, against the 50-digit OPL: within 1e-13 of the path length"""
    ext, K, amax, umax = fixture(ort, name)
    rng = np.random.default_rng(31)
    worst, n_cmp = 0.0, 0
    for _ in range(90):
        y, x = rng.uniform(-amax, amax), rng.uniform(-amax, amax)
        u, v = rng.uniform(-umax, umax), rng.uniform(-umax, umax)
        opl0 = orc.opl_start(0, ext[0, 2], y, x, u, v)
        base = None
        for rr in (0.0, 40.0, -40.0, 55.0):
            xc, yc = rng.uniform(-6.0, 6.0), rng.uniform(-6.0, 6.0)
            *_, opl, f = orc.trace3d_ext(ext, y, x, u, v, K=K, opl0=opl0, xc=xc, yc=yc, rr=rr)
            ref = dec_opl(ext, K, y, x, u, v, xc=xc, yc=yc, rr=rr)
            if f != 0:
                break                                                  # miss / TIR: positions already pinned elsewhere
            assert np.isnan(opl) == np.isnan(ref), (name, y, x, u, v, rr, opl, ref)
            if np.isnan(ref):
                continue                                               # the line misses the sphere: NaN on both sides
            if rr == 0.0:
                base = abs(ref)
            err = abs(opl - ref) / (base + abs(rr))
            worst = max(worst, err)
            n_cmp += 1
    assert n_cmp > 200 and worst < REL, f"{name}: {n_cmp} OPLs, worst error {worst:.3g} x path length"


@pytest.mark.parametrize("name", ["COOKE", "DOUBLE_GAUSS_CONIC", "REFLECTIVE", "PARABOLA"])
def test_oracle_opl_finite_object(orc, ort, name):
    """mode 1 (object point at z0, RayBasis slopes u = tan((ybar - y) / z0), v = tan(-x / z0)): the start term is the path
    from the plane z = z0 along the ray; orc_trace3d_ext and orc_grid_trace_ext against the 50-digit OPL"""
    ext, K, amax, _ = fixture(ort, name)
    z0, ybar = -250.0, 9.0
    worst = 0.0
    ys, xs = np.linspace(0.8 * amax, -0.8 * amax, 9), np.linspace(0.0, 0.8 * amax, 5)
    g = orc.grid_trace_ext(ext, ys, xs, 1, 1e9, 0.0, mode=1, ybar=ybar, z0=z0, K=K, xc=1.0, yc=-2.0, rr=45.0, opl_ref=0.0)
    for iy, y in enumerate(ys):
        for ix, x in enumerate(xs):
            u, v = math.tan((ybar - y) / z0), math.tan(-x / z0)
            opl0 = orc.opl_start(1, ext[0, 2], y, x, u, v, z0)
            ref_open = dec_opl(ext, K, y, x, u, v, mode=1, z0=z0)
            ref = dec_opl(ext, K, y, x, u, v, mode=1, z0=z0, xc=1.0, yc=-2.0, rr=45.0)
            *_, opl, f = orc.trace3d_ext(ext, y, x, u, v, K=K, opl0=opl0)
            assert f == 0 and abs(opl - ref_open) < REL * abs(ref_open), (name, y, x, opl, ref_open)
            worst = max(worst, abs(g["opd"][iy * len(xs) + ix] - ref) / (abs(ref_open) + 45.0))
    assert worst < REL, f"{name}: worst grid OPD error {worst:.3g} x path length"


def _wavefront_case(ort, be, name, Hs, k_rays=32):
    L, a, h = system_layout(ort, name)
    s = ort.solve(L, a, h, backend=be)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, k_rays, None, False, be, "test")
    return s, p, xs, ys, flds


@pytest.mark.parametrize("name", FIXTURES)
def test_oracle_grid_opd_of_wavefront_fields(orc, ort, name):
    """orc_grid_trace_ext on exactly the field records host._wavefront_setup builds (chief ray through the stop centre,
    opd_yc, opd_radius, opl_ref) at H = 0, 0.7, 1: a subsample of the kept rays against the 50-digit OPD, and the chief
    ray's OPD is 0 to rounding.  Path length = |closed OPL| + |rr|: the closed OPL of the parabola is 0 on axis."""
    be = OracleBackend()
    Hs = (0.0, 0.7, 1.0)
    s, p, xs, ys, flds = _wavefront_case(ort, be, name, Hs)
    S, K = be.S, be.K
    assert not np.isfinite(S[-1, 0])                                   # the closure's precondition: a plane last surface
    rng = np.random.default_rng(33)
    worst = 0.0
    y_c = ort.host.aim_rays(s.layout, -p["u"] * p["EP_t"], p["U"], np.zeros(len(Hs)), p["stop"], p["a_stop"], backend=be)
    for j, f in enumerate(flds):
        kw = dict(xc=0.0, yc=f["opd_yc"], rr=f["opd_radius"])
        g = orc.grid_trace_ext(S, ys[j], xs, p["stop"], p["a_stop"], f["h_prime"], u=f["u"], v=0.0, K=K,
                               opl_ref=f["opl_ref"], **kw)
        kept = np.flatnonzero(g["mask"])
        assert len(kept) > 0.5 * len(g["mask"])
        for idx in rng.choice(kept, size=min(100, len(kept)), replace=False):
            y, x = ys[j][idx // len(xs)], xs[idx % len(xs)]
            ref = dec_opl(S, K, y, x, f["u"], 0.0, **kw)
            worst = max(worst, abs(g["opd"][idx] - (ref - f["opl_ref"])) / (abs(ref) + abs(f["opd_radius"])))
        chief = dec_opl(S, K, y_c[j], 0.0, f["u"], 0.0, **kw)
        assert abs(chief - f["opl_ref"]) < REL * (abs(chief) + abs(f["opd_radius"])), (name, Hs[j], chief - f["opl_ref"])
    assert worst < REL, f"{name}: worst OPD error {worst:.3g} x path length"


# ---- physics: the reference sphere reproduces the Seidel field aberrations ------------------------------------------
def field_fit(ws, es):
    """least-squares fit of each field's OPD map in stop coordinates (px, py) = rho (sin, cos) of the meridional angle,
    through fifth order in the pupil (rho^5 cos, rho^4 cos^2 ...) -> (n_fields, 12) coefficients:
    [1, rho cos, rho^2, rho^2 cos^2, rho^4, rho^3 cos, rho^6, rho^5 cos, rho^4 cos^2, rho^8, rho^7 cos, rho^3 cos^3]"""
    C = []
    for w, e in zip(ws, es):
        n = len(w.opd) // 2
        assert len(e.x) == len(w.opd) and np.array_equal(e.x, w.x)       # same kept rays, same order
        rho, th = e.r[:n], e.t[:n]
        py, px = rho * np.sin(th), rho * np.cos(th)                      # theta = atan(y_s, x_s): py is the meridional
        r2 = px ** 2 + py ** 2
        A = np.column_stack([np.ones(n), py, r2, py ** 2, r2 ** 2, py * r2, r2 ** 3, py * r2 ** 2, py ** 2 * r2, r2 ** 4,
                             py * r2 ** 3, py ** 3])
        C.append(np.linalg.lstsq(A, w.opd[:n], rcond=None)[0])
    return np.array(C)


def seidel_from_fit(C, Hs, field_sign):
    """the H-dependence of the fitted coefficients, with the field sign of Aberration.__call__ (H -> H field_sign):
    rho^3 cos = W131 H + O(H^3), rho^2 cos^2 = W222 H^2 + O(H^4), rho^2 = W020 + W220 H^2 + O(H^4), rho cos = W111 H + ..."""
    Hf = np.asarray(Hs) * field_sign
    w131 = np.linalg.lstsq(np.column_stack([Hf, Hf ** 3]), C[:, 5], rcond=None)[0][0]
    w222 = np.linalg.lstsq(np.column_stack([Hf ** 2, Hf ** 4]), C[:, 3], rcond=None)[0][0]
    w020, w220, _ = np.linalg.lstsq(np.column_stack([np.ones(len(Hf)), Hf ** 2, Hf ** 4]), C[:, 2], rcond=None)[0]
    return dict(W131=w131, W222=w222, W220=w220, W020=w020, tilt=np.max(np.abs(C[:, 1] / Hf)))


PHYSICS_HS = (0.05, 0.1, 0.15, 0.2)


def check_seidel(fit, ab):
    """third-order theory against real rays.  Measured on the Cooke triplet, k_rays = 64: W131 0.947, W222 0.970,
    W220 0.967 (W040 on axis 0.981); the 5 % of coma is the fifth-order pupil terms the Seidel sum leaves out, so it gets
    0.07 and the field-curvature terms 0.05.  A reference sphere of the wrong radius adds defocus (W020, exactly 0 at the
    paraxial focus), a centre off the chief ray's image point adds tilt (rho cos; the Seidel W111 is 0 here)."""
    r131, r222, r220 = fit["W131"] / ab.W131, fit["W222"] / ab.W222, fit["W220"] / ab.W220
    msg = f"W131 {r131:.4f}, W222 {r222:.4f}, W220 {r220:.4f}, W020 {fit['W020']:.3g}, tilt {fit['tilt']:.3g}"
    assert abs(r131 - 1) < 0.07 and abs(r222 - 1) < 0.05 and abs(r220 - 1) < 0.05, msg
    assert ab.W020 == 0.0 and ab.W111 == 0.0 and abs(fit["W020"]) < 0.1 and fit["tilt"] < 0.05, msg
    return msg


def test_off_axis_seidel_terms_of_the_real_ray_opd(ort):
    """the real-ray OPD of COOKE at H = 0.05 .. 0.2 on the oracle backend reproduces W131, W222 and W220 of aberrations()"""
    be = OracleBackend()
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=be)
    ab = ort.aberrations(s.layout, s, backend=be)
    ws = ort.wavefront(s.layout, s, PHYSICS_HS, 64, backend=be)
    es = [ort.full_trace(s, H, 64, backend=be) for H in PHYSICS_HS]
    check_seidel(seidel_from_fit(field_fit(ws, es), PHYSICS_HS, ab.field_sign), ab)
