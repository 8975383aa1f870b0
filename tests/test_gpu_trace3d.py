"""GPU parity of the 3-D skew tracer (K1 grid sweep, arbitrary rays, candidates) against the CPU
oracle, called through the C ABI.  STRICT must be bit-identical (positions, mask, flags); FAST
within 1e-12 relative (north_star tolerance) with mask and flags bit-identical."""
import math

import numpy as np
import pytest

from util import abs_rel_err, bits_equal, n_bits_differ, relerr

pytestmark = pytest.mark.gpu

TOL = 1e-12   # north_star: positions, direction cosines, OPD within 1e-12 relative in Float64


def _inputs(pre, ort, name, H, k_rays=64):
    P = getattr(ort.prescriptions, name)
    sysm = pre.solve(P["surfaces"], P["a"], P["h"])
    return sysm, pre.full_trace_inputs(sysm, H, k_rays)


def _oracle_grid(orc, p):
    return orc.grid_trace(p.ext, p.ys, p.xs, p.stop, p.a_stop, p.h_prime, u=p.u, v=p.v, K=p.K)


@pytest.mark.parametrize("name,H", [("COOKE", 0.0), ("COOKE", 0.7), ("COOKE", 1.0),
                                    ("SINGLET", 0.7), ("DOUBLE_GAUSS", 0.5), ("TESSAR", 1.0)])
def test_grid_strict_bit_exact(ctx, orc, pre, ort, name, H):
    _, p = _inputs(pre, ort, name, H)
    g = _oracle_grid(orc, p)
    ctx.set_layout(p.ext, p.K)
    r = ctx.trace3d_grid([dict(u=p.u, v=p.v, h_prime=p.h_prime)], p.ys, p.xs, p.stop, p.a_stop,
                         arith=ort.STRICT, want=("ex", "ey", "r", "theta", "mask", "flags", "stats"))
    assert np.array_equal(r["mask"][0], g["mask"])
    assert np.array_equal(r["flags"][0], g["flags"])
    assert bits_equal(r["ex"][0], g["ex"])
    assert bits_equal(r["ey"][0], g["ey"])
    assert bits_equal(r["r"][0], g["r"])
    assert relerr(r["theta"][0], g["theta"]) < TOL      # atan2: CUDA libm vs glibc
    assert int(r["stats"]["n_kept"][0]) == g["n_kept"]


@pytest.mark.parametrize("name,H", [("COOKE", 0.0), ("COOKE", 0.7), ("COOKE", 1.0),
                                    ("SINGLET", 1.0), ("DOUBLE_GAUSS", 0.0), ("DOUBLE_GAUSS", 1.0),
                                    ("TESSAR", 0.7)])
def test_grid_fast_within_tolerance_mask_exact(ctx, orc, pre, ort, name, H):
    _, p = _inputs(pre, ort, name, H)
    g = _oracle_grid(orc, p)
    ctx.set_layout(p.ext, p.K)
    r = ctx.trace3d_grid([dict(u=p.u, v=p.v, h_prime=p.h_prime)], p.ys, p.xs, p.stop, p.a_stop,
                         arith=ort.FAST, want=("ex", "ey", "r", "theta", "mask", "flags", "stats"))
    assert np.array_equal(r["mask"][0], g["mask"]), "clip mask must be bit-exact in FAST mode too"
    assert np.array_equal(r["flags"][0], g["flags"])
    scale = max(abs(p.h_prime), p.y_EP)          # positions at the image plane are O(h', y_EP)
    # ex = xf is a position; ey = yf - h' is a difference of positions: error relative to position scale
    assert abs_rel_err(r["ex"][0], g["ex"], scale) < TOL
    assert abs_rel_err(r["ey"][0], g["ey"], scale) < TOL
    assert relerr(r["r"][0], g["r"]) < TOL or abs_rel_err(r["r"][0], g["r"], p.a_stop) < TOL
    m = g["mask"].astype(bool)
    assert abs_rel_err(r["theta"][0][m], g["theta"][m], math.pi) < 1e-11
    # the lean instantiation (exactly ex, ey, mask wanted) computes the same bits as the generic one
    rl = ctx.trace3d_grid([dict(u=p.u, v=p.v, h_prime=p.h_prime)], p.ys, p.xs, p.stop, p.a_stop,
                          arith=ort.FAST, want=("ex", "ey", "mask", "stats"))
    assert n_bits_differ(rl["ex"], r["ex"]) == 0 and n_bits_differ(rl["ey"], r["ey"]) == 0
    assert np.array_equal(rl["mask"], r["mask"]) and rl["stats"].tobytes() == r["stats"].tobytes()
    ro = ctx.trace3d_grid([dict(u=p.u, v=p.v, h_prime=p.h_prime)], p.ys, p.xs, p.stop, p.a_stop,
                          arith=ort.FAST, want=("stats",))                      # statistics-only instantiation
    assert ro["stats"].tobytes() == r["stats"].tobytes()


def test_grid_multi_field_compact_and_stats(ctx, orc, pre, ort):
    """Config 1: Cooke triplet, 64x64 grid (64 x 32 half pupil), 3 fields, spot RMS."""
    P = ort.prescriptions.COOKE
    sysm = pre.solve(P["surfaces"], P["a"], P["h"])
    Hs = (0.0, 0.7, 1.0)
    ps = [pre.full_trace_inputs(sysm, H, 64) for H in Hs]
    for arith in (ort.STRICT, ort.FAST):
        for p, H in zip(ps, Hs):
            g = _oracle_grid(orc, p)
            ref = pre.full_trace(sysm, H, 64)
            ctx.set_layout(p.ext, p.K)
            nu = sysm.marginal.nu[-1]
            r = ctx.trace3d_grid([dict(u=p.u, v=p.v, h_prime=p.h_prime)], p.ys, p.xs, p.stop, p.a_stop,
                                 arith=arith, compact=True,
                                 want=("ex", "ey", "r", "theta", "wx", "wy", "mask", "stats"),
                                 wavegrad=(nu, 587.5618e-6))
            st = r["stats"][0]
            n = int(st["n_kept"])
            assert n == g["n_kept"]
            m = g["mask"].astype(bool)
            scale = max(abs(p.h_prime), p.y_EP)
            for key in ("ex", "ey", "r"):
                assert abs_rel_err(r[key][0][:n], g[key][m], scale) < TOL, key
            assert abs_rel_err(r["theta"][0][:n], g["theta"][m], math.pi) < 1e-11
            # wavegrad (src/PupilSampling.jl:165-167)
            wx = orc.wavegrad(g["ex"][m], nu)
            assert abs_rel_err(r["wx"][0][:n], wx, scale * abs(nu) / 587.5618e-6) < TOL
            # statistics: mirrored RMS of the reference (:139-146,169-173) from the mergeable moments
            sxx = st["m2_x"] + n * st["mean_x"] ** 2          # mirrored x: mean 0, sum sq doubles
            rms = math.sqrt((2 * sxx + 2 * st["m2_y"]) / (2 * n))
            # STRICT: eps is bit-identical, only the summation order differs -> 1e-12 relative.
            # FAST: eps = yf - h' is a ~0.03 mm difference of ~20 mm positions that are themselves
            # good to 1e-12 relative, so the RMS is good to 1e-12 x the position scale (absolute).
            if arith == ort.STRICT:
                assert abs(rms / ref.RMS - 1) < TOL
            assert abs(rms - ref.RMS) < TOL * scale
            assert abs(st["r_max"] / g["r"][m].max() - 1) < TOL


def test_grid_edge_cases(ctx, orc, pre, ort):
    P = ort.prescriptions.COOKE
    sysm = pre.solve(P["surfaces"], P["a"], P["h"])
    p = pre.full_trace_inputs(sysm, 0.7, 64)
    ctx.set_layout(p.ext, p.K)
    fld = [dict(u=p.u, v=p.v, h_prime=p.h_prime)]
    # empty grid
    r = ctx.trace3d_grid(fld, np.zeros(0), p.xs, p.stop, p.a_stop)
    assert int(r["stats"]["n_kept"][0]) == 0 and r["ex"].shape == (1, 0)
    # ragged: sizes that are not multiples of the 256-ray tile, 1 x 1 grid, rays that miss / clip
    for ys, xs in [(p.ys[:1], p.xs[:1]), (p.ys[:7], p.xs[:13]), (np.linspace(-60, 60, 33), np.linspace(0, 60, 17))]:
        g = orc.grid_trace(p.ext, ys, xs, p.stop, p.a_stop, p.h_prime, u=p.u, v=p.v, K=p.K)
        for arith in (ort.STRICT, ort.FAST):
            r = ctx.trace3d_grid(fld, ys, xs, p.stop, p.a_stop, arith=arith, want=("ex", "ey", "mask", "flags", "stats"))
            assert np.array_equal(r["mask"][0], g["mask"])
            assert np.array_equal(r["flags"][0], g["flags"])
            assert int(r["stats"]["n_kept"][0]) == g["n_kept"]
            if arith == ort.STRICT:
                assert bits_equal(r["ex"][0], g["ex"]) and bits_equal(r["ey"][0], g["ey"])
            else:
                assert abs_rel_err(r["ex"][0], g["ex"], 25.0) < TOL
                assert abs_rel_err(r["ey"][0], g["ey"], 25.0) < TOL
    # NaN coordinates propagate as NaN and are dropped
    ys = p.ys[:4].copy(); ys[2] = np.nan
    g = orc.grid_trace(p.ext, ys, p.xs[:4], p.stop, p.a_stop, p.h_prime, u=p.u, v=p.v, K=p.K)
    for arith in (ort.STRICT, ort.FAST):
        r = ctx.trace3d_grid(fld, ys, p.xs[:4], p.stop, p.a_stop, arith=arith, want=("ex", "ey", "mask", "flags", "stats"))
        assert np.array_equal(r["mask"][0], g["mask"])
        assert np.array_equal(np.isnan(r["ex"][0]), np.isnan(g["ex"]))


def test_strict_exact_paths_adversarial(ctx, orc, ort):
    """k_grid<STRICT> takes divisions and square roots from xdiv / xsqrt (flag + per-ray re-trace with the intrinsics) and
    planes from an exact shortcut.  Operands chosen to sit on every seam: the x = 0 column and y = 0 row (zero numerators),
    -0.0, denormal / tiny / huge coordinates (|x| >= 1e150 leaves the plane shortcut; 1e200 overflows r^2), NaN and Inf
    coordinates, rays that miss a surface and then meet the planes, planes at both ends and in the middle, a plane with
    K != 0, a plane with polynomial terms (its tilt keeps dp_dy), R = -Inf.  Everything bit-identical to the CPU oracle."""
    inf = np.inf
    S = np.array([[inf, 0.0, 1.0], [inf, 3.0, 1.5], [40.0, 2.0, 1.0], [-inf, 4.0, 1.6], [-35.0, 3.0, 1.0],
                  [inf, 5.0, 1.0], [60.0, 2.0, 1.7], [inf, 30.0, 1.0], [inf, 0.0, 1.0]])
    K = np.array([0.0, 0.3, -0.5, -1.7, 0.2, 0.0, 0.0, 2.0, 0.0])
    xs = np.array([0.0, -0.0, 5e-324, 1e-310, 1e-200, 1e-30, 0.3, 2.0, 7.5, 11.0, 38.0, 41.0, 1e3, 1e149, 1e150, 1e160, 1e200,
                   inf, np.nan])
    ys = np.concatenate([-xs[::-1], xs])
    stop = 5
    for u, v in ((0.0, 0.0), (0.05, 0.0), (-0.03, 0.02)):
        fld = [dict(u=u, v=v, h_prime=0.25)]
        for poly in (None, "plane+curved"):
            P = None
            if poly:
                P = np.zeros((S.shape[0], 7)); P[3, 4] = 2e-6; P[3, 3] = -1e-5; P[2, 6] = 1e-9; P[7, 2] = 1e-4
            try:
                orc.set_poly(P)
                g = orc.grid_trace(S, ys, xs, stop, 9.0, 0.25, u=u, v=v, K=K)
            finally:
                orc.set_poly(None)
            ctx.set_layout(S, K); ctx.set_polynomials(P)
            with np.errstate(all="ignore"):
                r = ctx.trace3d_grid(fld, ys, xs, stop, 9.0, arith=ort.STRICT, want=("ex", "ey", "r", "theta", "mask", "flags", "stats"))
            assert np.array_equal(r["mask"][0], g["mask"]) and np.array_equal(r["flags"][0], g["flags"]), (u, v, poly)
            for k in ("ex", "ey", "r"):
                assert bits_equal(r[k][0], g[k]), (u, v, poly, k)
            assert np.array_equal(np.isnan(r["theta"][0]), np.isnan(g["theta"]))      # atan2: CUDA vs glibc, last ulp
            m = g["mask"].astype(bool)
            assert abs_rel_err(r["theta"][0][m], g["theta"][m], math.pi) < 1e-11
            assert int(r["stats"]["n_kept"][0]) == g["n_kept"] and g["n_kept"] > 20
            # the single-ray kernel (library intrinsics + the same plane shortcut) on the same rays
            yy, xx = np.meshgrid(ys, xs, indexing="ij")
            N = yy.size
            xo, yo, ko, fo = orc_rays(orc, S, yy.ravel(), xx.ravel(), u, v, K, P)
            with np.errstate(all="ignore"):
                xr, yr, kr, fr = ctx.trace3d_rays(yy.ravel(), xx.ravel(), np.full(N, u), np.full(N, v), arith=ort.STRICT)
            assert np.array_equal(fr, fo)
            assert n_bits_differ(xr, xo) == 0 and n_bits_differ(yr, yo) == 0 and n_bits_differ(kr, ko) == 0
    ctx.set_polynomials(None)


def orc_rays(orc, S, y0, x0, u, v, K, P):
    try:
        orc.set_poly(P)
        with np.errstate(all="ignore"):
            return orc.trace3d_batch(S, y0, x0, np.full(y0.size, u), np.full(y0.size, v), K=K)
    finally:
        orc.set_poly(None)


def test_grid_point_mode_raybasis(ctx, orc, pre, ort):
    """RayBasis mode (src/PupilSampling.jl:124-127): per-ray slopes through tan()."""
    P = ort.prescriptions.COOKE
    sysm = pre.solve(P["surfaces"], P["a"], P["h"])
    p = pre.full_trace_inputs(sysm, 0.0, 32)
    z0, ybar = -500.0, 12.0
    g = orc.grid_trace(p.ext, p.ys, p.xs, p.stop, p.a_stop, 0.3, mode=1, ybar=ybar, z0=z0, K=p.K)
    ctx.set_layout(p.ext, p.K)
    for arith in (ort.STRICT, ort.FAST):
        r = ctx.trace3d_grid([dict(mode=1, ybar=ybar, z0=z0, h_prime=0.3)], p.ys, p.xs, p.stop, p.a_stop,
                             arith=arith, want=("ex", "ey", "mask", "flags", "stats"))
        assert np.array_equal(r["mask"][0], g["mask"])
        assert abs_rel_err(r["ex"][0], g["ex"], 25.0) < TOL     # CUDA tan vs glibc tan: <= 2 ulp
        assert abs_rel_err(r["ey"][0], g["ey"], 25.0) < TOL


@pytest.mark.parametrize("name", ["COOKE", "DOUBLE_GAUSS", "REFLECTIVE", "PARABOLA"])
def test_rays_all_surfaces(ctx, orc, ort, name):
    """raytrace(surfaces, y, x, U, V, Vector{RealRay}): every surface, direction cosines, flags."""
    P = getattr(ort.prescriptions, name)
    S = P["surfaces"]
    amax = float(P["a"][0])
    rng = np.random.default_rng(11)
    N = 5000
    y0 = rng.uniform(-1.3 * amax, 1.3 * amax, N)     # beyond the aperture: some rays miss
    x0 = rng.uniform(-1.3 * amax, 1.3 * amax, N)
    u0 = rng.uniform(-0.3, 0.3, N)
    v0 = rng.uniform(-0.3, 0.3, N)
    y0[:4] = [0.0, 1.0, 0.0, amax]; x0[:4] = 0.0; u0[:4] = 0.0; v0[:4] = 0.0     # on-axis rays
    K = S[:, 3] if S.shape[1] > 3 else None
    xo, yo, ko, fo = orc.trace3d_batch(S[:, :3], y0, x0, u0, v0, K=K)
    ctx.set_layout(S[:, :3], K)
    xs, ys, ks, fs = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.STRICT)
    assert np.array_equal(fs, fo)
    assert n_bits_differ(xs, xo) == 0 and n_bits_differ(ys, yo) == 0 and n_bits_differ(ks, ko) == 0
    xf, yf, kf, ff = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.FAST)
    assert np.array_equal(ff, fo)
    with np.errstate(all="ignore"):
        scale = np.maximum(np.nan_to_num(np.nanmax(np.abs(np.stack([xo, yo])), axis=(0, 1)), nan=1.0), 1.0)
    assert np.array_equal(np.isnan(xf), np.isnan(xo)) and np.array_equal(np.isnan(yf), np.isnan(yo))

    def err(a, b):      # per-ray max over surfaces of |a - b| / position scale
        with np.errstate(all="ignore"):
            return np.nan_to_num(np.nanmax(np.abs(a - b), axis=0), nan=0.0) / scale

    # These rays are deliberately wild (1.3 x aperture, slopes to 0.3): some graze a surface and are
    # ill-conditioned -- the reference's own Float64 result is then uncertain at the 1e-12 level.
    # Conditioning is measured against an 80-bit evaluation of the same formulas.
    xl, yl, kl = orc.trace3d_ld_batch(S[:, :3], y0, x0, u0, v0, K=K)
    cond = np.maximum(err(xo, xl), err(yo, yl))              # strict (= reference arithmetic) vs truth
    e_fast = np.maximum(err(xf, xo), err(yf, yo))            # fast vs reference arithmetic
    e_true = np.maximum(err(xf, xl), err(yf, yl))            # fast vs truth
    well = cond < 1e-13
    assert well.mean() > 0.99
    assert e_fast[well].max() < TOL
    assert np.all(e_true <= TOL / 2 + 2 * cond), "FAST must be as accurate as the reference arithmetic"
    ok = ((fo & ort.FLAG_MISS) == 0) & well
    assert np.max(np.abs(kf[:, ok] - ko[:, ok])) < TOL        # direction cosines are O(1)


def test_three_d_equals_two_d(ctx, orc, ort):
    """test/runtests.jl:355-358, 376-387: the 3-D tracer reproduces the 2-D tracer on meridional rays."""
    for name in ("COOKE", "REFLECTIVE"):
        S = getattr(ort.prescriptions, name)["surfaces"]
        ctx.set_layout(S)
        y0 = np.array([15.0 if name == "REFLECTIVE" else 14.6, 5.0, 1.0])
        U0 = np.array([0.0, 0.05, -0.02])
        y2, U2, ts, f2 = ctx.trace2d_batch(y0, U0)
        xv, yv, k, f3 = ctx.trace3d_rays(y0, np.zeros(3), np.tan(U0), np.zeros(3), arith=ort.STRICT)
        assert np.allclose(yv, y2[1:], rtol=1e-13, atol=1e-13)
        assert np.all(xv == 0.0)


class _NoAimFields:
    """proxy that hides aim_fields so the host runs its own prelude (solve-consistent secant loops, several launches)"""

    def __init__(self, ctx):
        self._c = ctx

    def __getattr__(self, name):
        if name == "aim_fields":
            raise AttributeError(name)
        return getattr(self._c, name)


@pytest.mark.parametrize("name", ["COOKE", "DOUBLE_GAUSS", "TESSAR", "SINGLET", "COOKE_ASPHERIC"])
def test_one_call_prelude_equals_host_prelude(ctx, ort, name):
    """ort_aim_fields (the whole full_trace prelude of a field sweep in one call) against the host prelude that drives
    k_paraxial / k_aim2d / k_trace2d step by step: the same device arithmetic, so the aimed quantities agree to the last
    bits, and the spot they lead to is the same"""
    P = getattr(ort.prescriptions, name)
    system = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = [0.0, 0.5, 1.0]
    pa = ort.host._full_trace_setup(system.layout, system, Hs, 64, None, ctx)
    pb = ort.host._full_trace_setup(system.layout, system, Hs, 64, None, _NoAimFields(ctx))
    for k in ("y1", "y2", "u", "U", "h_prime"):
        assert np.max(np.abs(pa[k] - pb[k]) / np.maximum(np.abs(pb[k]), 1.0)) < 1e-14, k
    for k in ("y_EP", "EP_t", "focus", "a_stop", "nu"):
        assert abs(pa[k] - pb[k]) <= 1e-14 * max(abs(pb[k]), 1.0), k
    assert pa["stop"] == pb["stop"] and np.array_equal(pa["ext"], pb["ext"])
    ea = ort.full_trace_fields(system.layout, system, Hs, 64, backend=ctx)
    eb = ort.full_trace_fields(system.layout, system, Hs, 64, backend=_NoAimFields(ctx))
    scale = max(np.max(np.abs(pb["h_prime"])), pb["y_EP"])
    for j, (a, b) in enumerate(zip(ea, eb)):
        ya, yb = ort.host.jl_range(pa["y1"][j], pa["y2"][j], 64), ort.host.jl_range(pb["y1"][j], pb["y2"][j], 64)
        ka, kb = _kept_mask(ctx, ort, pa, j, ya), _kept_mask(ctx, ort, pb, j, yb)
        rim = np.zeros_like(ka)
        rim[[0, 63], :] = True                                       # the two rim rays (y1, y2) of every x column
        assert not np.any((ka != kb) & ~rim)                          # masks differ at most on the rim rays
        common = (ka & kb).reshape(-1)
        sa, sb = _spot(ctx, ort, pa, j, ya), _spot(ctx, ort, pb, j, yb)
        for q in range(2):
            assert np.max(np.abs(sa[q][common] - sb[q][common])) <= 1e-12 * scale
        ra, rb = (np.sqrt(np.mean(sa[0][common] ** 2 + (sa[1][common] - sa[1][common].mean()) ** 2)),
                  np.sqrt(np.mean(sb[0][common] ** 2 + (sb[1][common] - sb[1][common].mean()) ** 2)))
        assert abs(ra / rb - 1) <= 1e-12
        assert abs(len(a.x) - len(b.x)) <= 4 and np.all(np.isfinite([a.RMS, b.RMS]))


def _grid(ctx, ort, p, j, ys, want):
    ctx.set_layout(p["ext"], p["K"])
    xs = ort.host.jl_range(0.0, p["y_EP"], 32)
    return ctx.trace3d_grid([dict(u=p["u"][j], v=0.0, h_prime=p["h_prime"][j])], ys, xs, p["stop"], p["a_stop"],
                            arith=ort.STRICT, want=want)


def _kept_mask(ctx, ort, p, j, ys):
    return _grid(ctx, ort, p, j, ys, ("mask",))["mask"][0].reshape(64, 32).astype(bool)


def _spot(ctx, ort, p, j, ys):
    r = _grid(ctx, ort, p, j, ys, ("ex", "ey"))
    return r["ex"][0], r["ey"][0]


def test_rays_device_pointer_form(ctx, ort):
    """ort_trace3d_rays_dev == ort_trace3d_rays, bit for bit"""
    import torch
    P = ort.prescriptions.DOUBLE_GAUSS
    ctx.set_layout(P["surfaces"])
    rng = np.random.default_rng(9)
    N = 5000
    y0, x0, u0, v0 = rng.uniform(-12, 12, N), rng.uniform(-12, 12, N), rng.uniform(-0.2, 0.2, N), rng.uniform(-0.2, 0.2, N)
    dev = torch.device("cuda", 0)
    d = [torch.from_numpy(a).to(dev) for a in (y0, x0, u0, v0)]
    ns = P["surfaces"].shape[0] - 1
    xv = torch.empty((ns, N), dtype=torch.float64, device=dev); yv = torch.empty_like(xv)
    k = torch.empty((3, N), dtype=torch.float64, device=dev); fl = torch.empty(N, dtype=torch.uint8, device=dev)
    for arith in (ort.STRICT, ort.FAST):
        ctx.trace3d_rays_dev(N, *[t.data_ptr() for t in d], xv.data_ptr(), yv.data_ptr(), k.data_ptr(), fl.data_ptr(), arith=arith,
                             stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        hx, hy, hk, hf = ctx.trace3d_rays(y0, x0, u0, v0, arith=arith)
        assert n_bits_differ(xv.cpu().numpy(), hx) == 0 and n_bits_differ(yv.cpu().numpy(), hy) == 0
        assert n_bits_differ(k.cpu().numpy(), hk) == 0 and np.array_equal(fl.cpu().numpy(), hf)


def test_candidates(ctx, orc, pre, ort):
    P = ort.prescriptions.COOKE
    sysm = pre.solve(P["surfaces"], P["a"], P["h"])
    p = pre.full_trace_inputs(sysm, 0.7, 64)
    C = 96
    base = ort.prescriptions.perturbed_triplets(C)
    rows = p.ext.shape[0]
    RtnK = np.zeros((C, 4, rows))
    RtnK[:, :, :-1] = base
    RtnK[:, 0, -1] = np.inf; RtnK[:, 2, -1] = 1.0
    RtnK[:, 1, -2] = p.focus
    ys = np.linspace(p.y1, p.y2, 32)
    xs = np.linspace(-p.y_EP, p.y_EP, 32)
    ref = orc.candidates(RtnK, ys, xs, p.stop, p.a_stop, p.h_prime, p.u)
    for arith in (ort.STRICT, ort.FAST):
        out = ctx.trace3d_candidates(RtnK, dict(u=p.u, v=0.0, h_prime=p.h_prime), ys, xs, p.stop, p.a_stop, arith=arith)
        assert np.array_equal(out[:, 0], ref[:, 0])                 # kept counts exact
        assert np.max(np.abs(out[:, 1:3] - ref[:, 1:3])) / 25.0 < TOL
        assert np.max(np.abs(out[:, 3] / ref[:, 3] - 1)) < 1e-11     # RMS about the centroid


@pytest.mark.parametrize("H", [0.0, 0.7, 1.0])
def test_candidates_aimed(ctx, orc, pre, ort, H):
    """SURVEY.md section 8 f1: the whole full_trace prelude per candidate on the device, then every candidate over
    its own aimed pupil grid.  (a) the prelude records against the CPU restatement of the reference prelude;
    (b) the spot statistics against the oracle grid trace on IDENTICAL inputs (the device's records)."""
    P = ort.prescriptions.COOKE
    C = 40
    RtnK = ort.prescriptions.perturbed_triplets(C)
    aim = ctx.aim_candidates(RtnK, P["a"], P["h"], H)
    assert np.all(aim[:, 11] == 0.0)
    sub = range(0, C, 5)
    for c in sub:
        S = RtnK[c, :3].T.copy()
        sysm = pre.solve(S, P["a"], P["h"])
        p = pre.full_trace_inputs(sysm, H, 64)
        ref = np.array([p.y1, p.y2, p.y_EP, p.u, p.h_prime, p.focus, p.stop, p.a_stop, p.EP_t])
        got = aim[c, :9]
        assert got[6] == ref[6] and got[7] == ref[7]                  # stop index and stop radius exact
        assert got[5] == ref[5] and aim[c, 10] == sysm.f              # first-order quantities bit-exact (no libm)
        # aimed quantities: both sides stop the reference's secant at |f| <= sqrt(eps) (:229), so they agree to the
        # libm last-ulp differences amplified by that loop, far inside the loop's own tolerance
        assert np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)) < 1e-9
        assert aim[c, 12] == sysm.marginal.nu[-1]
    for arith in (ort.STRICT, ort.FAST):
        out = ctx.trace3d_candidates_aimed(RtnK, aim, 64, 32, arith=arith)
        for c in sub:
            y1, y2, y_EP, u, hp, focus, stop, a_stop = aim[c, :8]
            ext = np.concatenate([RtnK[c], np.array([[np.inf], [0.0], [1.0], [0.0]])], axis=1)
            ext[1, -2] = focus
            ref = orc.candidates(ext[None], np.linspace(y1, y2, 64), np.linspace(0.0, y_EP, 32), int(stop), a_stop, hp, u)[0]
            assert out[c, 0] == ref[0]
            assert np.max(np.abs(out[c, 1:3] - ref[1:3])) / 25.0 < TOL
            assert abs(out[c, 3] / ref[3] - 1) < 1e-10
    # the aimed population agrees with the product's own single-system full_trace (same algorithm, one system)
    S0 = RtnK[3, :3].T.copy()
    system = ort.solve(S0, P["a"], P["h"], backend=ctx)
    e = ort.full_trace(S0, system, H, 64, backend=ctx, arith=ort.STRICT)
    spot, _ = ort.full_trace_candidates(RtnK[3:4], P["a"], P["h"], H, 64, backend=ctx, arith=ort.STRICT)
    assert spot[0, 0] * 2 == len(e.x)
    assert abs(math.sqrt(spot[0, 3] ** 2 + spot[0, 1] ** 2) / e.RMS - 1) < 1e-9


@pytest.mark.parametrize("name,H,conic", [("DOUBLE_GAUSS", 1.0, False), ("DOUBLE_GAUSS", 0.5, False), ("TESSAR", 0.7, False),
                                          ("SINGLET", 1.0, False), ("COOKE", 0.7, True), ("DOUBLE_GAUSS", 0.7, True)])
def test_candidates_aimed_other_systems(ctx, orc, pre, ort, name, H, conic):
    """the per-candidate prelude + aimed sweep on other prescriptions (12-row double-Gauss, Tessar, a singlet whose
    stop is its first surface) and with conic surfaces (Layout{Aspheric}: K enters sag and tilt, the reversed chief-ray
    layout carries reverse(K) shifted by one row, src/RayTracing.jl:272-274)"""
    P = getattr(ort.prescriptions, name)
    S = P["surfaces"][:, :3]
    rows = S.shape[0]
    rng = np.random.default_rng(11)
    C = 6
    RtnK = np.zeros((C, 4, rows))
    for c in range(C):
        RtnK[c, 0] = np.where(np.isfinite(S[:, 0]), S[:, 0] * (1 + rng.uniform(-0.01, 0.01, rows)), S[:, 0])
        RtnK[c, 1] = S[:, 1] * (1 + rng.uniform(-0.005, 0.005, rows))
        RtnK[c, 2] = S[:, 2]
        if conic:
            RtnK[c, 3] = np.where(np.isfinite(S[:, 0]), rng.uniform(-0.6, 0.3, rows), 0.0)
            RtnK[c, 3, 0] = 0.0
            RtnK[c, 3, 1 + (c % 2)::2] = 0.0        # K exactly 0 on every other surface: the atan branch on spheres
    aim = ctx.aim_candidates(RtnK, P["a"], P["h"], H, aspheric=conic)
    assert np.all(aim[:, 11] == 0.0)
    for c in range(C):
        Sc, Kc = RtnK[c, :3].T.copy(), RtnK[c, 3].copy()
        sysm = pre.solve(Sc, P["a"], P["h"])
        p = pre.full_trace_inputs(sysm, H, 48, K=Kc if conic else None, aspheric=conic)
        ref = np.array([p.y1, p.y2, p.y_EP, p.u, p.h_prime, p.focus, p.stop, p.a_stop, p.EP_t])
        got = aim[c, :9]
        assert got[6] == ref[6] and got[7] == ref[7] and got[5] == ref[5] and aim[c, 10] == sysm.f
        assert np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)) < 1e-9
    for arith in (ort.STRICT, ort.FAST):
        out = ctx.trace3d_candidates_aimed(RtnK, aim, 48, 24, arith=arith)
        for c in range(C):
            y1, y2, y_EP, u, hp, focus, stop, a_stop = aim[c, :8]
            ext = np.concatenate([RtnK[c], np.array([[np.inf], [0.0], [1.0], [0.0]])], axis=1)
            ext[1, -2] = focus
            ref = orc.candidates(ext[None], np.linspace(y1, y2, 48), np.linspace(0.0, y_EP, 24), int(stop), a_stop, hp, u)[0]
            assert out[c, 0] == ref[0] and ref[0] > 500
            assert np.max(np.abs(out[c, 1:3] - ref[1:3])) / max(abs(hp), y_EP) < TOL
            assert abs(out[c, 3] / ref[3] - 1) < 1e-9


def test_candidates_aimed_failures(ctx, ort):
    """a candidate whose prelude cannot be completed gives NaN statistics and a status, never an error"""
    P = ort.prescriptions.COOKE
    RtnK = ort.prescriptions.perturbed_triplets(4)
    RtnK[1, 0, 1] = 1.0                        # first surface radius 1 mm: the marginal ray misses it
    RtnK[2, 1, -1] = 3.0                       # last row has a finite thickness: Lens() keeps it, solve() cannot use it
    aim = ctx.aim_candidates(RtnK, P["a"], P["h"], 0.7)
    assert aim[0, 11] == 0.0 and aim[3, 11] == 0.0
    assert aim[1, 11] != 0.0 and aim[2, 11] == 8.0
    out = ctx.trace3d_candidates_aimed(RtnK, aim, 16, 8)
    assert np.all(np.isnan(out[1])) and np.all(np.isnan(out[2]))
    assert np.all(np.isfinite(out[0])) and np.all(np.isfinite(out[3]))
    with pytest.raises(ort.OrtError):
        ctx.aim_candidates(RtnK, P["a"], P["h"], 1.5)


# ------------------------------------------------------------------------------------------------
# EXTENSION (SURVEY.md section 8 f3/f4): OPL / OPD accumulation and per-surface aperture clipping
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,H,vig", [("COOKE", 0.0, False), ("COOKE", 1.0, True), ("DOUBLE_GAUSS", 0.7, True),
                                        ("TESSAR", 1.0, True), ("SINGLET", 0.7, False)])
def test_grid_opd_and_vignetting(ctx, orc, pre, ort, name, H, vig):
    P = getattr(ort.prescriptions, name)
    sysm = pre.solve(P["surfaces"], P["a"], P["h"])
    p = pre.full_trace_inputs(sysm, H, 64)
    a = np.append(P["a"], np.inf) if vig else None               # image plane: unlimited
    rr, yc = p.focus - sysm.XP.t, p.h_prime
    opl_ref, scale = 100.0, -1.0 / 587.5618e-6
    g = orc.grid_trace_ext(p.ext, p.ys, p.xs, p.stop, p.a_stop, p.h_prime, u=p.u, v=p.v, K=p.K, a=a, xc=0.0, yc=yc,
                           rr=rr, opl_ref=opl_ref, opd_scale=scale)
    ctx.set_layout(p.ext, p.K)
    ctx.set_apertures(a)
    fld = dict(u=p.u, v=p.v, h_prime=p.h_prime, opd_xc=0.0, opd_yc=yc, opd_radius=rr, opl_ref=opl_ref)
    ext = ort.EXT_OPD | (ort.EXT_VIGNETTE if vig else 0)
    m = g["mask"].astype(bool)
    for arith in (ort.STRICT, ort.FAST):
        r = ctx.trace3d_grid([fld], p.ys, p.xs, p.stop, p.a_stop, arith=arith, ext=ext, opd_scale=scale,
                             want=("ex", "ey", "opd", "mask", "flags", "stats"))
        assert np.array_equal(r["mask"][0], g["mask"]) and np.array_equal(r["flags"][0], g["flags"])
        st = r["stats"][0]
        assert int(st["n_kept"]) == g["n_kept"] and int(st["n_vig"]) == int(((g["flags"] & 16) != 0).sum())
        if arith == ort.STRICT:
            assert bits_equal(r["opd"][0], g["opd"]) and bits_equal(r["ex"][0], g["ex"])
        else:
            # OPD is a difference of ~100 mm optical paths: 1e-12 relative to the path length
            err_mm = np.nanmax(np.abs(r["opd"][0] - g["opd"])) / abs(scale)
            assert np.array_equal(np.isnan(r["opd"][0]), np.isnan(g["opd"])) and err_mm / 100.0 < TOL
        if m.any():
            assert abs(st["mean_opd"] - g["opd"][m].mean()) / abs(scale) / 100.0 < TOL
            ref_m2 = ((g["opd"][m] - g["opd"][m].mean()) ** 2).sum()
            assert abs(st["m2_opd"] - ref_m2) <= 1e-9 * max(ref_m2, 1.0)
        # compacted OPD follows the same order
        rc = ctx.trace3d_grid([fld], p.ys, p.xs, p.stop, p.a_stop, arith=arith, ext=ext, opd_scale=scale, compact=True,
                              want=("opd", "mask", "stats"))
        assert np.array_equal(rc["opd"][0][:int(st["n_kept"])], r["opd"][0][m])
    ctx.set_apertures(None)


def test_rays_opl(ctx, orc, ort):
    S = ort.prescriptions.DOUBLE_GAUSS["surfaces"]
    rng = np.random.default_rng(12)
    N = 3000
    y0, x0 = rng.uniform(-20, 20, N), rng.uniform(-20, 20, N)
    u0, v0 = rng.uniform(-0.15, 0.15, N), rng.uniform(-0.15, 0.15, N)
    ref = np.array([orc.trace3d_ext(S, y0[i], x0[i], u0[i], v0[i])[3] for i in range(N)])
    truth = np.array([orc.trace3d_ext(S, y0[i], x0[i], u0[i], v0[i], truth=True) for i in range(N)])
    ctx.set_layout(S)
    xs, ys, ks, fs, ols = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.STRICT, opl=True)
    assert n_bits_differ(ols, ref) == 0
    xf, yf, kf, ff, olf = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.FAST, opl=True)
    ok = ~np.isnan(ref)
    assert np.array_equal(np.isnan(olf), np.isnan(ref))
    cond = np.abs(ref[ok] / truth[ok] - 1)
    assert np.all(np.abs(olf[ok] / truth[ok] - 1) <= TOL / 2 + 2 * cond)


def test_wavefront_api(ctx, ort):
    """the public wavefront() on the GPU: parabola = perfect imaging, Cooke W040 = Seidel (book) value"""
    ort.set_default_backend(ctx)
    P = ort.prescriptions.PARABOLA
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"])
    w = ort.wavefront(s.layout, s, [0.0], 64)[0]
    assert w.rms < 1e-9
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"])
    w = ort.wavefront(s.layout, s, [0.0], 64)[0]
    e = ort.full_trace(s, 0.0)
    n = len(w.opd) // 2
    rho = e.r[:n]
    c = np.linalg.lstsq(np.column_stack([rho ** 2, rho ** 4, rho ** 6, rho ** 8]), w.opd[:n], rcond=None)[0]
    assert abs(c[1] / (2 * s.marginal.u[-1] / 587.5618e-6 * (-0.186575) / 8) - 1) < 0.03


def test_many_fields_one_call_equals_per_field_calls(ctx, ort, pre):
    """fields are a grid dimension of the kernel: 11 fields (own aimed y-range each) in ONE call -- host-pointer path
    (single launch sequence) and device-pointer path, with ordered compaction -- equal 11 single-field calls bit for bit"""
    import torch
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = np.linspace(0.0, 1.0, 11)
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ctx.set_layout(p["ext"], p["K"])
    ny, nx = 53, 29                                   # ragged: 1537 rays per field, not a multiple of the 256-ray tile
    ys = np.stack([np.linspace(p["y1"][j], p["y2"][j], ny) for j in range(11)])
    xs = np.linspace(0.0, p["y_EP"], nx)
    flds = [dict(u=float(p["u"][j]), h_prime=float(p["h_prime"][j])) for j in range(11)]
    want = ("ex", "ey", "r", "theta", "mask", "flags", "stats")
    for compact in (False, True):
        allr = ctx.trace3d_grid(flds, ys, xs, p["stop"], p["a_stop"], compact=compact, want=want)
        for j in range(11):
            one = ctx.trace3d_grid([flds[j]], ys[j], xs, p["stop"], p["a_stop"], compact=compact, want=want)
            n = int(one["stats"]["n_kept"][0]) if compact else ny * nx
            assert allr["stats"][j].tobytes() == one["stats"][0].tobytes()
            assert np.array_equal(allr["mask"][j], one["mask"][0]) and np.array_equal(allr["flags"][j], one["flags"][0])
            for k in ("ex", "ey", "r", "theta"):
                assert np.array_equal(allr[k][j][:n], one[k][0][:n], equal_nan=True), (k, j, compact)
        # device-pointer path, all fields in one enqueue
        dev = torch.device("cuda", 0)
        NN = ny * nx
        d = {k: torch.empty((11, NN), dtype=torch.float64, device=dev) for k in ("ex", "ey", "r", "theta")}
        d["mask"] = torch.empty((11, NN), dtype=torch.uint8, device=dev)
        st = torch.zeros((11, ort.STATS_BYTES), dtype=torch.uint8, device=dev)
        d_ys, d_xs = torch.from_numpy(ys).to(dev), torch.from_numpy(xs).to(dev)
        ptrs = {k: v.data_ptr() for k, v in d.items()}
        ptrs["stats"] = st.data_ptr()
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), ny, d_xs.data_ptr(), nx, p["stop"], p["a_stop"], ptrs,
                             stream=torch.cuda.current_stream().cuda_stream, compact=compact, ys_per_field=True)
        torch.cuda.synchronize()
        recs = np.frombuffer(st.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
        for j in range(11):
            n = int(recs[j]["n_kept"]) if compact else NN
            assert recs[j].tobytes() == allr["stats"][j].tobytes()
            assert np.array_equal(d["ex"][j][:n].cpu().numpy(), allr["ex"][j][:n], equal_nan=True)
            assert np.array_equal(d["theta"][j][:n].cpu().numpy(), allr["theta"][j][:n], equal_nan=True)


# ------------------------------------------------------------------------------------------------
# EXTENSION: aspheric polynomial terms in coefficient form (the reference's p closures cannot cross the C ABI)
# ------------------------------------------------------------------------------------------------
def _poly_layout(ort, name, rng):
    S = getattr(ort.prescriptions, name)["surfaces"][:, :3]
    rows = S.shape[0]
    P = np.zeros((rows, 9))
    for i in range(1, rows):
        if np.isfinite(S[i, 0]) and rng.uniform() < 0.7:
            P[i, 4] = rng.uniform(-3e-7, 3e-7); P[i, 6] = rng.uniform(-3e-10, 3e-10); P[i, 8] = rng.uniform(-1e-13, 1e-13)
    P[rows - 1, 3] = 1e-7                              # an odd term too
    K = np.where(np.isfinite(S[:, 0]), rng.uniform(-0.5, 0.2, rows), 0.0); K[0] = 0.0
    return S, K, P


@pytest.mark.parametrize("name", ["COOKE", "DOUBLE_GAUSS", "SINGLET"])
def test_polynomial_terms_rays(ctx, orc, ort, name):
    """3-D and 2-D tracers with polynomial terms == the CPU restatement, bit for bit (same Horner / complex-step order);
    FAST within 1e-12 of it with the oracle's flags; zero coefficients == no polynomial; clearing works."""
    rng = np.random.default_rng(21)
    S, K, P = _poly_layout(ort, name, rng)
    N = 3000
    y0, x0 = rng.uniform(-9, 9, N), rng.uniform(-9, 9, N)
    u0, v0 = rng.uniform(-0.1, 0.1, N), rng.uniform(-0.1, 0.1, N)
    try:
        orc.set_poly(P)
        xo, yo, ko, fo = orc.trace3d_batch(S, y0, x0, u0, v0, K=K)
        y2o, U2o, tso, f2o = orc.trace2d_batch(S, y0, np.arctan(u0), K=K, aspheric=True)
    finally:
        orc.set_poly(None)
    xn, yn, kn, fn = orc.trace3d_batch(S, y0, x0, u0, v0, K=K)
    assert np.nanmax(np.abs(yo - yn)) > 1e-6                      # the terms do something
    ctx.set_layout(S, K)
    ctx.set_polynomials(P)
    xs, ys, ks, fs = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.STRICT)
    assert np.array_equal(fs, fo)
    assert n_bits_differ(xs, xo) == 0 and n_bits_differ(ys, yo) == 0 and n_bits_differ(ks, ko) == 0
    # FAST: the K-form body for surfaces with terms (fast_step, kcode 7); rays it cannot vouch for are re-traced in the
    # reference arithmetic, so the flags and the NaN pattern are the oracle's
    xf, yf, kf, ff = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.FAST)
    assert np.array_equal(ff, fo)
    assert np.array_equal(np.isnan(yf), np.isnan(yo)) and np.array_equal(np.isnan(kf), np.isnan(ko))
    assert n_bits_differ(yf, yo) > 0                              # it is not the reference arithmetic
    tame = (np.hypot(y0, x0) < 6.0) & (np.hypot(u0, v0) < 0.06) & (fo == 0)
    assert tame.sum() > 300
    with np.errstate(all="ignore"):
        e_pos = np.nan_to_num(np.maximum(np.nanmax(np.abs(xf - xo), axis=0), np.nanmax(np.abs(yf - yo), axis=0)) / 10.0, nan=0.0)
        e_dir = np.nan_to_num(np.nanmax(np.abs(kf - ko), axis=0), nan=0.0)
    assert e_pos[tame].max() < TOL and e_dir[tame].max() < TOL    # north_star tolerance on well-conditioned rays
    assert e_pos.max() < 1e-9 and e_dir.max() < 1e-9              # the wild ones (1.3 x aperture, grazing) stay close too
    y2, U2, ts, f2 = ctx.trace2d_batch(y0, np.arctan(u0), aspheric=True)
    assert np.array_equal(f2, f2o)
    # libm (tan, atan, asin) differs in the last ulp: error relative to the position / angle scale
    assert abs_rel_err(y2, y2o, 10.0) < TOL and abs_rel_err(U2, U2o, 1.0) < TOL
    # 3-D == 2-D on meridional rays
    xm, ym, km, fm = ctx.trace3d_rays(y0, np.zeros(N), u0, np.zeros(N), arith=ort.STRICT)
    ok = ~np.isnan(ym[-1]) & ~np.isnan(y2[-1])
    assert np.max(np.abs(ym[:, ok] - y2[1:, ok])) < 1e-10 and np.all(xm[:, ok] == 0.0)
    # zero coefficients and clearing
    ctx.set_polynomials(np.zeros_like(P))
    xz, yz, kz, fz = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.STRICT)
    assert n_bits_differ(yz, yn) == 0
    ctx.set_polynomials(P); ctx.set_polynomials(None)
    xc, yc, kc, fc = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.STRICT)
    assert n_bits_differ(yc, yn) == 0
    ctx.set_polynomials(P); ctx.set_layout(S, K)                  # a new layout clears them too
    xc, yc, kc, fc = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.FAST)
    assert np.nanmax(np.abs(yc - yn)) < 1e-9


def test_polynomial_terms_grid_and_full_trace(ctx, orc, pre, ort):
    """grid sweep with polynomial terms (EXT instantiation): STRICT == oracle bit for bit, FAST within 1e-12 with the same mask;
    full_trace through the host API (prelude with the 2-D polynomial tracer, reversed chief-ray layout with reverse(p))"""
    rng = np.random.default_rng(22)
    S, K, P = _poly_layout(ort, "COOKE", rng)
    K[:] = 0.0
    Pc = ort.prescriptions.COOKE
    sysm = pre.solve(S, Pc["a"], Pc["h"])
    p = pre.full_trace_inputs(sysm, 0.7, 48)
    # <= 10 coefficients travel as a kernel parameter (unrolled Horner, fast_step<POLY = 2>), longer rows are read from
    # global memory in a run-time loop (POLY = 1): 9 columns, then 13 with a y^12 term
    P13 = np.hstack([P, np.zeros((P.shape[0], 4))]); P13[2, 12] = 3e-19
    scale = max(abs(p.h_prime), 1.0)
    for Pq in (P, P13):
        Pext = np.vstack([Pq, np.zeros((1, Pq.shape[1]))])
        try:
            orc.set_poly(Pext)
            g = orc.grid_trace(p.ext, p.ys, p.xs, p.stop, p.a_stop, p.h_prime, u=p.u, v=p.v, K=p.K)
        finally:
            orc.set_poly(None)
        ctx.set_layout(p.ext, p.K)
        ctx.set_polynomials(Pext)
        for arith in (ort.STRICT, ort.FAST):
            for want in (("ex", "ey", "r", "theta", "mask", "flags", "stats"), ("ex", "ey", "mask", "stats")):
                r = ctx.trace3d_grid([dict(u=p.u, v=p.v, h_prime=p.h_prime)], p.ys, p.xs, p.stop, p.a_stop, arith=arith, want=want)
                assert np.array_equal(r["mask"][0], g["mask"]) and int(r["stats"]["n_kept"][0]) == g["n_kept"]
                if arith == ort.STRICT:
                    assert bits_equal(r["ex"][0], g["ex"]) and bits_equal(r["ey"][0], g["ey"])
                else:                                   # the K-form polynomial body; a handful of rays re-traced strictly
                    assert abs_rel_err(r["ex"][0], g["ex"], scale) < TOL and abs_rel_err(r["ey"][0], g["ey"], scale) < TOL
                    assert not bits_equal(r["ex"][0], g["ex"]) and int(r["stats"]["n_strict"][0]) < 48 * 24 // 20
                    if "flags" in want: assert np.array_equal(r["flags"][0], g["flags"])
        ctx.set_polynomials(None)
    # host API: a Layout with coefficient polynomials, against the oracle prelude + grid on the same layout
    L = ort.Layout(S, p=list(P))
    system = ort.solve(L, Pc["a"], Pc["h"], backend=ctx)
    e = ort.full_trace(L, system, 0.7, 48, backend=ctx)
    e0 = ort.full_trace(ort.Layout(S), system, 0.7, 48, backend=ctx)
    assert e.RMS != e0.RMS and len(e.x) > 1500
    pp = ort.host._full_trace_setup(L, system, [0.7], 48, None, ctx)      # the product prelude's inputs -> the oracle grid
    assert pp["P"] is not None and pp["P"].shape[0] == pp["ext"].shape[0]
    try:
        orc.set_poly(pp["P"])
        g = orc.grid_trace(pp["ext"], pre.jl_range(pp["y1"][0], pp["y2"][0], 48), pre.jl_range(0.0, pp["y_EP"], 24), pp["stop"],
                           pp["a_stop"], float(pp["h_prime"][0]), u=float(pp["u"][0]), v=0.0, K=pp["K"])
    finally:
        orc.set_poly(None)
    m = g["mask"]
    *_, rms = orc.mirror_stats(orc.compact(m, g["ex"]), orc.compact(m, g["ey"]), orc.compact(m, g["r"]), orc.compact(m, g["theta"]))
    assert len(e.x) == 2 * g["n_kept"] and abs(e.RMS / rms - 1) < 1e-11
