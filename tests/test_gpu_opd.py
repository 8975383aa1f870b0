"""The OPD of every device path that produces one, against the CPU oracle and the independent 50-digit tracer.

Grid sweeps (ort_trace3d_grid with ORT_EXT_OPD): STRICT bit-identical to orc_grid_trace_ext, FAST within 1e-12 of it
relative to the case's path length (largest |OPL| + |rr|: the closed OPL of a parabola is 0), mask, flags and counts
equal, OPD moments within tolerance, and a subsample compared directly with the 50-digit OPD.  The field records are
those host._wavefront_setup builds (reference sphere through the chief ray's image point); its precondition holds in every
case: the last surface is the appended image plane, the only place where the closure is exact.  Then the raw OPL of
ort_trace3d_rays_opl, the public wavefront() on a mirror system, the three mergers of the OPD statistics, the
multi-context sweep, and the Seidel check of the reference sphere off axis on the device."""
import math

import numpy as np
import pytest

from oracle_backend import OracleBackend
from test_opd_independent import (PHYSICS_HS, check_seidel, dec_opl, field_fit, fixture, seidel_from_fit,
                                  system_layout)
from util import bits_equal, n_bits_differ

pytestmark = pytest.mark.gpu

TOL = 1e-12
LAM = 587.5618e-6
SCALE = -1.0 / LAM                                   # opd_scale of wavefront(): waves, W = OPL_chief - OPL
LEAN = ("ex", "ey", "opd", "mask", "stats")
WIDE = ("ex", "ey", "opd", "mask", "flags", "r", "theta", "stats")


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _poly(rows, ncol):
    """polynomial terms on the COOKE extended layout (no term on the image plane): 9 columns travel as a kernel parameter,
    13 are read from global memory"""
    P = np.zeros((rows, ncol))
    P[1, 4], P[3, 6], P[6, 4], P[7, 3] = 2e-7, -1e-10, -1.5e-7, 1e-7
    P[2, ncol - 1] = 1e-13 if ncol == 9 else 3e-19
    return P


def _case(ort, name, Hs, vignette, k_rays=48, extra_fields=False):
    """the OPD sweep inputs of wavefront() for `name`, built by the host code on the oracle backend, so that the device and
    the oracle trace the same layout, apertures and field records.  extra_fields appends a finite-object field (mode 1)
    and a collimated field with v != 0, both closed on the first field's sphere -> (be, p, xs, ys, flds, ext)"""
    be = OracleBackend()
    L, a, h = system_layout(ort, name)
    s = ort.solve(L, a, h, backend=be)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, k_rays, None, vignette, be, "test")
    if extra_fields:
        f0 = flds[-1]
        sphere = {k: f0[k] for k in ("h_prime", "opd_xc", "opd_yc", "opd_radius", "opl_ref")}
        flds = flds + [dict(mode=1, ybar=-0.4 * p["y_EP"], z0=-400.0, **sphere), dict(mode=0, u=f0["u"], v=0.02, **sphere)]
        ys = np.vstack([ys, ys[-1:], ys[-1:]])
    return be, p, xs, ys, flds, ext


def _run(ctx, ort, be, p, xs, ys, flds, ext, arith, want, compact=False, poly=None):
    ctx.set_layout(be.S, be.K)
    ctx.set_polynomials(poly)
    ctx.set_apertures(be.a if ext & ort.EXT_VIGNETTE else None)
    return ctx.trace3d_grid(flds, ys, xs, p["stop"], p["a_stop"], arith=arith, ext=ext, opd_scale=SCALE, want=want,
                            compact=compact)


def _path_scale(g, flds, j):
    m = g["mask"][j].astype(bool)
    return float(np.max(np.abs(g["opd"][j][m] / SCALE + flds[j]["opl_ref"]))) + abs(flds[j]["opd_radius"])


def check_case(ctx, ort, be, p, xs, ys, flds, ext, n_dec=12, seed=0, poly=None):
    """STRICT == oracle bits, FAST within TOL x path length, lean == wide epilogue, compacted == full grid at the kept rays,
    and a subsample of every field against the 50-digit OPD (polynomial terms: oracle only, n_dec = 0).
    -> worst errors {strict, fast, oracle} against the 50-digit OPD, x path length"""
    g = be.trace3d_grid(flds, ys, xs, p["stop"], p["a_stop"], ext=ext, opd_scale=SCALE, want=WIDE)
    rng = np.random.default_rng(seed)
    worst = dict(strict=0.0, fast=0.0, oracle=0.0)
    res = {}
    for arith in (ort.STRICT, ort.FAST):
        r = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, WIDE, poly=poly)
        rl = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, LEAN, poly=poly)
        rc = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, LEAN, compact=True, poly=poly)
        res[arith] = r
        assert np.array_equal(r["mask"], g["mask"]) and np.array_equal(r["flags"], g["flags"])
        assert np.array_equal(rl["mask"], r["mask"]) and n_bits_differ(rl["opd"], r["opd"]) == 0
        assert rl["stats"].tobytes() == r["stats"].tobytes() == rc["stats"].tobytes()
        for j in range(len(flds)):
            st, gs = r["stats"][j], g["stats"][j]
            m = g["mask"][j].astype(bool)
            n = int(st["n_kept"])
            assert n == int(gs["n_kept"]) > 0 and int(st["n_vig"]) == int(gs["n_vig"]) and int(st["n_clip"]) == int(gs["n_clip"])
            assert np.array_equal(rc["opd"][j][:n], r["opd"][j][m])                   # compacted: same values, same order
            L = _path_scale(g, flds, j)
            if arith == ort.STRICT:
                assert bits_equal(r["opd"][j], g["opd"][j]) and bits_equal(r["ex"][j], g["ex"][j]), j
            else:
                assert np.array_equal(np.isnan(r["opd"][j]), np.isnan(g["opd"][j]))
                err = np.nanmax(np.abs(r["opd"][j] - g["opd"][j])) / abs(SCALE) / L
                assert err < TOL, (j, err)
            # statistics: the device folds a shifted sum in its own order
            assert abs(st["mean_opd"] - gs["mean_opd"]) / abs(SCALE) / L < TOL, j
            assert abs(st["m2_opd"] - gs["m2_opd"]) <= 1e-9 * max(float(gs["m2_opd"]), 1.0), j
    for j, f in enumerate(flds):
        kept = np.flatnonzero(g["mask"][j])
        for idx in rng.choice(kept, size=min(n_dec, len(kept)), replace=False):
            y, x = ys[j][idx // len(xs)], xs[idx % len(xs)]
            u, v = (math.tan((f["ybar"] - y) / f["z0"]), math.tan(-x / f["z0"])) if f.get("mode") == 1 else (f["u"], f.get("v", 0.0))
            ref = dec_opl(be.S, be.K, y, x, u, v, mode=f.get("mode", 0), z0=f.get("z0", 0.0), xc=f["opd_xc"], yc=f["opd_yc"],
                          rr=f["opd_radius"]) - f["opl_ref"]
            L = _path_scale(g, flds, j)
            for key, o in (("strict", res[ort.STRICT]["opd"][j][idx]), ("fast", res[ort.FAST]["opd"][j][idx]),
                           ("oracle", g["opd"][j][idx])):
                worst[key] = max(worst[key], abs(o / SCALE - ref) / L)
    assert max(worst.values()) < TOL, worst
    return worst


# Each case names the k_grid instantiation its FAST sweep reaches (launch_grid, csrc/kern_trace3d.cu); the STRICT sweep of
# every case is k_grid<STRICT, STRICT_RPT, 1>.  WIDE adds flags / r / theta to the lean OPD output set.
@pytest.mark.parametrize("name,Hs,vignette", [
    ("COOKE", (0.0, 0.7, 1.0), False),          # SIMPLE x EXT: <FAST, SE_RPT, 2, 1> (lean) and <.., 2, 0> (wide)
    ("COOKE", (0.0, 0.7, 1.0), True),           # SIMPLE x EXT with EXT_VIGNETTE: <FAST, SE_RPT, 1, 1> and <.., 1, 0>
    ("TESSAR", (0.0, 0.7, 1.0), True),          # the same two, another prescription
    ("DOUBLE_GAUSS", (0.0, 0.7, 1.0), False),   # SIMPLE x EXT, planes in the glass
    ("COOKE_ASPHERIC", (0.0, 0.7, 1.0), False), # general EXT without mirrors (a conic): <FAST, FAST_RPT, 1, 0, false>
    ("DOUBLE_GAUSS_CONIC", (0.0, 0.7, 1.0), True),  # the same with apertures
    ("REFLECTIVE", (0.0, 0.7, 1.0), False),     # EXT with mirrors: <FAST, FAST_RPT, 1>
    ("PARABOLA", (0.0, 0.7, 1.0), True),        # the same, a conic mirror, with apertures
])
def test_grid_opd(ctx, ort, name, Hs, vignette):
    be, p, xs, ys, flds, ext = _case(ort, name, Hs, vignette)
    check_case(ctx, ort, be, p, xs, ys, flds, ext)
    ctx.set_apertures(None)


@pytest.mark.parametrize("name", ["COOKE", "REFLECTIVE"])
def test_grid_opd_finite_object_and_skew_field(ctx, ort, name):
    """a field of mode 1 (start term -n0^2 z0 / Kz through fast_div) and a collimated field with v != 0 (start term
    x Kx + y Ky), in one call with the wavefront fields: COOKE reaches SIMPLE x EXT, REFLECTIVE the mirror EXT kernel"""
    be, p, xs, ys, flds, ext = _case(ort, name, (0.0, 0.7), False, extra_fields=True)
    check_case(ctx, ort, be, p, xs, ys, flds, ext, seed=1)


@pytest.mark.parametrize("ncol", [9, 13])
def test_grid_opd_polynomial_terms(ctx, orc, ort, ncol):
    """polynomial terms with OPD: 9 columns reach <FAST, FAST_RPT, 1, 0, false, 0, 2> (terms as a kernel parameter), 13
    columns <.., 0, 1> (global memory).  The 50-digit tracer has no polynomial sag: oracle only"""
    be, p, xs, ys, flds, ext = _case(ort, "COOKE", (0.0, 0.7, 1.0), True)
    P = _poly(be.S.shape[0], ncol)
    try:
        be.set_polynomials(P)
        g0 = be.trace3d_grid(flds, ys, xs, p["stop"], p["a_stop"], ext=ext, opd_scale=SCALE, want=WIDE)
        check_case(ctx, ort, be, p, xs, ys, flds, ext, n_dec=0, poly=P)
        r = _run(ctx, ort, be, p, xs, ys, flds, ext, ort.FAST, LEAN, poly=P)
        assert int(r["stats"]["n_strict"].max()) < ys.shape[1] * len(xs) // 20          # the polynomial body, not re-traces
    finally:
        be.set_polynomials(None)
        ctx.set_polynomials(None)
        ctx.set_apertures(None)
    be.set_layout(be.S, be.K)
    g1 = be.trace3d_grid(flds, ys, xs, p["stop"], p["a_stop"], ext=ext, opd_scale=SCALE, want=WIDE)
    assert np.nanmax(np.abs(g1["opd"] - g0["opd"])) > 1e-3                             # the terms change the OPD


def test_grid_opd_many_fields_compacted(ctx, ort):
    """eleven fields in one call with ys_per_field (the shape of wavefront()'s sweep), full grid and compacted: the
    compacted OPD is the full-grid OPD at the kept rays, in order, and every field equals its single-field call"""
    be, p, xs, ys, flds, ext = _case(ort, "DOUBLE_GAUSS", np.linspace(0.0, 1.0, 11), True, k_rays=64)
    for arith in (ort.FAST, ort.STRICT):
        full = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, LEAN)
        comp = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, LEAN, compact=True)
        for j in range(len(flds)):
            n = int(full["stats"][j]["n_kept"])
            m = full["mask"][j].astype(bool)
            assert full["stats"][j].tobytes() == comp["stats"][j].tobytes() and n == m.sum() > 0
            assert np.array_equal(comp["opd"][j][:n], full["opd"][j][m]), (arith, j)
            one = ctx.trace3d_grid([flds[j]], ys[j], xs, p["stop"], p["a_stop"], arith=arith, ext=ext, opd_scale=SCALE,
                                   want=LEAN)
            assert one["stats"][0].tobytes() == full["stats"][j].tobytes()
            assert n_bits_differ(one["opd"][0], full["opd"][j]) == 0
    ctx.set_apertures(None)


# ---- raw OPL of ort_trace3d_rays_opl ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["REFLECTIVE", "PARABOLA", "DOUBLE_GAUSS_CONIC", "POLY"])
def test_rays_opl(ctx, orc, ort, name):
    """STRICT bits == orc_trace3d_ext; FAST against the oracle's 80-bit truth (polynomial terms: against the oracle, which
    has no 80-bit polynomial form) within 1e-12 plus the conditioning of the ray"""
    ext, K, amax, umax = fixture(ort, "COOKE" if name == "POLY" else name)
    P = _poly(ext.shape[0], 9) if name == "POLY" else None
    rng = np.random.default_rng(41)
    N = 2000
    y0, x0 = rng.uniform(-amax, amax, N), rng.uniform(-amax, amax, N)
    u0, v0 = rng.uniform(-umax, umax, N), rng.uniform(-umax, umax, N)
    try:
        orc.set_poly(P)
        ref = np.array([orc.trace3d_ext(ext, y0[i], x0[i], u0[i], v0[i], K=K)[3] for i in range(N)])
    finally:
        orc.set_poly(None)
    ctx.set_layout(ext, K)
    if P is not None:
        ctx.set_polynomials(P)
    try:
        *_, fs, ols = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.STRICT, opl=True)
        *_, ff, olf = ctx.trace3d_rays(y0, x0, u0, v0, arith=ort.FAST, opl=True)
    finally:
        ctx.set_polynomials(None)
    assert n_bits_differ(ols, ref) == 0
    ok = ~np.isnan(ref)
    assert ok.sum() > N // 2 and np.array_equal(np.isnan(olf), np.isnan(ref))
    if P is not None:
        assert np.max(np.abs(olf[ok] - ref[ok]) / np.abs(ref[ok])) < TOL
        return
    truth = np.array([orc.trace3d_ext(ext, y0[i], x0[i], u0[i], v0[i], K=K, truth=True) for i in range(N)])
    cond = np.abs(ref[ok] / truth[ok] - 1)
    assert np.all(np.abs(olf[ok] / truth[ok] - 1) <= TOL / 2 + 2 * cond)


# ---- public wavefront ------------------------------------------------------------------------------------------------
def test_wavefront_reflective_equals_oracle_backend(ctx, ort):
    """wavefront() on the device (FAST) for REFLECTIVE at H = 1 equals the oracle backend's, element by element"""
    be = OracleBackend()
    P = ort.prescriptions.REFLECTIVE
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=be)
    wo = ort.wavefront(s.layout, s, [1.0], 64, backend=be)[0]
    wd = ort.wavefront(s.layout, s, [1.0], 64, backend=ctx)[0]
    tol = TOL * 200.0 / LAM                          # waves: paths here are < 200 mm (|rr| + |OPL|)
    assert len(wd.opd) == len(wo.opd) > 2000
    assert np.max(np.abs(wd.opd - wo.opd)) < tol and np.max(np.abs(wd.x - wo.x)) < TOL * 100 and np.max(np.abs(wd.y - wo.y)) < TOL * 100
    assert abs(wd.mean - wo.mean) < tol and abs(wd.pv - wo.pv) < 2 * tol and abs(wd.rms - wo.rms) < tol
    assert wo.rms > 0.05                             # a real aberration to compare, not a perfect focus


# ---- merging OPD statistics ------------------------------------------------------------------------------------------
def test_merge_opd_statistics(ctx, ort):
    """records of row blocks of one OPD + vignetting sweep (one block empty), merged by host.merge_stats, ort_merge_stats
    and ort_merge_stats_dev: the same bytes on every field (all three take the same operations in the same order); against
    the whole-grid record the counts are exact and the OPD moments within a reordered sum's rounding"""
    import torch
    be, p, xs, ys, flds, ext = _case(ort, "COOKE", (0.0, 0.7, 1.0), True, k_rays=64)
    shards = [(0, 20), (20, 20), (20, 47), (47, 64)]
    for arith in (ort.FAST, ort.STRICT):
        recs = np.stack([_run(ctx, ort, be, p, xs, ys[:, lo:hi], flds, ext, arith, ("opd", "stats"))["stats"]
                         for lo, hi in shards])
        assert recs["n_vig"].sum() > 0 and recs["n_kept"][1].sum() == 0
        c = ort._lib.merge_stats_c(recs)
        h = np.array([ort.host.merge_stats(recs[:, f]) for f in range(len(flds))], dtype=ort.STATS_DTYPE)
        d_in = torch.from_numpy(np.ascontiguousarray(recs).view(np.uint8).reshape(-1)).cuda()
        d_out = torch.zeros(len(flds) * ort.STATS_BYTES, dtype=torch.uint8, device="cuda")
        ctx.merge_stats_dev(d_in.data_ptr(), len(shards), len(flds), d_out.data_ptr(),
                            stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        dev = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
        assert c.tobytes() == dev.tobytes() == h.tobytes()
        whole = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, ("opd", "mask", "stats"))
        for f in range(len(flds)):
            a, b = c[f], whole["stats"][f]
            for k in ("n_kept", "n_miss", "n_tir", "n_domain", "n_clip", "n_vig"):
                assert int(a[k]) == int(b[k]), (k, f)
            spread = math.sqrt(float(b["m2_opd"]) / int(b["n_kept"]))
            assert abs(a["mean_opd"] - b["mean_opd"]) <= 1e-12 * (abs(float(b["mean_opd"])) + spread), f
            assert abs(a["m2_opd"] - b["m2_opd"]) <= 1e-11 * float(b["m2_opd"]), f
    ctx.set_apertures(None)


def _multi_case(ort):
    be, p, xs, ys, flds, ext = _case(ort, "COOKE", (0.0, 0.7, 1.0), True, k_rays=64)
    return be, p, xs, ys, flds, ext, ("ex", "ey", "opd", "mask", "flags", "stats")


def test_grid_multi_opd_one_context(ctx, ort):
    """ort_trace3d_grid_multi with EXT_OPD | EXT_VIGNETTE over one context equals the plain sweep byte for byte: opd,
    statistics, mask and flags, full grid and compacted"""
    be, p, xs, ys, flds, ext, want = _multi_case(ort)
    for arith in (ort.FAST, ort.STRICT):
        for compact in (False, True):
            one = _run(ctx, ort, be, p, xs, ys, flds, ext, arith, want, compact=compact)
            m = ort._lib.trace3d_grid_multi([ctx], flds, ys, xs, p["stop"], p["a_stop"], arith=arith, compact=compact,
                                            want=want, ext=ext, opd_scale=SCALE)
            assert m["stats"].tobytes() == one["stats"].tobytes()
            assert np.array_equal(m["mask"], one["mask"]) and np.array_equal(m["flags"], one["flags"])
            for f in range(len(flds)):                  # compacted: the tail behind the kept rays is not written
                n = int(one["stats"][f]["n_kept"]) if compact else one["opd"].shape[1]
                assert m["opd"][f][:n].tobytes() == one["opd"][f][:n].tobytes(), (arith, compact, f)
    ctx.set_apertures(None)


@pytest.mark.skipif("_ngpu() < 2")
def test_grid_multi_opd_two_gpus(ort):
    """the same sweep over two devices: the opd is the one-device opd byte for byte, the merged record is ort_merge_stats
    of the shard records, with exact counts and the OPD moments of the whole grid"""
    be, p, xs, ys, flds, ext, want = _multi_case(ort)
    cs = [ort.Context(0), ort.Context(1)]
    try:
        ort._lib.comm_init_all(cs)
        for arith in (ort.FAST, ort.STRICT):
            one = _run(cs[0], ort, be, p, xs, ys, flds, ext, arith, want)
            two = ort._lib.trace3d_grid_multi(cs, flds, ys, xs, p["stop"], p["a_stop"], arith=arith, want=want, ext=ext,
                                              opd_scale=SCALE)
            assert two["opd"].tobytes() == one["opd"].tobytes() and np.array_equal(two["mask"], one["mask"])
            assert two["stats"].tobytes() == ort._lib.merge_stats_c(two["stats_local"]).tobytes()
            for f in range(len(flds)):
                a, b = two["stats"][f], one["stats"][f]
                assert int(a["n_kept"]) == int(b["n_kept"]) and int(a["n_vig"]) == int(b["n_vig"]) > 0
                spread = math.sqrt(float(b["m2_opd"]) / int(b["n_kept"]))
                assert abs(a["mean_opd"] - b["mean_opd"]) <= 1e-12 * (abs(float(b["mean_opd"])) + spread)
                assert abs(a["m2_opd"] - b["m2_opd"]) <= 1e-11 * float(b["m2_opd"])
    finally:
        for c in cs:
            c.close()


# ---- physics on the device -------------------------------------------------------------------------------------------
def test_off_axis_seidel_terms_on_the_device(ctx, ort):
    """the Seidel check of test_opd_independent on the device's wavefront (FAST), and the same ratios as the oracle
    backend's.  The device prelude aims its own pupil grids (aim_fields), equal to the host's only to the aiming
    tolerance, so the fits differ slightly: measured 6e-4 on the W131 ratio, 3e-4 on W220"""
    be = OracleBackend()
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=be)
    ab = ort.aberrations(s.layout, s, backend=be)
    fits = {}
    for key, bk in (("device", ctx), ("oracle", be)):
        C = field_fit(ort.wavefront(s.layout, s, PHYSICS_HS, 64, backend=bk), [ort.full_trace(s, H, 64, backend=bk) for H in PHYSICS_HS])
        fits[key] = seidel_from_fit(C, PHYSICS_HS, ab.field_sign)
    check_seidel(fits["device"], ab)
    for k in ("W131", "W222", "W220"):
        assert abs(fits["device"][k] / fits["oracle"][k] - 1) < 3e-3, (k, fits)
