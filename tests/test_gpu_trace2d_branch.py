"""The tilt branch of the device's 2-D meridional tracer (trace2d_step: k_trace2d, k_aim2d, k_aim_candidates).  A
Layout{Aspheric} takes atan(tilt(y, R, K, p)) on every surface (src/RayTracing.jl:162, src/Types.jl:27, 91); the rays of
trace2d_ref.grazing_rays() hit a K = 0 sphere where that form and asin(tilt(y, R)) differ by 32 ulp or more, so they tell
which one the kernel took.  The geometry is pinned against the independent 50-digit tracer.

The aiming kernels are covered by tolerance only.  Their outputs are the roots of secant loops on the height at the stop,
and near grazing the tilt is so steep a function of the ray's parameter (d theta / dy = 1 / (R sqrt(1 - (y/R)^2)), ~700 / R
at 1 - 1e-6) that a few hundred ulp in theta move the root by less than one ulp of it: the branch cannot show in an aimed
value.  There they are compared with the CPU prelude, which the CPU tests pin to the atan form bit for bit."""
import numpy as np
import pytest

import trace2d_ref as tr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cases(ort, pre):
    return tr.branch_cases(ort, pre)


@pytest.mark.parametrize("case", ["COOKE_ASPHERIC", "REFLECTIVE", "REVERSED_COOKE", "REVERSED_DOUBLE_GAUSS", "DEEP"])
def test_k_trace2d_aspheric_layout_takes_atan(ctx, cases, case):
    """k_trace2d through ctx.trace2d_batch(aspheric=True): after the grazed K = 0 sphere, U is within 4 ulp (of the tilt's
    magnitude, where its rounding is made) of the atan form taken from the kernel's own hit height and incoming U, and
    four times closer to it than to the asin form; the whole table agrees with the atan_always restatement to 1e-12"""
    S, K, surf = cases[case]
    y0, U0, ng = tr.case_rays(S, K, surf)
    ctx.set_layout(S, K)
    yk, Uk, tsk, fk = ctx.trace2d_batch(y0, U0, aspheric=True)
    Rj, n1, n2 = float(S[surf, 0]), float(S[surf - 1, 2]), float(S[surf, 2])
    n_disc = 0
    for i in range(ng):
        y, Uin = float(yk[surf, i]), float(Uk[surf - 1, i])
        ua = tr.surface_step(Rj, 0.0, n1, n2, y, Uin, False)
        us = tr.surface_step(Rj, 0.0, n1, n2, y, Uin, True)
        if tr.ulp_diff(ua, us) < 32:          # the kernel's own hit height may sit where the forms round alike
            continue
        n_disc += 1
        err_a, err_s = abs(float(Uk[surf, i]) - ua), abs(float(Uk[surf, i]) - us)
        assert err_a <= 4 * np.spacing(np.pi / 2), (i, y0[i], err_a, err_s)
        assert err_a < err_s / 4, (i, y0[i], err_a, err_s)
    assert n_disc >= min(40, ng // 2), (n_disc, ng)
    ry, rU, rts, rf = tr.batch(S, K, y0, U0, "atan_always")
    assert np.array_equal(rf, fk)
    ok = rf == 0
    sc = np.maximum(np.nanmax(np.abs(ry), axis=0), 1.0)
    assert np.max(np.abs(yk[:, ok] - ry[:, ok]) / sc[ok]) < 1e-12
    # U after a grazing hit carries the steep tilt: 1e-12 only off grazing, the rebased check above covers the rest
    assert np.max(np.abs(Uk[:, ng:][:, ok[ng:]] - rU[:, ng:][:, ok[ng:]])) < 1e-12


@pytest.mark.parametrize("name", tr.MERIDIONAL_FIXTURES)
def test_k_trace2d_meridional_rays_match_independent_50_digit_tracer(ctx, ort, name):
    """hit heights and tan U of k_trace2d at every surface against the 50-digit vector tracer at x = v = 0: 2e-14 of the
    position scale on well-conditioned rays; miss / TIR status agrees off the edge"""
    S, K, asph, ymax, umax = tr.meridional_fixture(ort, name)
    y0, U0, edge = tr.meridional_rays(S, K, ymax, umax)
    ctx.set_layout(S, K)
    yt, Ut, _, fl = ctx.trace2d_batch(y0, U0, aspheric=asph)
    cond = ~edge & tr.conditioning(lambda y, u: ctx.trace2d_batch(y, u, aspheric=asph), y0, U0)
    r = tr.meridional_compare(S, K, y0, U0, yt, Ut, fl, cond, edge)
    assert r["compared"] > 1000 and r["status_differs"] == 0, r
    assert r["status_differs_at_edge"] <= 0.05 * r["edge_rays"], r
    assert r["max_position_err_rel"] < 2e-14 and r["max_tanU_err_rel"] < 2e-14, r


class _NoAimFields:
    """proxy that hides aim_fields so the host runs its own prelude (k_aim2d and k_trace2d, step by step)"""

    def __init__(self, ctx):
        self._c = ctx

    def __getattr__(self, name):
        if name == "aim_fields":
            raise AttributeError(name)
        return getattr(self._c, name)


@pytest.mark.parametrize("name", ["COOKE_ASPHERIC", "COOKE", "DOUBLE_GAUSS", "TESSAR"])
def test_aimed_prelude_matches_cpu_prelude(ctx, ort, pre, name):
    """k_aim_candidates (ort_aim_fields) and k_aim2d (host trace_chief_ray / aim_rays) against the CPU prelude: the
    reversed chief ray of every full_trace is a Layout{Aspheric}, so this covers the atan branch on K = 0 spheres in
    every system.  Covered by tolerance only (see the module docstring)"""
    P = getattr(ort.prescriptions, name)
    S = P["surfaces"]
    K = S[:, 3] if S.shape[1] > 3 else None
    system = ort.solve(S, P["a"], P["h"], backend=ctx)
    Hs = [0.0, 0.5, 1.0]
    sysm = pre.solve(S[:, :3], P["a"], P["h"])
    refs = [pre.full_trace_inputs(sysm, H, 64, K=K, aspheric=K is not None) for H in Hs]
    for be in (ctx, _NoAimFields(ctx)):
        p = ort.host._full_trace_setup(system.layout, system, Hs, 64, None, be)
        for j, r in enumerate(refs):
            for k in ("y1", "y2", "u", "h_prime"):
                assert abs(p[k][j] - getattr(r, k)) <= 1e-14 * max(abs(getattr(r, k)), 1.0), (k, j, p[k][j], getattr(r, k))
        r = refs[0]
        # y_EP is the real marginal ray's secant stopped at |f| <= sqrt(eps) (src/RayTracing.jl:229): the last bits of the
        # libm calls move where it stops, far inside that tolerance (as in test_candidates_aimed)
        assert abs(p["y_EP"] - r.y_EP) <= 1e-9 * max(abs(r.y_EP), 1.0), (p["y_EP"], r.y_EP)
        # EP_t is a difference of nearly equal terms: a last-bit change in the chief ray's angles moves it by thousands of
        # ulp (the branch fix itself moved it 668 ulp for COOKE and 3060 for DOUBLE_GAUSS), so libm alone does too
        assert abs(p["EP_t"] - r.EP_t) <= 1e-11 * max(abs(r.EP_t), 1.0), (p["EP_t"], r.EP_t)
