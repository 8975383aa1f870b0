"""through_focus host logic without a GPU: a backend whose trace3d_focus loops the oracle's grid sweep over the foci (the
image-plane distance t[rows-2] set to each focus in turn), against the oracle's own full_trace at each focus."""
import math

import numpy as np
import pytest

from oracle_backend import OracleBackend


class FocusOracleBackend(OracleBackend):
    """trace3d_focus answered by M oracle grid sweeps, one per focus, in the layout of Context.trace3d_focus"""

    def trace3d_focus(self, fields, ys, xs, stop, a_stop, foci, arith=1, compact=False, want=("stats",)):
        from ort_b200 import STATS_DTYPE
        S0 = self.S.copy()
        ys = np.asarray(ys, dtype=np.float64)
        nf, M, NN = len(fields), len(foci), ys.shape[-1] * len(xs)
        res = {"stats": np.zeros((nf, M), dtype=STATS_DTYPE)}
        res.update({k: np.full((nf, M, NN), np.nan) for k in ("ex", "ey") if k in want})
        try:
            for m, f in enumerate(foci):
                self.S = S0.copy()
                self.S[-2, 1] = f
                g = OracleBackend.trace3d_grid(self, fields, ys, xs, stop, a_stop, arith=arith, compact=compact)
                res["stats"][:, m] = g["stats"]
                for k in ("ex", "ey"):
                    if k in res:
                        res[k][:, m] = g[k]
        finally:
            self.S = S0
        return res


@pytest.fixture(scope="module")
def be(orc):
    return FocusOracleBackend()


def _systems(ort, pre, be, name):
    P = getattr(ort.prescriptions, name)
    return ort.solve(P["surfaces"], P["a"], P["h"], backend=be), pre.solve(P["surfaces"], P["a"], P["h"])


def _bfd(system):
    return float(system.marginal.z[-1] - system.marginal.z[-2])


def _golden_min(fun, a, b, tol=1e-10):
    g = (math.sqrt(5.0) - 1.0) / 2.0
    c, d = b - g * (b - a), a + g * (b - a)
    fc, fd = fun(c), fun(d)
    while b - a > tol:
        if fc < fd:
            b, d, fd = d, c, fc
            c = b - g * (b - a)
            fc = fun(c)
        else:
            a, c, fc = c, d, fd
            d = a + g * (b - a)
            fd = fun(d)
    return 0.5 * (a + b)


@pytest.mark.parametrize("name", ["SINGLET", "COOKE"])
def test_rms_per_focus_equals_oracle_full_trace(ort, pre, be, name):
    s, so = _systems(ort, pre, be, name)
    bfd = _bfd(s)
    foci = bfd + np.linspace(-0.02, 0.02, 5) * bfd
    Hs = (0.0, 0.7, 1.0)
    tf = ort.through_focus(s.layout, s, Hs, foci, 64, backend=be, spots=True)
    assert len(tf) == len(Hs)
    for H, t in zip(Hs, tf):
        assert t.H == H and np.array_equal(t.foci, foci) and t.stats.shape == (len(foci),)
        for j, f in enumerate(foci):
            e = pre.full_trace(so, H, 64, focus=float(f))
            assert math.isclose(t.rms[j], e.RMS, rel_tol=1e-12), (name, H, f, t.rms[j], e.RMS)
            assert t.n_kept == len(e.x) // 2
            assert np.array_equal(t.spots[j][0], e.x) and np.array_equal(t.spots[j][1], e.y)


@pytest.mark.parametrize("name", ["SINGLET", "COOKE"])
def test_best_focus_matches_golden_section(ort, pre, be, name):
    s, so = _systems(ort, pre, be, name)
    bfd = _bfd(s)
    H = 0.7
    foci = bfd + np.linspace(-0.1, 0.03, 7) * bfd         # the singlet's real-ray best focus is ~7 % short of its BFD
    t = ort.through_focus(s.layout, s, [H], foci, 64, backend=be)[0]
    assert t.bracketed and math.isfinite(t.best_focus)
    fbest = _golden_min(lambda f: pre.full_trace(so, H, 64, focus=f).RMS, foci[0], foci[-1])
    assert math.isclose(t.best_focus, fbest, rel_tol=1e-6), (t.best_focus, fbest)
    rbest = pre.full_trace(so, H, 64, focus=fbest).RMS
    assert math.isclose(t.best_rms, rbest, rel_tol=1e-6, abs_tol=1e-12), (t.best_rms, rbest)
    assert t.best_rms <= t.rms.min() * (1 + 1e-12)


def test_best_focus_nan_and_bracketed(ort, pre, be):
    s, _ = _systems(ort, pre, be, "COOKE")
    bfd = _bfd(s)
    two = ort.through_focus(s.layout, s, [0.7], [bfd - 0.5, bfd + 0.5, bfd - 0.5, bfd + 0.5], 32, backend=be)[0]
    assert math.isnan(two.best_focus) and math.isnan(two.best_rms) and not two.bracketed
    one = ort.through_focus(s.layout, s, [0.7], [bfd], 32, backend=be)[0]
    assert math.isnan(one.best_focus) and one.rms.shape == (1,) and not one.bracketed
    # three foci on one side of the minimum: the parabola is still exact, its vertex lies outside the range
    inside = ort.through_focus(s.layout, s, [0.7], bfd + np.linspace(-2.0, 2.0, 5), 32, backend=be)[0]
    side = ort.through_focus(s.layout, s, [0.7], inside.best_focus + np.array([3.0, 4.0, 5.0]), 32, backend=be)[0]
    assert inside.bracketed and not side.bracketed
    assert math.isclose(side.best_focus, inside.best_focus, rel_tol=1e-6)


def test_best_focus_fit_is_the_vertex(ort):
    f = np.array([1.0, 2.0, 3.0, 4.0])
    rms = np.sqrt(2.0 * (f - 2.5) ** 2 + 0.25)
    bf, br = ort.host.best_focus_fit(f, rms)
    assert math.isclose(bf, 2.5, rel_tol=1e-12) and math.isclose(br, 0.5, rel_tol=1e-12)
    assert all(math.isnan(v) for v in ort.host.best_focus_fit(f, np.sqrt(4.0 - (f - 2.5) ** 2)))     # opens downwards


def test_argument_checks(ort, pre, be):
    s, _ = _systems(ort, pre, be, "COOKE")
    with pytest.raises(ValueError):
        ort.through_focus(s.layout, s, [0.0], [], backend=be)
    with pytest.raises(ValueError):
        ort.through_focus(s.layout, s, [0.0], np.zeros(ort._lib.MAX_FOCI + 1), backend=be)
    with pytest.raises(ValueError):
        ort.through_focus(s.layout, s, [0.0], [1.0, np.nan], backend=be)
    P = ort.prescriptions.COOKE
    poly = ort.Layout(P["surfaces"], p=[None] * 2 + [(0.0, 0.0, 1e-6)] + [None] * (len(P["surfaces"]) - 3))
    with pytest.raises(NotImplementedError):
        ort.through_focus(poly, s, [0.0], [70.0, 80.0], backend=be)
