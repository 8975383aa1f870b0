"""encircled_energy host logic without a GPU: a backend whose trace3d_energy runs the oracle's full-grid sweep (once per
focus) and answers with numpy sort / searchsorted, against a direct computation on full_trace's mirrored RealRayError."""
import math

import numpy as np
import pytest

from energy_ref import distances, set_energy
from oracle_backend import OracleBackend


class EnergyOracleBackend(OracleBackend):
    """trace3d_energy answered by oracle grid sweeps (one per focus) and numpy, in the layout of Context.trace3d_energy"""

    def trace3d_energy(self, fields, ys, xs, stop, a_stop, radii=None, fracs=None, foci=None, arith=1, metric="circle",
                       center="centroid"):
        from ort_b200 import STATS_DTYPE
        r = np.empty(0) if radii is None else np.asarray(radii, dtype=np.float64)
        q = np.empty(0) if fracs is None else np.asarray(fracs, dtype=np.float64)
        nf = len(fields)
        planes = [None] if foci is None else list(foci)
        M = len(planes)
        stats = np.zeros((nf, M), dtype=STATS_DTYPE)
        counts = np.zeros((nf, M, len(r)), dtype=np.int64)
        radius = np.zeros((nf, M, len(q)))
        S0 = self.S.copy()
        try:
            for m, f in enumerate(planes):
                self.S = S0.copy()
                if f is not None:
                    self.S[-2, 1] = f
                g = OracleBackend.trace3d_grid(self, fields, ys, xs, stop, a_stop, arith=arith, compact=False)
                stats[:, m] = g["stats"]
                for j in range(nf):
                    st = g["stats"][j]
                    counts[j, m], radius[j, m] = set_energy(g["ex"][j], g["ey"][j], g["mask"][j], int(st["n_kept"]),
                                                            float(st["mean_y"]), r, q, metric, center)
        finally:
            self.S = S0
        if foci is None:
            stats, counts, radius = stats[:, 0], counts[:, 0], radius[:, 0]
        return dict(stats=stats, counts=counts, radius=radius)


@pytest.fixture(scope="module")
def be(orc):
    return EnergyOracleBackend()


def _system(ort, be, name="COOKE"):
    P = getattr(ort.prescriptions, name)
    return ort.solve(P["surfaces"], P["a"], P["h"], backend=be)


def _mirrored_direct(e, radii, fracs, metric):
    """the curve and radii of the 2n-point mirrored spot of a RealRayError, measured from (0, mean y)"""
    cy = float(e.stats[0]["mean_y"])
    d = np.sort(distances(e.x, e.y, cy, metric))
    n2 = len(d)
    frac = np.searchsorted(d, radii, side="right") / n2
    rad = np.array([d[min(max(math.ceil(q * n2), 1), n2) - 1] for q in fracs])
    return frac, rad


@pytest.mark.parametrize("metric", ["circle", "square"])
@pytest.mark.parametrize("name", ["COOKE", "SINGLET"])
def test_equals_mirrored_full_trace(ort, be, name, metric):
    s = _system(ort, be, name)
    Hs = (0.0, 0.7, 1.0)
    radii = np.linspace(0.0, 0.05, 41)
    fracs = (0.3, 0.5, 0.8, 0.9, 1.0)
    ee = ort.encircled_energy(s.layout, s, Hs, radii=radii, fractions=fracs, k_rays=64, metric=metric, backend=be)
    assert len(ee) == len(Hs)
    for H, e in zip(Hs, ee):
        rre = ort.full_trace(s.layout, s, H, 64, backend=be)
        frac, rad = _mirrored_direct(rre, radii, fracs, metric)
        assert e.H == H and e.n_kept == len(rre.x) // 2 and e.fraction.shape == (1, len(radii))
        assert np.array_equal(e.fraction[0], frac)
        assert np.array_equal(e.radius[0].view(np.uint64), rad.view(np.uint64))
        assert np.array_equal(e.foci, [s.marginal.z[-1] - s.marginal.z[-2]])
        assert np.array_equal(e.fractions, fracs) and np.array_equal(e.radii, radii)


def test_through_focus_equals_full_trace_per_focus(ort, be):
    s = _system(ort, be)
    bfd = float(s.marginal.z[-1] - s.marginal.z[-2])
    foci = bfd + np.array([-0.5, 0.0, 0.5])
    radii = np.linspace(0.0, 0.2, 9)
    ee = ort.encircled_energy(s.layout, s, (0.0, 1.0), radii=radii, fractions=(0.8,), k_rays=32, foci=foci, backend=be)
    for e in ee:
        assert e.fraction.shape == (3, len(radii)) and e.radius.shape == (3, 1) and np.array_equal(e.foci, foci)
        for j, f in enumerate(foci):
            frac, rad = _mirrored_direct(ort.full_trace(s.layout, s, e.H, 32, float(f), backend=be), radii, (0.8,), "circle")
            assert np.array_equal(e.fraction[j], frac) and np.array_equal(e.radius[j], rad)


@pytest.mark.parametrize("H", [0.0, 0.7, 1.0])
def test_properties(ort, be, H):
    s = _system(ort, be)
    rre = ort.full_trace(s.layout, s, H, 64, backend=be)
    d = distances(rre.x, rre.y, float(rre.stats[0]["mean_y"]), "circle")
    dmax = float(d.max())
    radii = np.concatenate([np.linspace(0.0, dmax, 50)[:-1], [dmax, 2 * dmax]])
    q = (0.1, 0.25, 0.5, 0.8, 0.9, 0.95, 0.99, 1.0)
    c = ort.encircled_energy(s.layout, s, [H], radii=radii, fractions=q, k_rays=64, backend=be)[0]
    sq = ort.encircled_energy(s.layout, s, [H], radii=radii, fractions=q, k_rays=64, metric="square", backend=be)[0]
    assert np.all(np.diff(c.fraction[0]) >= 0) and c.fraction[0][-2] == 1.0 and c.fraction[0][-1] == 1.0
    assert c.radius[0][-1] == dmax                              # radius(q = 1) is the largest distance
    assert np.all(np.diff(c.radius[0]) >= 0)                    # non-decreasing in q
    assert np.all(sq.radius[0] <= c.radius[0])                  # the square's half-width never exceeds the circle's radius
    assert np.all(sq.fraction[0] >= c.fraction[0])


def test_centroid_and_paraxial_agree_on_axis(ort, be):
    s = _system(ort, be)
    q = (0.5, 0.8, 0.9, 1.0)
    c = ort.encircled_energy(s.layout, s, [0.0], fractions=q, k_rays=64, backend=be)[0]
    p = ort.encircled_energy(s.layout, s, [0.0], fractions=q, k_rays=64, center="paraxial", backend=be)[0]
    cy = abs(float(c.stats[0]["mean_y"]))
    assert cy < 1e-3 * c.radius[0][0]
    # moving the centre by cy moves every distance, hence every order statistic, by at most cy
    assert np.all(np.abs(c.radius[0] - p.radius[0]) <= cy * (1 + 1e-12) + 4 * np.spacing(c.radius[0]))
    assert c.fraction.shape == (1, 0)


def test_argument_checks(ort, be):
    s = _system(ort, be)
    L, ee = s.layout, ort.encircled_energy
    bad = [dict(radii=[0.1, 0.1]), dict(radii=[0.2, 0.1]), dict(radii=[-0.1, 0.1]), dict(radii=[0.0, np.inf]),
           dict(radii=[np.nan]), dict(radii=np.linspace(0, 1, ort._lib.MAX_RADII + 1)), dict(fractions=(0.0,)),
           dict(fractions=(1.5,)), dict(fractions=(np.nan,)), dict(fractions=tuple(np.linspace(0.1, 1, 9))),
           dict(radii=None, fractions=None), dict(radii=[], fractions=()), dict(metric="disc"), dict(center="chief"),
           dict(foci=[]), dict(foci=np.full(ort._lib.MAX_FOCI + 1, 80.0)), dict(foci=[80.0, np.nan]),
           dict(foci=[80.0], focus=80.0)]
    for kw in bad:
        with pytest.raises(ValueError):
            ee(L, s, [0.0], backend=be, **kw)
    P = ort.prescriptions.COOKE
    poly = ort.Layout(P["surfaces"], p=[None] * 2 + [(0.0, 0.0, 1e-6)] + [None] * (len(P["surfaces"]) - 3))
    with pytest.raises(NotImplementedError):
        ee(poly, s, [0.0], foci=[70.0, 80.0], backend=be)
