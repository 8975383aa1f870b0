"""Zernike fit without a GPU: the numpy reference module (orthonormality, closed forms, the mirror split), and zernike()'s
host logic through a backend whose trace3d_zernike runs the oracle's full-grid OPD sweep and tests/zernike_ref.py --
record assembly, chunking over MAX_FIELDS, both pupil norms, the parabola and the Seidel W040 of the Cooke triplet."""
import math

import numpy as np
import pytest

import zernike_ref as zr
from oracle_backend import OracleBackend

LAM = 587.5618e-6


class ZernikeOracleBackend(OracleBackend):
    """trace3d_zernike answered by an oracle grid sweep and zernike_ref, in the layout of Context.trace3d_zernike"""

    def trace3d_zernike(self, fields, ys, xs, stop, a_stop, n_max, r_norm=0.0, arith=1, ext=1, opd_scale=1.0):
        g = OracleBackend.trace3d_grid(self, fields, ys, xs, stop, a_stop, arith=arith, compact=False,
                                       want=("opd", "r", "theta", "mask", "stats"), ext=ext, opd_scale=opd_scale)
        nf = len(fields)
        coef = np.zeros((nf, zr.n_terms(n_max)))
        resid = np.zeros((nf, 2))
        status = np.zeros(nf, dtype=np.int32)
        for j in range(nf):
            st = g["stats"][j]
            coef[j], resid[j], status[j] = zr.set_fit(g["opd"][j], g["r"][j], g["theta"][j], g["mask"][j],
                                                      int(st["n_kept"]), float(st["r_max"]), n_max, r_norm)
        return dict(stats=g["stats"], coef=coef, resid=resid, status=status)


@pytest.fixture(scope="module")
def be(orc):
    return ZernikeOracleBackend()


def _system(ort, be, name="COOKE"):
    P = getattr(ort.prescriptions, name)
    return ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=be)


# ---- the reference module --------------------------------------------------------------------------------------------
def test_orthonormal_over_unit_disk():
    """Gauss-Legendre in rho (weight rho) x uniform theta integrates every product of terms of order <= 12 exactly"""
    n_max = 12
    x, w = np.polynomial.legendre.leggauss(20)
    rho, wr = 0.5 * (x + 1.0), 0.5 * w
    th = np.arange(64) * (2 * np.pi / 64)
    R, T = np.meshgrid(rho, th, indexing="ij")
    W = (wr[:, None] * R) * (2 * np.pi / 64) / np.pi
    Z = zr.basis(n_max, R.ravel(), T.ravel(), np.longdouble).astype(np.float64)
    G = Z.T @ (Z * W.ravel()[:, None])
    assert np.max(np.abs(G - np.eye(zr.n_terms(n_max)))) < 1e-13


def test_closed_forms():
    rng = np.random.default_rng(1)
    rho, th = rng.uniform(0, 1, 200), rng.uniform(-np.pi, np.pi, 200)
    Z = zr.basis(4, rho, th)
    s3, s5, s6, s8 = math.sqrt(3), math.sqrt(5), math.sqrt(6), math.sqrt(8)
    forms = {0: np.ones_like(rho), 1: 2 * rho * np.sin(th), 2: 2 * rho * np.cos(th), 3: s6 * rho ** 2 * np.sin(2 * th),
             4: s3 * (2 * rho ** 2 - 1), 5: s6 * rho ** 2 * np.cos(2 * th), 7: s8 * (3 * rho ** 3 - 2 * rho) * np.sin(th),
             8: s8 * (3 * rho ** 3 - 2 * rho) * np.cos(th), 12: s5 * (6 * rho ** 4 - 6 * rho ** 2 + 1)}
    for j, f in forms.items():
        assert np.max(np.abs(Z[:, j] - f)) < 1e-14, j
    n, m = zr.ansi_index(4)
    assert list(zip(n[:6], m[:6])) == [(0, 0), (1, -1), (1, 1), (2, -2), (2, 0), (2, 2)]


def test_mirror_split():
    for n_max, count in ((0, 1), (1, 2), (8, 25), (12, 49)):
        assert int(zr.symmetric(n_max).sum()) == count
    rng = np.random.default_rng(2)
    rho, th = rng.uniform(0, 1, 300), rng.uniform(-np.pi, np.pi, 300)
    n_max = 12
    Z, Zm = zr.basis(n_max, rho, th), zr.basis(n_max, rho, np.pi - th)
    sym = zr.symmetric(n_max)
    assert np.allclose(Zm[:, sym], Z[:, sym], atol=1e-12) and np.allclose(Zm[:, ~sym], -Z[:, ~sym], atol=1e-12)
    # the full-basis fit of the mirrored set equals the symmetric-subset normal equations; antisymmetric terms vanish
    W = Z @ rng.standard_normal(zr.n_terms(n_max))
    c_full = zr.lstsq_mirrored(W, rho, th, n_max)
    c_norm, G = zr.normal_fit(W, rho, th, n_max)
    assert np.max(np.abs(c_full[~sym])) < 1e-10
    assert c_norm is not None and np.all(c_norm[~sym] == 0.0)
    assert np.max(np.abs(c_full - c_norm)) < zr.cond_tol(G, len(W)) * np.sqrt(np.mean(W ** 2)) * 100


# ---- zernike() through the oracle backend ----------------------------------------------------------------------------
@pytest.mark.parametrize("norm", ["stop", "rmax"])
def test_equals_fit_of_wavefront(ort, be, norm):
    s = _system(ort, be)
    Hs = (0.0, 0.7, 1.0)
    fits = ort.zernike(s.layout, s, Hs, n_max=6, k_rays=48, norm=norm, backend=be)
    waves = ort.wavefront(s.layout, s, Hs, 48, backend=be)
    n_idx, m_idx = zr.ansi_index(6)
    sym = zr.symmetric(6)
    for H, z, w in zip(Hs, fits, waves):
        e = ort.full_trace(s.layout, s, H, 48, backend=be)
        n = len(w.opd) // 2
        assert z.H == H and z.n_max == 6 and z.status == 0 and z.n_kept == n
        assert np.array_equal(z.n, n_idx) and np.array_equal(z.m, m_idx) and z.coef.shape == (zr.n_terms(6),)
        assert np.all(z.coef[~sym] == 0.0)
        rho = e.r[:n] * (float(e.stats[0]["r_max"]) / s.a[s.stop - 1] if norm == "stop" else 1.0)
        c = zr.lstsq_mirrored(w.opd[:n], rho, e.t[:n], 6)
        scale = max(np.sqrt(np.mean(w.opd ** 2)), 1e-3)
        assert np.max(np.abs(z.coef - c)) < 1e-9 * scale, (H, norm)
        res = w.opd[:n] - zr.basis(6, rho, e.t[:n]) @ z.coef
        assert abs(z.rms_resid - np.sqrt(np.mean(res ** 2))) < 1e-9 * scale
        assert abs(z.pv_resid - (res.max() - res.min())) < 1e-9 * scale


def test_more_fields_than_one_call(ort, be):
    s = _system(ort, be, "SINGLET")
    Hs = np.linspace(0.0, 1.0, ort._lib.MAX_FIELDS + 3)
    fits = ort.zernike(s.layout, s, Hs, n_max=4, k_rays=16, backend=be)
    one = [ort.zernike(s.layout, s, [H], n_max=4, k_rays=16, backend=be)[0] for H in (Hs[0], Hs[-1])]
    assert len(fits) == len(Hs) and [f.H for f in fits] == list(Hs)
    assert np.array_equal(fits[0].coef, one[0].coef) and np.array_equal(fits[-1].coef, one[1].coef)


def test_parabola_has_zero_wavefront(ort, be):
    P = ort.prescriptions.PARABOLA
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=be)
    z = ort.zernike(s.layout, s, [0.0], n_max=8, k_rays=64, backend=be)[0]
    assert z.status == 0 and np.max(np.abs(z.coef)) < 1e-9 and z.rms_resid < 1e-9 and z.pv_resid < 1e-9


def test_on_axis_w040_matches_seidel(ort, be):
    """the rho^4 monomial of the m = 0 terms (norm rmax) reproduces the Seidel W040, as the monomial fit of
    test_extension_opd does (test/runtests.jl:184,215: W040 = alpha * (-0.186575) / 8 waves, alpha = 2 u' / lambda)"""
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=be)
    z = ort.zernike(s.layout, s, [0.0], n_max=8, k_rays=64, norm="rmax", backend=be)[0]
    assert z.status == 0
    mono = np.zeros(9)                      # coefficient of rho^k
    for j in np.flatnonzero(z.m == 0):
        n = int(z.n[j])
        for k in range(n // 2 + 1):
            c = (-1) ** k * math.factorial(n - k) / (math.factorial(k) * math.factorial(n // 2 - k) ** 2)
            mono[n - 2 * k] += z.coef[j] * math.sqrt(n + 1) * c
    w040_seidel = 2 * s.marginal.u[-1] / LAM * (-0.186575) / 8
    assert abs(mono[4] / w040_seidel - 1) < 0.03
    # on axis the map is rotationally symmetric; the square pupil grid leaves ~1e-5 in the m = 4, 8 terms
    assert np.max(np.abs(z.coef[z.m != 0])) < 1e-4 * np.max(np.abs(z.coef))


def test_vignetting_and_argument_checks(ort, be):
    s = _system(ort, be)
    v = ort.zernike(s.layout, s, [1.0], n_max=4, k_rays=48, vignette=True, backend=be)[0]
    u = ort.zernike(s.layout, s, [1.0], n_max=4, k_rays=48, backend=be)[0]
    assert v.n_kept < u.n_kept and int(v.stats["n_vig"][0]) > 0 and v.status == 0
    for kw in (dict(n_max=13), dict(n_max=-1), dict(n_max=2.0), dict(norm="edge")):
        with pytest.raises(ValueError):
            ort.zernike(s.layout, s, [0.0], backend=be, **kw)
