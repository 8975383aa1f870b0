"""Diffraction MTF without a GPU: mtf()'s host logic through a backend whose trace3d_mtf runs the oracle's full-grid OPD
sweep and tests/mtf_ref.py -- frequencies, defaults, cutoffs, chunking over MAX_FIELDS, argument checks, RayBasis
rejection -- and the physics of the definition: the OTF is the Fourier transform of psf_ref's PSF over one alias period,
the diffraction-limited paraboloid follows the circular-pupil MTF, and the exact properties OTF(0) = 1, |OTF| <= 1, a
real sagittal OTF and 0 past the cutoff."""
import math

import numpy as np
import pytest

import mtf_ref as mr
import psf_ref as pr
from oracle_backend import OracleBackend

LAM = 587.5618e-6


class MtfOracleBackend(OracleBackend):
    """trace3d_mtf (and trace3d_psf) answered by an oracle grid sweep and mtf_ref / psf_ref, in the layout of Context"""

    def _sweep(self, fields, ys, xs, stop, a_stop, arith, ext, opd_scale):
        return OracleBackend.trace3d_grid(self, fields, ys, xs, stop, a_stop, arith=arith, compact=False,
                                          want=("opd", "mask", "stats"), ext=ext, opd_scale=opd_scale)

    def trace3d_mtf(self, fields, ys, xs, stop, a_stop, freqs, scale, arith=1, ext=1, opd_scale=1.0):
        g = self._sweep(fields, ys, xs, stop, a_stop, arith, ext, opd_scale)
        otf, status = mr.sets_otf(g["opd"], g["mask"], g["stats"], ys, xs, freqs, scale)
        self.last = dict(ys=np.asarray(ys), xs=np.asarray(xs), scale=scale, freqs=np.array(freqs), n_calls=len(fields))
        return dict(stats=g["stats"], otf=otf, status=status)

    def trace3d_psf(self, fields, ys, xs, stop, a_stop, n_u, n_v, du, dv, scale, arith=1, ext=1, opd_scale=1.0):
        g = self._sweep(fields, ys, xs, stop, a_stop, arith, ext, opd_scale)
        psf, strehl, peak, status = pr.sets_psf(g["opd"], g["mask"], g["stats"], ys, xs, n_u, n_v, du, dv, scale)
        return dict(stats=g["stats"], psf=psf, strehl=strehl, peak=peak, status=status)


@pytest.fixture()
def be(orc):
    return MtfOracleBackend()


def _system(ort, be, name="COOKE", a=None):
    P = getattr(ort.prescriptions, name)
    return ort.solve(ort.Layout(P["surfaces"]), P["a"] if a is None else a, P["h"], backend=be)


def test_frequencies_defaults_and_cutoffs(ort, be):
    s = _system(ort, be)
    k = 24
    f = ort.mtf(s.layout, s, [0.0, 1.0], k_rays=k, backend=be)
    sc = 1.0 / (LAM * s.f)
    p = ort.host._full_trace_setup(s.layout, s, [0.0, 1.0], k, None, be)
    nu_c = 2.0 * sc * p["y_EP"]                                      # 1 / (lam F#)
    assert be.last["scale"] == sc and np.array_equal(be.last["freqs"], np.linspace(0.0, nu_c, 32))
    xs = be.last["xs"]
    assert xs[0] == 0.0 and len(xs) == k // 2
    for j, (x, H) in enumerate(zip(f, (0.0, 1.0))):
        assert x.H == H and x.status == 0 and x.n_kept == int(x.stats["n_kept"][0]) > 0
        assert x.otf.shape == (2, 32) and x.otf.dtype == np.complex128
        assert np.array_equal(x.mtf, np.abs(x.otf)) and np.array_equal(x.ptf, np.angle(x.otf))
        assert np.array_equal(x.freqs, np.linspace(0.0, nu_c, 32))
        ys = be.last["ys"][j]
        assert ys[0] > ys[-1]                                        # the host's ys run downwards: dy < 0
        assert x.cutoff[0] == pytest.approx(nu_c, rel=1e-14)         # 2 (nx - 1) dx s = 2 y_EP s
        assert x.cutoff[1] == pytest.approx(sc * abs(ys[-1] - ys[0]), rel=1e-14)
        assert x.mtf[0][0] == 1.0 and x.mtf[1][0] == 1.0
    g = ort.mtf(s.layout, s, [0.5], freqs=[3.0, 0.0, 1e9, 17.5], k_rays=k, backend=be)[0]
    assert g.otf.shape == (2, 4) and list(g.freqs) == [3.0, 0.0, 1e9, 17.5]
    assert np.all(g.otf[:, 1] == 1.0) and np.all(g.otf[:, 2] == 0.0)


def test_argument_checks(ort, be):
    s = _system(ort, be)
    for kw in (dict(freqs=[-1.0]), dict(freqs=[1.0, math.inf]), dict(freqs=[math.nan]), dict(freqs=[]),
               dict(freqs=np.zeros(ort._lib.MTF_MAX_FREQS + 1)), dict(k_rays=3), dict(k_rays=8.0)):
        with pytest.raises(ValueError):
            ort.mtf(s.layout, s, [0.0], backend=be, **kw)
    assert not hasattr(be, "last")                                   # refused before anything was traced
    assert len(ort.mtf(s.layout, s, [0.0], freqs=np.zeros(ort._lib.MTF_MAX_FREQS), k_rays=4, backend=be)[0].freqs) \
        == ort._lib.MTF_MAX_FREQS
    assert be.a is None


def test_more_fields_than_one_call(ort, be):
    s = _system(ort, be, "SINGLET")
    Hs = np.linspace(0.0, 1.0, ort._lib.MAX_FIELDS + 3)
    f = ort.mtf(s.layout, s, Hs, freqs=[0.0, 20.0, 55.5], k_rays=12, backend=be)
    assert be.last["n_calls"] == 3
    one = [ort.mtf(s.layout, s, [H], freqs=[0.0, 20.0, 55.5], k_rays=12, backend=be)[0] for H in (Hs[0], Hs[-1])]
    assert len(f) == len(Hs) and [x.H for x in f] == list(Hs)
    assert np.array_equal(f[0].otf, one[0].otf) and np.array_equal(f[-1].otf, one[1].otf)


def test_raybasis_rejected(ort, be):
    s = _system(ort, be)
    rb = ort.host.raybasis(s, 0.5, -200.0)
    with pytest.raises(NotImplementedError):
        ort.mtf(s.layout, rb, [0.0], k_rays=16, backend=be)
    assert be.a is None


def test_otf_is_the_transform_of_the_psf(ort, be):
    """at lattice frequencies the OTF equals the normalised DFT of psf_ref's PSF over exactly one alias period:
    n_u du = 1 / (s dx), n_v dv = 1 / (s |dy|), n_u = 4 nx - 3, n_v = 2 ny - 1 (every lag of the mirrored pupil is one
    DFT bin), pixel centres at (i - (n - 1)/2) d.  1e-10: the grid is a lattice only to the ulp of Julia's range."""
    s = _system(ort, be)
    k, H = 20, 0.8
    sc = 1.0 / (LAM * s.f)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [H], k, None, False, be, "test")
    ys = ys[0]
    dx, dy = mr.steps(ys, xs)
    nx, ny = len(xs), len(ys)
    n_u, n_v = 4 * nx - 3, 2 * ny - 1
    du, dv = 1 / (sc * dx * n_u), 1 / (sc * abs(dy) * n_v)
    x = ort.psf(s.layout, s, [H], n_pix=(n_u, n_v), pixel=(du, dv), k_rays=k, backend=be)[0]
    assert x.status == 0
    ks, kt = np.arange(2 * nx - 1), np.arange(ny)
    nu_s, nu_t = ks * sc * dx, kt * sc * abs(dy)
    dft_s = (x.psf.sum(axis=0) @ np.exp(-2j * np.pi * nu_s[None, :] * x.u[:, None])) / x.psf.sum()
    dft_t = (x.psf.sum(axis=1) @ np.exp(-2j * np.pi * nu_t[None, :] * x.v[:, None])) / x.psf.sum()
    m = ort.mtf(s.layout, s, [H], freqs=np.concatenate([nu_s, nu_t]), k_rays=k, backend=be)[0]
    assert m.status == 0
    assert np.max(np.abs(m.otf[0][:len(ks)] - dft_s)) < 1e-10, np.max(np.abs(m.otf[0][:len(ks)] - dft_s))
    assert np.max(np.abs(m.otf[1][len(ks):] - dft_t)) < 1e-10, np.max(np.abs(m.otf[1][len(ks):] - dft_t))
    assert np.max(np.abs(dft_t.imag)) > 1e-3                          # an aberrated field: the tangential PTF is not 0


def test_diffraction_limited_paraboloid(ort, be):
    """PARABOLA at NA 0.1 on axis, k_rays = 1024 (nx = 512): the circular-pupil MTF (2/pi)(acos v - v sqrt(1 - v^2)),
    v = nu / nu_c, nu_c = 2 s y_EP.  The sampled pupil departs from the disk in two ways, both of order 1/nx:
    - the x = 0 column counts twice, an excess weight n0 / n ~ (2 y_EP / |dy|) / (pi y_EP^2 / (dx |dy|)) = 2 dx / (pi y_EP)
      at every lag that pairs it (C(0) = 2n + 2n0);
    - the cells cut by the rim: their share of the disk is ~ perimeter x step / area = 2 (dx + |dy|) / y_EP, and their
      share of the overlap of two shifted disks is of the same order.
    With dx = |dy| = y_EP / (nx - 1) the sum is (2/pi + 4) / (nx - 1) = 0.0091; half of it, 0.0045, bounds what the
    curve (a difference of two areas, each normalised by C(0)) can move.  A frequency scale off by 1 % moves the curve by
    up to 0.01 max v |dMTF/dv| = 0.01 (4/pi) / 2 = 0.0064, above that bound: the second half of the test checks it."""
    s = _system(ort, be, "PARABOLA", a=np.array([5.0]))
    k = 1024
    p = ort.host._full_trace_setup(s.layout, s, [0.0], k, None, be)
    nu_c = 2.0 * p["y_EP"] / (LAM * s.f)
    assert abs(nu_c / (2 * 0.1 / LAM) - 1) < 1e-9                     # 1 / (lam F#) = 2 NA / lam
    v = np.linspace(0.0, 1.2, 25)
    m = ort.mtf(s.layout, s, [0.0], freqs=v * nu_c, k_rays=k, backend=be)[0]
    nx = k // 2
    tol = 0.5 * (2 / np.pi + 4) / (nx - 1)

    def ideal(vv):
        vv = np.minimum(vv, 1.0)
        return (2 / np.pi) * (np.arccos(vv) - vv * np.sqrt(1 - vv ** 2))

    assert m.status == 0
    for az in range(2):
        err = np.max(np.abs(m.mtf[az] - ideal(v)))
        assert err < tol, (az, err, tol)
        assert np.max(np.abs(m.mtf[az] - ideal(v * 1.01))) > tol      # the same comparison fails at a 1 % scale error
        assert np.max(np.abs(m.mtf[az] - ideal(v / 1.01))) > tol
    assert np.all(m.otf[:, v > 1.0] == 0.0)                          # past the sampled cutoff 2 (nx - 1) dx s = nu_c
    assert np.max(np.abs(m.otf[1].imag)) < 1e-12                      # a symmetric pupil: no phase


def test_exact_properties(ort, be):
    """MTF(0) = 1 exactly, MTF <= 1 + 1e-12, the sagittal imaginary part 0, exactly 0 past the cutoff (unsorted
    frequencies, on, between and past lattice lags)"""
    s = _system(ort, be)
    k = 32
    sc = 1.0 / (LAM * s.f)
    p = ort.host._full_trace_setup(s.layout, s, [0.0], k, None, be)
    nu_c = 2.0 * sc * p["y_EP"]
    rng = np.random.default_rng(5)
    freqs = np.concatenate([[0.0, nu_c * 1.0001, 3 * nu_c], rng.uniform(0, 1.1 * nu_c, 40)])
    for x in ort.mtf(s.layout, s, [0.0, 0.6, 1.0], freqs=freqs, k_rays=k, vignette=True, backend=be):
        assert x.status == 0
        assert x.otf[0][0] == 1.0 and x.otf[1][0] == 1.0 and x.mtf[0][0] == 1.0 and x.mtf[1][0] == 1.0
        assert np.all(x.mtf <= 1 + 1e-12)
        assert np.all(x.otf[0].imag == 0.0)
        assert np.all(x.otf[0][freqs > x.cutoff[0]] == 0.0) and np.all(x.otf[1][freqs > x.cutoff[1]] == 0.0)
        assert np.all(x.otf[:, 1:3] == 0.0)


def test_reference_forms_agree():
    """brute (explicit multiset, all pairs) against fast (mirrored amplitude, shifted products) in float64, and brute in
    longdouble, on random masked sets, ascending and descending ys, |W| up to 1e6 waves, frequencies unsorted"""
    rng = np.random.default_rng(3)
    for ny, nx, sgn in ((10, 6, 1), (7, 2, -1), (3, 9, -1), (12, 5, 1)):
        ys = sgn * (0.3 + np.arange(ny) * 0.25)
        xs = np.arange(nx) * 0.31
        opd = rng.uniform(-1e6, 1e6, ny * nx)
        mask = (rng.random(ny * nx) < 0.85).astype(np.uint8)
        n = int(mask.sum())
        s = 1.7
        dx, dy = mr.steps(ys, xs)
        freqs = rng.permutation(np.concatenate([np.arange(0, 2 * nx) * s * dx, rng.uniform(0, 2.2 * nx * s * dx, 9),
                                                np.arange(0, ny + 1) * s * abs(dy), rng.uniform(0, 1.1 * ny * s * abs(dy), 9)]))
        a, sa = mr.set_otf(opd, mask, n, ys, xs, freqs, s, "fast")
        b, sb = mr.set_otf(opd, mask, n, ys, xs, freqs, s, "brute")
        c, sc = mr.set_otf(opd, mask, n, ys, xs, freqs, s, "brute", dtype=np.longdouble)
        assert sa == sb == sc == 0
        assert np.max(np.abs(a - b)) < 1e-13 and np.max(np.abs(b - c)) < 1e-13, (np.max(np.abs(a - b)), np.max(np.abs(b - c)))
        P = np.where(mask.reshape(ny, nx) == 1, pr.phase(opd.reshape(ny, nx)), 0)
        cs, ct = mr.lags_brute(P, 2 * (nx - 1), ny - 1)
        n0 = int(np.sum(mask.reshape(ny, nx)[:, 0] == 1))
        assert abs(cs[0] - (2 * n + 2 * n0)) < 1e-12 and abs(ct[0] - (2 * n + 2 * n0)) < 1e-12
        assert np.max(np.abs(cs.imag)) < 1e-12                        # the mirror makes the sagittal sums real
    # statuses: no kept ray, a non-finite kept opd, a grid that is not a mirrored lattice
    ys, xs = np.linspace(-1, 1, 5), np.linspace(0, 1, 4)
    opd, mask = np.zeros(20), np.ones(20, dtype=np.uint8)
    assert mr.set_otf(opd, 0 * mask, 0, ys, xs, [1.0], 1.0)[1] == 1
    assert mr.set_otf(np.where(np.arange(20) == 7, np.nan, opd), mask, 20, ys, xs, [1.0], 1.0)[1] == 3
    assert mr.set_otf(opd, mask, 20, ys, xs + 0.1, [1.0], 1.0)[1] == 4
    assert mr.set_otf(opd, mask, 20, np.zeros(5), xs, [1.0], 1.0)[1] == 4
    assert mr.set_otf(opd, mask, 20, ys, -xs, [1.0], 1.0)[1] == 4
