"""Diffraction PSF without a GPU: psf()'s host logic through a backend whose trace3d_psf runs the oracle's full-grid OPD
sweep and tests/psf_ref.py -- pixel coordinates, defaults, the alias check, chunking over MAX_FIELDS, RayBasis
rejection -- and the physics of the definition: Strehl against the wavefront, the tilt shift, Parseval over one alias
period, the PSF centroid against the geometric spot centroid, and the Airy pattern of a diffraction-limited mirror."""
import math

import numpy as np
import pytest

import psf_ref as pr
from oracle_backend import OracleBackend

LAM = 587.5618e-6


class PsfOracleBackend(OracleBackend):
    """trace3d_psf answered by an oracle grid sweep and psf_ref, in the layout of Context.trace3d_psf"""

    def __init__(self):
        super().__init__()
        self.opd_hook = None                    # tests may replace the OPD map: f(opd [ny][nx], ys, xs) -> opd

    def trace3d_psf(self, fields, ys, xs, stop, a_stop, n_u, n_v, du, dv, scale, arith=1, ext=1, opd_scale=1.0):
        g = OracleBackend.trace3d_grid(self, fields, ys, xs, stop, a_stop, arith=arith, compact=False,
                                       want=("opd", "mask", "stats"), ext=ext, opd_scale=opd_scale)
        opd = g["opd"]
        if self.opd_hook is not None:
            ys2 = np.asarray(ys)
            opd = np.stack([self.opd_hook(opd[j].reshape(ys2.shape[-1], len(xs)), ys2[j] if ys2.ndim == 2 else ys2,
                                          np.asarray(xs)).ravel() for j in range(len(fields))])
        psf, strehl, peak, status = pr.sets_psf(opd, g["mask"], g["stats"], ys, xs, n_u, n_v, du, dv, scale)
        self.last = dict(ys=np.asarray(ys), xs=np.asarray(xs), scale=scale, du=du, dv=dv)
        return dict(stats=g["stats"], psf=psf, strehl=strehl, peak=peak, status=status)


@pytest.fixture()
def be(orc):
    return PsfOracleBackend()


def _system(ort, be, name="COOKE", a=None):
    P = getattr(ort.prescriptions, name)
    return ort.solve(ort.Layout(P["surfaces"]), P["a"] if a is None else a, P["h"], backend=be)


def test_coordinates_and_defaults(ort, be):
    s = _system(ort, be)
    k = 24
    f = ort.psf(s.layout, s, [0.0, 1.0], k_rays=k, backend=be)
    sc = 1.0 / (LAM * s.f)
    p = ort.host._full_trace_setup(s.layout, s, [0.0], k, None, be)
    pitch = 1.0 / (4.0 * sc * p["y_EP"])                          # lam F# / 2
    assert be.last["scale"] == sc and be.last["du"] == pitch and be.last["dv"] == pitch
    assert abs(pitch / (LAM * s.f / (2 * p["y_EP"]) / 2) - 1) < 1e-15
    for x, H in zip(f, (0.0, 1.0)):
        assert x.H == H and x.status == 0 and x.psf.shape == (k - 1, k - 1)
        assert np.array_equal(x.u, (np.arange(k - 1) - (k - 2) / 2) * pitch) and np.array_equal(x.v, x.u)
        assert x.u[(k - 2) // 2] == 0.0                              # odd n_pix: the chief ray's image point is a pixel
        iv, iu = np.unravel_index(int(np.argmax(x.psf)), x.psf.shape)
        assert x.peak == x.psf.max() and x.peak_uv == (x.u[iu], x.v[iv])
        assert x.strehl == pytest.approx(x.psf[(k - 2) // 2, (k - 2) // 2], rel=1e-12)
        assert x.n_kept == int(x.stats["n_kept"][0]) > 0
    g = ort.psf(s.layout, s, [0.5], n_pix=(7, 4), pixel=(2e-3, 3e-3), k_rays=k, backend=be)[0]
    assert g.psf.shape == (4, 7) and np.array_equal(g.u, (np.arange(7) - 3) * 2e-3)
    assert np.array_equal(g.v, (np.arange(4) - 1.5) * 3e-3)


def test_argument_checks_and_alias(ort, be):
    s = _system(ort, be)
    for kw in (dict(n_pix=0), dict(n_pix=1025), dict(n_pix=(3, 4, 5)), dict(pixel=0.0), dict(pixel=-1e-3),
               dict(pixel=math.inf), dict(k_rays=1)):
        with pytest.raises(ValueError):
            ort.psf(s.layout, s, [0.0], backend=be, **kw)
    with pytest.raises(ValueError, match=r"k_rays >= \d+ would fit") as e:
        ort.psf(s.layout, s, [1.0], n_pix=200, k_rays=32, backend=be)
    k_fit = int(str(e.value).rsplit(">= ", 1)[1].split()[0])
    assert not hasattr(be, "last")                                  # refused before anything was traced
    assert ort.psf(s.layout, s, [1.0], n_pix=200, k_rays=k_fit, backend=be)[0].status == 0
    with pytest.raises(ValueError, match="alias period"):
        ort.psf(s.layout, s, [1.0], n_pix=(5, 5), pixel=(1e-3, 1.0), k_rays=32, backend=be)
    assert be.a is None                                             # the apertures are reset after a refusal too


def test_more_fields_than_one_call(ort, be):
    s = _system(ort, be, "SINGLET")
    Hs = np.linspace(0.0, 1.0, ort._lib.MAX_FIELDS + 3)
    f = ort.psf(s.layout, s, Hs, n_pix=9, k_rays=12, backend=be)
    one = [ort.psf(s.layout, s, [H], n_pix=9, k_rays=12, backend=be)[0] for H in (Hs[0], Hs[-1])]
    assert len(f) == len(Hs) and [x.H for x in f] == list(Hs)
    assert np.array_equal(f[0].psf, one[0].psf) and np.array_equal(f[-1].psf, one[1].psf)


def test_raybasis_rejected(ort, be):
    s = _system(ort, be)
    rb = ort.host.raybasis(s, 0.5, -200.0)
    with pytest.raises(NotImplementedError):
        ort.psf(s.layout, rb, [0.0], k_rays=16, backend=be)


def test_strehl_equals_wavefront_mean_phase(ort, be):
    s = _system(ort, be)
    Hs = (0.0, 0.7, 1.0)
    f = ort.psf(s.layout, s, Hs, k_rays=32, n_pix=5, backend=be)
    w = ort.wavefront(s.layout, s, Hs, 32, backend=be)
    for x, wf in zip(f, w):
        ref = abs(np.mean(np.exp(2j * np.pi * wf.opd))) ** 2
        assert abs(x.strehl - ref) <= 1e-12, (x.H, x.strehl, ref)
        assert 0.0 < x.strehl <= 1.0


def test_tilt_moves_the_peak(ort, be):
    """W = a y: E(eta) = sum exp(2 pi i (a + s eta) y) peaks at eta = -a / s, at the diffraction-limited value"""
    s = _system(ort, be, "PARABOLA", a=np.array([5.0]))
    sc = 1.0 / (LAM * s.f)
    pitch = 1e-3
    a = 12 * pitch * sc                                             # -a / s: twelve pixels below the centre
    be.opd_hook = lambda o, ys, xs: np.where(np.isfinite(o), a * ys[:, None] + 0.0 * xs[None, :], o)
    x = ort.psf(s.layout, s, [0.0], n_pix=41, pixel=pitch, k_rays=64, backend=be)[0]
    assert x.status == 0 and abs(x.peak - 1.0) < 1e-12
    assert x.peak_uv == (0.0, x.v[20 - 12]) and abs(x.v[20 - 12] + a / sc) < 1e-15
    assert x.strehl < 1e-2                                          # ~4 waves of tilt over the pupil


def test_parseval_over_one_alias_period(ort, be):
    """pixels covering exactly one alias period in xi and in eta sample the mirrored pupil's DFT: the pixel sum is
    n_u n_v sum |c|^2 / (2n)^2 with c = 2 P at x = 0 (the column counted twice) and P elsewhere"""
    s = _system(ort, be)
    k = 20
    p = ort.host._full_trace_setup(s.layout, s, [0.8], k, None, be)
    sc = 1.0 / (LAM * s.f)
    dx = ort.host.jl_range(0.0, p["y_EP"], k // 2)[1]
    ys = ort.host.jl_range(p["y1"][0], p["y2"][0], k)
    dy = abs(ys[1] - ys[0])
    n_u, n_v = k - 1, k                                             # 2 nx - 1 distinct x, ny distinct y
    x = ort.psf(s.layout, s, [0.8], n_pix=(n_u, n_v), pixel=(1 / (sc * dx * n_u), 1 / (sc * dy * n_v)), k_rays=k,
                backend=be)[0]
    n = x.n_kept
    w = ort.wavefront(s.layout, s, [0.8], k, backend=be)[0]
    n0 = int(np.sum(w.x[:n] == 0.0))
    expect = n_u * n_v * (2 * n + 2 * n0) / (2 * n) ** 2
    assert n0 > 0 and abs(x.psf.sum() / expect - 1) < 1e-12, (x.psf.sum(), expect)


def test_centroid_matches_geometric_spot(ort, be):
    """Cooke H = 1, k_rays = 512: the PSF centroid (over the default pixel grid) against the geometric spot centroid,
    both relative to the chief ray's image point, within 0.05 x the geometric RMS radius"""
    s = _system(ort, be)
    k = 512
    x = ort.psf(s.layout, s, [1.0], k_rays=k, backend=be)[0]
    e = ort.full_trace(s.layout, s, 1.0, k, backend=be)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [1.0], k, None, False, be, "test")
    geo = float(np.mean(e.y)) + flds[0]["h_prime"] - flds[0]["opd_yc"]
    cen = float((x.psf.sum(axis=1) @ x.v) / x.psf.sum())
    assert x.status == 0 and abs(cen - geo) < 0.05 * e.RMS, (cen, geo, e.RMS)
    assert abs(float((x.psf.sum(axis=0) @ x.u) / x.psf.sum())) < 1e-12 * e.RMS     # even in xi


def test_airy_pattern_of_the_parabola(ort, be):
    """PARABOLA at NA 0.1 (stop semi-aperture 5 mm at f = 50 mm), on axis, k_rays = 256: the cut along xi is
    [2 J1(v) / v]^2, v = 2 pi NA r / lam, and strehl_ref = 1"""
    from scipy.special import j1
    s = _system(ort, be, "PARABOLA", a=np.array([5.0]))
    x = ort.psf(s.layout, s, [0.0], k_rays=256, backend=be)[0]
    c = (len(x.v) - 1) // 2
    na = 5.0 / s.f
    v = 2 * np.pi * na * x.u / LAM
    airy = np.where(v == 0, 1.0, (2 * j1(np.where(v == 0, 1.0, v)) / np.where(v == 0, 1.0, v)) ** 2)
    assert abs(x.strehl - 1.0) < 1e-12 and x.peak_uv == (0.0, 0.0)
    assert np.max(np.abs(x.psf[c] - airy)) < 5e-3, np.max(np.abs(x.psf[c] - airy))


def test_reference_forms_agree():
    """the float64 and longdouble statements of psf_ref agree on a small random set with |W| up to 1e6 waves"""
    rng = np.random.default_rng(3)
    ny, nx = 9, 6
    ys, xs = np.linspace(-1.0, 1.2, ny), np.linspace(0.0, 1.1, nx)
    opd = rng.uniform(-1e6, 1e6, ny * nx)
    mask = (rng.random(ny * nx) < 0.8).astype(np.uint8)
    n = int(mask.sum())
    a = pr.set_psf(opd, mask, n, ys, xs, 7, 6, 0.05, 0.07, 3.0)
    b = pr.set_psf(opd, mask, n, ys, xs, 7, 6, 0.05, 0.07, 3.0, dtype=np.longdouble)
    assert a[3] == b[3] == 0 and np.max(np.abs(a[0] - b[0])) < 1e-14 and abs(a[1][0] - b[1][0]) < 1e-14
    assert np.max(np.abs(a[0] - a[0][:, ::-1])) < 1e-14                 # even in xi
