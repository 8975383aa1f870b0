"""The tilt branch of the 2-D meridional tracer in the CPU oracle.  The reference chooses it with
iszero(Ks) && ps === zero ? asin(tilt(y, R)) : atan(tilt(y, R, K, p)) (src/RayTracing.jl:162), and a Layout{Aspheric}
holds Polynomial(zero) in p, which is not === zero (src/Types.jl:27, 91): every surface of an aspheric layout -- K = 0
spheres, mirrors and planes included, and so the reversed chief-ray layout of every full_trace -- takes atan.  At ordinary
heights the two forms agree to 1-2 ulp; near grazing they do not, and the rays of trace2d_ref.grazing_rays() are chosen
where they differ by 32 ulp or more.  The oracle is compared bit for bit with trace2d_ref, a plain restatement that makes
the same glibc libm calls.  The geometry itself is pinned against the independent 50-digit tracer."""
import ctypes
import os

import numpy as np
import pytest

import trace2d_ref as tr
from util import n_bits_differ


@pytest.fixture(scope="module")
def cases(ort, pre):
    return tr.branch_cases(ort, pre)


def _mapped_libm():
    with open("/proc/self/maps") as f:
        return sorted({ln.split()[-1] for ln in f if os.path.basename(ln.split()[-1]).startswith("libm.so")})


def test_restatement_and_oracle_share_glibc_libm(orc):
    """the bit-for-bit comparisons below need both sides to round tan / cos / sin / asin / atan alike: the restatement
    calls them through glibc's libm, and the oracle, loaded into the same process, resolves them to that one libm"""
    orc.lib()
    libc = ctypes.CDLL(None)
    libc.gnu_get_libc_version.restype = ctypes.c_char_p
    assert libc.gnu_get_libc_version()                             # glibc, not another C library
    assert tr.LIBM_NAME == "libm.so.6"
    maps = _mapped_libm()
    assert len(maps) == 1, maps                                    # one libm in the process: the oracle's and ours
    with open(os.path.join(os.path.dirname(orc.__file__), "ort_oracle.c")) as f:
        src = f.read()
    assert "#include <math.h>" in src


@pytest.mark.parametrize("case", ["COOKE_ASPHERIC", "REFLECTIVE", "REVERSED_COOKE", "REVERSED_DOUBLE_GAUSS", "DEEP"])
def test_oracle_aspheric_layout_takes_atan_on_every_surface(orc, cases, case):
    """orc.trace2d_batch(aspheric=True) == the atan_always restatement bit for bit on the whole y / U / ts table and the
    flags, for the grazing rays on a K = 0 surface and a random bundle; the grazing rays do tell the branches apart"""
    S, K, surf = cases[case]
    y0, U0, ng = tr.case_rays(S, K, surf)
    assert ng >= 40, ng
    got = orc.trace2d_batch(S, y0, U0, K=K, aspheric=True)
    ref = tr.batch(S, K, y0, U0, "atan_always")
    for a, b in zip(got[:3], ref[:3]):
        assert n_bits_differ(a, b) == 0
    assert np.array_equal(got[3], ref[3])
    old = tr.batch(S, K, y0[:ng], U0[:ng], "per_surface")
    assert n_bits_differ(old[1][surf], ref[1][surf, :ng]) == ng      # every grazing ray discriminates


@pytest.mark.parametrize("case", ["COOKE_ASPHERIC", "REFLECTIVE", "REVERSED_COOKE", "DEEP"])
def test_oracle_matrix_method_takes_asin(orc, cases, case):
    """aspheric=False (AbstractMatrix / Layout{Spherical}: K forced to 0) == the asin restatement bit for bit"""
    S, K, surf = cases[case]
    y0, U0, _ = tr.case_rays(S, K, surf, n_random=300, seed=3)
    got = orc.trace2d_batch(S, y0, U0, K=K, aspheric=False)
    ref = tr.batch(S, K, y0, U0, "asin")
    for a, b in zip(got[:3], ref[:3]):
        assert n_bits_differ(a, b) == 0
    assert np.array_equal(got[3], ref[3])


def test_planes_take_either_form_alike(orc, ort):
    """a plane has tilt 0 in both forms (asin(y / Inf) and atan(y / sqrt(Inf))), so a layout of planes traces the same
    through both methods, and the same as the atan_always restatement"""
    S = np.array([[np.inf, 0.0, 1.0], [np.inf, 5.0, 1.5], [np.inf, 3.0, 1.7], [np.inf, 0.0, 1.0]])
    rng = np.random.default_rng(4)
    y0, U0 = rng.uniform(-20, 20, 500), rng.uniform(-0.5, 0.5, 500)
    a = orc.trace2d_batch(S, y0, U0, K=np.zeros(4), aspheric=True)
    b = orc.trace2d_batch(S, y0, U0, aspheric=False)
    for x, z in zip(a, b):
        assert np.array_equal(x, z, equal_nan=True) if x.dtype != np.uint8 else np.array_equal(x, z)
    assert n_bits_differ(a[1], tr.batch(S, None, y0, U0, "atan_always")[1]) == 0


@pytest.mark.parametrize("name", tr.MERIDIONAL_FIXTURES)
def test_oracle_meridional_rays_match_independent_50_digit_tracer(orc, ort, name):
    """hit heights and tan U of orc_trace2d at every surface against the 50-digit vector tracer at x = v = 0: 2e-14 of
    the position scale on well-conditioned rays; miss / TIR status agrees on every ray, near-grazing and near-TIR ones too"""
    S, K, asph, ymax, umax = tr.meridional_fixture(ort, name)
    y0, U0, edge = tr.meridional_rays(S, K, ymax, umax)
    yt, Ut, _, fl = orc.trace2d_batch(S, y0, U0, K=K, aspheric=asph)
    cond = ~edge & tr.conditioning(lambda y, u: orc.trace2d_batch(S, y, u, K=K, aspheric=asph), y0, U0)
    r = tr.meridional_compare(S, K, y0, U0, yt, Ut, fl, cond, edge)
    assert r["compared"] > 1000 and r["status_differs"] == 0, r
    # a ray 1e-9 mm from the edge of a deep layout can sit within the trace's own rounding of it (a few in a hundred)
    assert r["status_differs_at_edge"] <= 0.05 * r["edge_rays"], r
    assert r["max_position_err_rel"] < 2e-14 and r["max_tanU_err_rel"] < 2e-14, r
