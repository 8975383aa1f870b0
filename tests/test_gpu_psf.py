"""Diffraction PSF of the wavefront on the device (ort_wavefront_psf_dev, ort_trace3d_psf) against tests/psf_ref.py:
synthetic sets at edge sizes and statuses, the outputs of traced OPD sweeps, the bench-size grid, and determinism,
enqueue-only behaviour, launch counts and validation."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import psf_ref as pr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAM = 587.5618e-6
TOL_PSF, TOL_REF = 1e-11, 1e-12


def _tensor(a):
    import torch
    return torch.from_numpy(np.array(a, copy=True)).cuda()


def _stats(ort, n_kept):
    st = np.zeros(len(n_kept), dtype=ort.STATS_DTYPE)
    st["n_kept"] = n_kept
    return st


def _outs(n_sets, n_u, n_v):
    import torch
    return (torch.full((n_sets, n_v, n_u), -5.0, dtype=torch.float64, device="cuda"),
            torch.full((n_sets, 2), -5.0, dtype=torch.float64, device="cuda"),
            torch.full((n_sets,), -5, dtype=torch.int32, device="cuda"),
            torch.full((n_sets,), -5, dtype=torch.int32, device="cuda"))


def _dev(ctx, ort, opd, mask, stats, ys, xs, n_u, n_v, du, dv, s, stream=0):
    """ort_wavefront_psf_dev on torch copies of [n_sets][ny * nx] arrays -> (psf, strehl, peak, status) numpy"""
    import torch
    n_sets, stride = opd.shape
    ys = np.asarray(ys, dtype=np.float64)
    t_opd, t_mask = _tensor(opd), _tensor(mask.astype(np.uint8))
    t_st = _tensor(np.frombuffer(stats.tobytes(), dtype=np.uint8))
    t_ys, t_xs = _tensor(ys), _tensor(np.asarray(xs, dtype=np.float64))
    out = _outs(n_sets, n_u, n_v)
    sets = dict(n_sets=n_sets, stride=stride, opd=t_opd.data_ptr(), mask=t_mask.data_ptr(), stats=t_st.data_ptr())
    ctx.wavefront_psf_dev(sets, t_ys.data_ptr(), ys.ndim == 2, ys.shape[-1], t_xs.data_ptr(), len(xs), n_u, n_v, du, dv,
                          s, *[o.data_ptr() for o in out], stream=stream)
    torch.cuda.synchronize()
    return tuple(o.cpu().numpy() for o in out)


def _check(got, ref, what=""):
    psf, strehl, peak, status = got
    rpsf, rstrehl, _, rstatus = ref
    assert np.array_equal(status, rstatus), (what, status, rstatus)
    for j in range(len(status)):
        if status[j]:
            assert np.all(np.isnan(psf[j])) and np.all(np.isnan(strehl[j])) and peak[j] == -1, (what, j)
            continue
        err = np.max(np.abs(psf[j] - rpsf[j]))
        assert err <= TOL_PSF, (what, j, err)
        assert abs(strehl[j][0] - rstrehl[j][0]) <= TOL_REF, (what, j, strehl[j][0] - rstrehl[j][0])
        # the peak: the device's own maximum at its lowest index, within the tolerance of the reference maximum
        assert peak[j] == int(np.argmax(psf[j])) and strehl[j][1] == psf[j].ravel()[peak[j]], (what, j)
        assert abs(strehl[j][1] - rstrehl[j][1]) <= TOL_PSF
        assert np.array_equal(psf[j], psf[j][:, ::-1]), (what, j)      # both mirrored columns carry the same value


def _synthetic(rng, n_sets, ny, nx, w_amp=3.0, keep=0.85, per_set_ys=True):
    opd = rng.uniform(-w_amp, w_amp, (n_sets, ny * nx))
    mask = (rng.random((n_sets, ny * nx)) < keep).astype(np.uint8)
    mask[rng.random((n_sets, ny * nx)) < 0.03] = 2                  # a mask value other than 1 is not kept
    ys = np.sort(rng.uniform(-2.0, 2.5, (n_sets if per_set_ys else 1, ny)), axis=1)[:, ::-1]
    ys = ys if per_set_ys else ys[0]
    xs = np.linspace(0.0, 2.2, nx)
    return opd, mask, ys, xs


SIZES = [(1, 1), (2, 3), (7, 8), (64, 65), (129, 128), (255, 255), (1024, 1024)]
GRIDS = [(1, 17), (23, 1), (37, 29), (301, 150)]


@pytest.mark.parametrize("grid", GRIDS, ids=lambda g: f"{g[0]}x{g[1]}")
@pytest.mark.parametrize("size", SIZES, ids=lambda z: f"{z[0]}x{z[1]}")
def test_synthetic_sets(ctx, ort, size, grid):
    n_u, n_v = size
    ny, nx = grid
    rng = np.random.default_rng(n_u * 7 + n_v * 13 + ny * 31 + nx)
    opd, mask, ys, xs = _synthetic(rng, 3, ny, nx, per_set_ys=(ny + nx) % 2 == 0)
    st = _stats(ort, (mask == 1).sum(axis=1))
    du, dv, s = 0.9 / max(n_u, 1) * 1.3, 0.8 / max(n_v, 1) * 1.1, 1.7
    got = _dev(ctx, ort, opd, mask, st, ys, xs, n_u, n_v, du, dv, s)
    _check(got, pr.sets_psf(opd, mask, st, ys, xs, n_u, n_v, du, dv, s), (size, grid))


def test_32_sets_and_statuses(ctx, ort):
    """32 sets: n = 0, n = 1, a NaN opd on a dropped ray (ignored) and on a kept ray (status 3), |W| up to 1e6 waves"""
    rng = np.random.default_rng(11)
    ny, nx, n_u, n_v = 41, 23, 33, 30
    opd, mask, ys, xs = _synthetic(rng, 32, ny, nx)
    opd[5:9] = rng.uniform(-1e6, 1e6, (4, ny * nx))
    mask[0] = 0                                                      # n = 0: status 1
    mask[1] = 0
    mask[1, 17] = 1                                                  # n = 1: one kept ray
    opd[2, np.flatnonzero(mask[2] != 1)[:5]] = np.nan                # dropped NaN rays: ignored
    opd[3, np.flatnonzero(mask[3] == 1)[7]] = np.nan                 # a kept NaN: status 3
    opd[4, np.flatnonzero(mask[4] == 1)[3]] = np.inf
    st = _stats(ort, (mask == 1).sum(axis=1))
    got = _dev(ctx, ort, opd, mask, st, ys, xs, n_u, n_v, 0.031, 0.029, 2.3)
    ref = pr.sets_psf(opd, mask, st, ys, xs, n_u, n_v, 0.031, 0.029, 2.3)
    assert list(got[3][:5]) == [1, 0, 0, 3, 3] and np.all(got[3][5:] == 0)
    _check(got, ref, "32 sets")
    # a small case in extended precision: the float64 reference is not the limit of the comparison
    lref = pr.sets_psf(opd[5:7, :], mask[5:7], st[5:7], ys[5:7], xs, n_u, n_v, 0.031, 0.029, 2.3, dtype=np.longdouble)
    _check(tuple(g[5:7] for g in got), lref, "longdouble")


# ---- traced OPD sweeps -----------------------------------------------------------------------------------------------
SYSTEMS = ("COOKE", "DOUBLE_GAUSS", "REFLECTIVE", "PARABOLA")


def _sweep(ctx, ort, name, arith, vignette, Hs=(0.0, 0.7, 1.0), k_rays=96):
    """the OPD sweep of psf() on the device, full grid, into torch buffers -> (s, p, xs, ys, flds, ext, tensors)"""
    import torch
    P = getattr(ort.prescriptions, name)
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, k_rays, None, vignette, ctx, "test")
    nf, NN = len(flds), ys.shape[1] * len(xs)
    out = {"opd": torch.full((nf, NN), -7.0, dtype=torch.float64, device="cuda"),
           "mask": torch.zeros((nf, NN), dtype=torch.uint8, device="cuda"),
           "stats": torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device="cuda")}
    d_ys, d_xs = _tensor(ys), _tensor(xs)
    ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), ys.shape[1], d_xs.data_ptr(), len(xs), p["stop"], p["a_stop"],
                         {k: v.data_ptr() for k, v in out.items()}, arith=arith, compact=False, ys_per_field=True,
                         ext=ext, opd_scale=-1.0 / LAM)
    torch.cuda.synchronize()
    out["ys"], out["xs"] = d_ys, d_xs
    return s, p, xs, ys, flds, ext, out


def _psf_dev(ctx, out, ny, nx, n_u, n_v, du, dv, sc):
    import torch
    nf = out["opd"].shape[0]
    res = _outs(nf, n_u, n_v)
    sets = dict(n_sets=nf, stride=ny * nx, opd=out["opd"].data_ptr(), mask=out["mask"].data_ptr(),
                stats=out["stats"].data_ptr())
    ctx.wavefront_psf_dev(sets, out["ys"].data_ptr(), 1, ny, out["xs"].data_ptr(), nx, n_u, n_v, du, dv, sc,
                          *[o.data_ptr() for o in res])
    torch.cuda.synchronize()
    return tuple(o.cpu().numpy() for o in res)


@pytest.mark.parametrize("vignette", [False, True])
@pytest.mark.parametrize("arith", ["FAST", "STRICT"])
@pytest.mark.parametrize("name", SYSTEMS)
def test_traced_sweeps(ctx, ort, name, arith, vignette):
    ar = getattr(ort, arith)
    k = 96
    s, p, xs, ys, flds, ext, out = _sweep(ctx, ort, name, ar, vignette, k_rays=k)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    opd, mask = out["opd"].cpu().numpy(), out["mask"].cpu().numpy()
    sc = 1.0 / (LAM * s.f)
    pitch = 1.0 / (4.0 * sc * p["y_EP"])
    for n_u, n_v in ((k - 1, k - 1), (40, 17)):
        got = _psf_dev(ctx, out, ys.shape[1], len(xs), n_u, n_v, pitch, pitch, sc)
        assert np.all(got[3] == 0), got[3]
        _check(got, pr.sets_psf(opd, mask, stats, ys, xs, n_u, n_v, pitch, pitch, sc), (name, arith, vignette))
        # the host form runs the same sweep full grid and the same kernels: the same bytes, statistics included
        h = ctx.trace3d_psf(flds, ys, xs, p["stop"], p["a_stop"], n_u, n_v, pitch, pitch, sc, arith=ar, ext=ext,
                            opd_scale=-1.0 / LAM)
        assert h["stats"].tobytes() == stats.tobytes()
        for a, b in zip((h["psf"], h["strehl"], h["peak"], h["status"]), got):
            assert a.tobytes() == b.tobytes()
    if name == "COOKE":
        # psf() is the host form at the default pixel grid (it leaves no apertures set behind it)
        f = ort.psf(s.layout, s, (0.0, 0.7, 1.0), k_rays=k, vignette=vignette, backend=ctx, arith=ar)
        got = _psf_dev(ctx, out, ys.shape[1], len(xs), k - 1, k - 1, pitch, pitch, sc)
        assert np.array_equal(np.stack([x.psf for x in f]), got[0])
        assert [x.strehl for x in f] == list(got[1][:, 0]) and [x.peak for x in f] == list(got[1][:, 1])
    ctx.set_apertures(None)


def test_mirror_centroid(ctx, ort):
    """REFLECTIVE H = 1, k_rays = 1024: the PSF centroid against the geometric spot centroid, both relative to the chief
    ray's image point, within 0.05 x the geometric RMS radius.  The spot (RMS 0.375 mm) is wider than the default grid
    (+-0.5 mm), so the grid is one whole alias period, +-1.01 mm: 1021 pixels of lam F#"""
    P = ort.prescriptions.REFLECTIVE
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    k = 1024
    p = ort.host._full_trace_setup(s.layout, s, [1.0], k, None, ctx)
    x = ort.psf(s.layout, s, [1.0], k_rays=k, n_pix=1021, pixel=LAM * s.f / (2 * p["y_EP"]), backend=ctx)[0]
    e = ort.full_trace(s.layout, s, 1.0, k, backend=ctx)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [1.0], k, None, False, ctx, "test")
    ctx.set_apertures(None)
    geo = float(np.mean(e.y)) + flds[0]["h_prime"] - flds[0]["opd_yc"]
    cen = float((x.psf.sum(axis=1) @ x.v) / x.psf.sum())
    assert x.status == 0 and abs(cen - geo) < 0.05 * e.RMS, (cen, geo, e.RMS)


def test_bench_size(ctx, ort):
    """the bench grid: double-Gauss, 5792 x 2896 rays x 5 fields, FAST; the field H = 1 at n_pix 127 against psf_ref on
    the copied-back outputs"""
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    s, p, xs, ys, flds, ext, out = _sweep(ctx, ort, "DOUBLE_GAUSS", ort.FAST, False, Hs, 5792)
    assert ys.shape[1] * len(xs) == 5792 * 2896
    sc = 1.0 / (LAM * s.f)
    pitch = 1.0 / (4.0 * sc * p["y_EP"])
    got = _psf_dev(ctx, out, ys.shape[1], len(xs), 127, 127, pitch, pitch, sc)
    assert np.all(got[3] == 0)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    f = len(Hs) - 1
    ref = pr.set_psf(out["opd"][f].cpu().numpy(), out["mask"][f].cpu().numpy(), int(stats[f]["n_kept"]), ys[f], xs, 127,
                     127, pitch, pitch, sc)
    _check(tuple(g[f:f + 1] for g in got), tuple(np.array([r]) for r in ref), "bench")


# ---- determinism, enqueue only, validation ---------------------------------------------------------------------------
def _sets_for(ort, n_sets, ny, nx):
    rng = np.random.default_rng(n_sets + ny + nx)
    opd, mask, ys, xs = _synthetic(rng, n_sets, ny, nx)
    t = dict(opd=_tensor(opd), mask=_tensor(mask), ys=_tensor(ys), xs=_tensor(xs),
             stats=_tensor(np.frombuffer(_stats(ort, (mask == 1).sum(axis=1)).tobytes(), dtype=np.uint8)))
    sets = dict(n_sets=n_sets, stride=ny * nx, opd=t["opd"].data_ptr(), mask=t["mask"].data_ptr(),
                stats=t["stats"].data_ptr())
    return sets, t


def _run(ctx, sets, t, ny, nx, n_u, n_v, stream=0):
    out = _outs(sets["n_sets"], n_u, n_v)
    ctx.wavefront_psf_dev(sets, t["ys"].data_ptr(), 1, ny, t["xs"].data_ptr(), nx, n_u, n_v, 0.01, 0.012, 1.5,
                          *[o.data_ptr() for o in out], stream=stream)
    return out


def test_determinism_and_launch_count(ctx, ort):
    import torch
    sets, t = _sets_for(ort, 5, 2000, 1000)
    runs = []
    for _ in range(2):
        out = _run(ctx, sets, t, 2000, 1000, 255, 255)
        torch.cuda.synchronize()
        runs.append(b"".join(o.cpu().numpy().tobytes() for o in out))
    assert runs[0] == runs[1]
    launches = set()
    for n_sets, ny, nx, n_u, n_v in ((1, 1, 1, 1, 1), (5, 2000, 1000, 1024, 3), (32, 50, 40, 64, 64), (3, 7, 900, 9, 1024)):
        sets, t = _sets_for(ort, n_sets, ny, nx)
        l0 = ctx.launch_count()
        _run(ctx, sets, t, ny, nx, n_u, n_v)
        launches.add(ctx.launch_count() - l0)
    torch.cuda.synchronize()
    assert launches == {5}, launches


def test_enqueue_only(ctx, ort):
    import torch
    sets, t = _sets_for(ort, 5, 2000, 1000)
    _run(ctx, sets, t, 2000, 1000, 255, 255)
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        torch.cuda._sleep(int(100e-3 * 2.0e9))           # ~100 ms at ~2 GHz
        t0 = time.perf_counter()
        _run(ctx, sets, t, 2000, 1000, 255, 255, stream=st.cuda_stream)
        dt = time.perf_counter() - t0
    st.synchronize()
    assert dt < 0.02, dt


def test_validation(ctx, ort):
    import torch
    L = ort._lib
    ny, nx = 20, 10
    sets, t = _sets_for(ort, 2, ny, nx)
    ws = lambda **kw: L.WaveSets(*[dict(sets, **kw).get(k) or 0 for k in L.WAVE_SETS_NAMES])
    out = [o.data_ptr() for o in _outs(2, 8, 8)]
    good = dict(n_u=8, n_v=8, du=0.01, dv=0.01, scale=1.0, ys=t["ys"].data_ptr(), xs=t["xs"].data_ptr(), ny=ny, nx=nx,
                psf=out[0], strehl=out[1], peak=out[2], status=out[3])
    cases = [(ws(), dict(n_u=0)), (ws(), dict(n_v=0)), (ws(), dict(n_u=L.PSF_MAX_SIDE + 1)),
             (ws(), dict(n_v=L.PSF_MAX_SIDE + 1)), (ws(), dict(du=0.0)), (ws(), dict(dv=-1.0)), (ws(), dict(du=np.inf)),
             (ws(), dict(dv=np.nan)), (ws(), dict(scale=0.0)), (ws(), dict(scale=-2.0)), (ws(), dict(scale=np.nan)),
             (ws(n_sets=0), {}), (ws(n_sets=L.MAX_FIELDS + 1), {}), (ws(stride=ny * nx + 1), {}), (ws(), dict(ny=0)),
             (ws(), dict(nx=0)), (ws(opd=0), {}), (ws(mask=0), {}), (ws(stats=0), {}), (ws(), dict(ys=0)),
             (ws(), dict(xs=0)), (ws(), dict(psf=0)), (ws(), dict(strehl=0)), (ws(), dict(peak=0)),
             (ws(), dict(status=0))]
    for s_, kw in cases:
        a = dict(good, **kw)
        req = L.PsfReq(a["n_u"], a["n_v"], a["du"], a["dv"], a["scale"])
        l0 = ctx.launch_count()
        rc = ctx.L.ort_wavefront_psf_dev(ctx.h, C.byref(s_), C.c_void_p(a["ys"]), 1, a["ny"], C.c_void_p(a["xs"]),
                                         a["nx"], C.byref(req), *[C.c_void_p(a[k]) for k in ("psf", "strehl", "peak",
                                                                                               "status")], None)
        assert rc == L.ORT_EINVAL, (kw, rc)
        assert ctx.launch_count() == l0
    # the host form: ORT_EXT_OPD required, compaction invalid, gather_stats unsupported, the request checked first
    P = ort.prescriptions.COOKE
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [0.0], 16, None, False, ctx, "test")
    fa, nf = L.make_fields(flds)
    st = np.zeros(1, dtype=ort.STATS_DTYPE)
    ps, sr, pk, ss = np.zeros(64), np.zeros(2), np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
    good = L.PsfReq(8, 8, 0.01, 0.01, 1.0)
    for op, req, code in ((L._opts(ort.FAST, False, True, ext=0), good, L.ORT_EINVAL),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_VIGNETTE), good, L.ORT_EINVAL),
                          (L._opts(ort.FAST, True, True, ext=L.EXT_OPD), good, L.ORT_EINVAL),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_OPD, gather=True), good, L.ORT_EUNSUPPORTED),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_OPD), L.PsfReq(8, 0, 0.01, 0.01, 1.0), L.ORT_EINVAL),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_OPD), L.PsfReq(8, 8, 0.01, 0.01, 0.0), L.ORT_EINVAL)):
        l0 = ctx.launch_count()
        rc = ctx.L.ort_trace3d_psf(ctx.h, fa, nf, L._vp(ys), ys.shape[1], L._vp(xs), len(xs), p["stop"], p["a_stop"],
                                   C.byref(op), C.byref(req), st.ctypes.data, ps.ctypes.data, sr.ctypes.data,
                                   pk.ctypes.data, ss.ctypes.data)
        assert rc == code and ctx.launch_count() == l0, (rc, code)
    ctx.set_apertures(None)
    torch.cuda.synchronize()


def test_abi_struct_sizes(ort):
    assert C.sizeof(ort._lib.PsfReq) == 32


@pytest.mark.skipif(os.environ.get("ORT_POISON_SCRATCH") == "1", reason="already inside the poisoned run")
def test_parity_with_poisoned_scratch():
    env = dict(os.environ, ORT_POISON_SCRATCH="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_psf.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", "synthetic or statuses or traced or determinism"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
