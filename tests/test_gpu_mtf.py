"""Diffraction MTF of the wavefront on the device (ort_wavefront_mtf_dev, ort_trace3d_mtf) against tests/mtf_ref.py:
synthetic sets at edge sizes and statuses, the tilt property, the outputs of traced OPD sweeps, the device PSF, the
bench-size grid, and determinism, enqueue-only behaviour, launch counts and validation."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import mtf_ref as mr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAM = 587.5618e-6
TOL = 1e-12


def _tensor(a):
    import torch
    return torch.from_numpy(np.array(a, copy=True)).cuda()


def _stats(ort, n_kept):
    st = np.zeros(len(n_kept), dtype=ort.STATS_DTYPE)
    st["n_kept"] = n_kept
    return st


def _outs(n_sets, n_freq):
    import torch
    return (torch.full((n_sets, 2, n_freq, 2), -5.0, dtype=torch.float64, device="cuda"),
            torch.full((n_sets,), -5, dtype=torch.int32, device="cuda"))


def _dev(ctx, ort, opd, mask, stats, ys, xs, freqs, s, stream=0):
    """ort_wavefront_mtf_dev on torch copies of [n_sets][ny * nx] arrays -> (otf (n_sets, 2, n_freq) complex, status)"""
    import torch
    n_sets, stride = opd.shape
    ys = np.asarray(ys, dtype=np.float64)
    t_opd, t_mask = _tensor(opd), _tensor(mask.astype(np.uint8))
    t_st = _tensor(np.frombuffer(stats.tobytes(), dtype=np.uint8))
    t_ys, t_xs = _tensor(ys), _tensor(np.asarray(xs, dtype=np.float64))
    otf, status = _outs(n_sets, len(freqs))
    sets = dict(n_sets=n_sets, stride=stride, opd=t_opd.data_ptr(), mask=t_mask.data_ptr(), stats=t_st.data_ptr())
    ctx.wavefront_mtf_dev(sets, t_ys.data_ptr(), ys.ndim == 2, ys.shape[-1], t_xs.data_ptr(), len(xs), freqs, s,
                          otf.data_ptr(), status.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    o = otf.cpu().numpy()
    return o[..., 0] + 1j * o[..., 1], status.cpu().numpy()


def _check(got, ref, what="", tol=TOL):
    otf, status = got
    rotf, rstatus = ref
    assert np.array_equal(status, rstatus), (what, status, rstatus)
    for j in range(len(status)):
        if status[j]:
            assert np.all(np.isnan(otf[j].real)) and np.all(np.isnan(otf[j].imag)), (what, j)
            continue
        err = np.max(np.abs(otf[j] - rotf[j]))
        assert err <= tol, (what, j, err)
        assert np.all(otf[j][0].imag == 0.0), (what, j)
        assert np.all(np.abs(otf[j]) <= 1 + 1e-12), (what, j)


def _lattice(rng, n, d, per_set, n_sets):
    """ys: (n,) or (n_sets, n) lattices of step +-d with random origins (descending or ascending)"""
    rows = [rng.uniform(-2, 2) + np.arange(n) * d * (1 if rng.random() < 0.5 else -1) for _ in range(n_sets)]
    return np.stack(rows) if per_set else rows[0]


def _synthetic(rng, n_sets, ny, nx, w_amp=3.0, keep=0.85, per_set_ys=True):
    opd = rng.uniform(-w_amp, w_amp, (n_sets, ny * nx))
    mask = (rng.random((n_sets, ny * nx)) < keep).astype(np.uint8)
    mask[rng.random((n_sets, ny * nx)) < 0.03] = 2                  # a mask value other than 1 is not kept
    ys = _lattice(rng, ny, 0.037, per_set_ys, n_sets)
    xs = np.arange(nx) * 0.041
    return opd, mask, ys, xs


def _freqs(rng, s, dx, dy, nx, ny, n=None):
    """on, between and past lattice lags of both azimuths, unsorted"""
    f = [np.arange(0, 2 * nx + 1) * s * dx, rng.uniform(0, 2.3 * nx * s * dx, 12),
         np.arange(0, ny + 1) * s * dy, rng.uniform(0, 1.2 * ny * s * dy, 12), [0.0, 1e30]]
    f = rng.permutation(np.concatenate(f))
    return f[:n] if n else f


GRIDS = [(2, 2), (3, 2), (9, 7), (64, 33), (301, 5), (4, 517), (130, 96), (6150, 3), (2, 6145)]   # the last two: rows
# longer than the shared-memory stage (6144), read from global memory


@pytest.mark.parametrize("grid", GRIDS, ids=lambda g: f"{g[0]}x{g[1]}")
def test_synthetic_sets(ctx, ort, grid):
    ny, nx = grid
    rng = np.random.default_rng(ny * 31 + nx)
    opd, mask, ys, xs = _synthetic(rng, 3, ny, nx, per_set_ys=(ny + nx) % 2 == 1)
    st = _stats(ort, (mask == 1).sum(axis=1))
    s = 1.7
    freqs = _freqs(rng, s, 0.041, 0.037, nx, ny, n=ort._lib.MTF_MAX_FREQS)
    got = _dev(ctx, ort, opd, mask, st, ys, xs, freqs, s)
    assert np.all(got[1] == 0)
    _check(got, mr.sets_otf(opd, mask, st, ys, xs, freqs, s), grid)
    if ny * nx <= 64:                                                # the explicit multiset in extended precision
        _check(got, mr.sets_otf(opd, mask, st, ys, xs, freqs, s, "brute", np.longdouble), (grid, "brute"))


def test_32_sets_and_statuses(ctx, ort):
    """32 sets: n = 0, n = 1, a NaN opd on a dropped ray (ignored) and on a kept ray (status 3), a zero and a NaN y step
    (status 4), |W| up to 1e6 waves; then an x grid that does not start at 0 (status 4 for every set with rays)"""
    rng = np.random.default_rng(11)
    ny, nx = 41, 23
    opd, mask, ys, xs = _synthetic(rng, 32, ny, nx)
    opd[7:11] = rng.uniform(-1e6, 1e6, (4, ny * nx))
    mask[0] = 0                                                      # n = 0: status 1
    mask[1] = 0
    mask[1, 17] = 1                                                  # n = 1: one kept ray
    opd[2, np.flatnonzero(mask[2] != 1)[:5]] = np.nan                # dropped NaN rays: ignored
    opd[3, np.flatnonzero(mask[3] == 1)[7]] = np.nan                 # a kept NaN: status 3
    opd[4, np.flatnonzero(mask[4] == 1)[3]] = np.inf
    ys[5] = 0.25                                                     # dy = 0: status 4
    ys[6, -1] = np.nan                                               # dy not finite: status 4
    ys[12, :] = ys[12, ::-1].copy()
    st = _stats(ort, (mask == 1).sum(axis=1))
    freqs = _freqs(rng, 2.3, 0.041, 0.037, nx, ny, n=200)
    got = _dev(ctx, ort, opd, mask, st, ys, xs, freqs, 2.3)
    assert list(got[1][:7]) == [1, 0, 0, 3, 3, 4, 4] and np.all(got[1][7:] == 0)
    _check(got, mr.sets_otf(opd, mask, st, ys, xs, freqs, 2.3), "32 sets")
    for bad_xs in (xs + 1e-3, xs[::-1].copy(), -xs):
        got = _dev(ctx, ort, opd, mask, st, ys, bad_xs, freqs, 2.3)
        assert got[1][0] == 1 and list(got[1][3:5]) == [3, 3] and np.all(got[1][5:] == 4), got[1]


@pytest.mark.parametrize("sign", [1, -1])
def test_tilt_property(ctx, ort, sign):
    """W + t iy multiplies the tangential OTF at lag k by exp(+-2 pi i t k) (the sign of dy) and leaves the sagittal OTF
    unchanged"""
    rng = np.random.default_rng(17)
    ny, nx, s, t = 90, 40, 1.3, 0.137
    opd, mask, _, xs = _synthetic(rng, 2, ny, nx)
    ys = sign * (0.5 + np.arange(ny) * 0.037)
    st = _stats(ort, (mask == 1).sum(axis=1))
    dx, dy = mr.steps(ys, xs)
    ks = np.arange(ny)
    freqs = np.concatenate([ks * s * abs(dy), np.arange(2 * nx - 1) * s * dx])
    a = _dev(ctx, ort, opd, mask, st, ys, xs, freqs, s)
    b = _dev(ctx, ort, opd + t * np.repeat(np.arange(ny), nx)[None, :], mask, st, ys, xs, freqs, s)
    assert np.all(a[1] == 0) and np.all(b[1] == 0)
    rot = np.exp(sign * 2j * np.pi * t * ks)
    assert np.max(np.abs(b[0][:, 1, :ny] - a[0][:, 1, :ny] * rot[None, :])) < 1e-12
    assert np.max(np.abs(b[0][:, 0] - a[0][:, 0])) < 1e-12
    assert np.max(np.abs(a[0][:, 1, 1:ny].imag)) > 1e-3


# ---- traced OPD sweeps -----------------------------------------------------------------------------------------------
SYSTEMS = ("COOKE", "DOUBLE_GAUSS", "REFLECTIVE", "PARABOLA")


def _sweep(ctx, ort, name, arith, vignette, Hs=(0.0, 0.7, 1.0), k_rays=96):
    """the OPD sweep of mtf() on the device, full grid, into torch buffers -> (s, p, xs, ys, flds, ext, tensors)"""
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


def _mtf_dev(ctx, out, ny, nx, freqs, sc):
    import torch
    nf = out["opd"].shape[0]
    otf, status = _outs(nf, len(freqs))
    sets = dict(n_sets=nf, stride=ny * nx, opd=out["opd"].data_ptr(), mask=out["mask"].data_ptr(),
                stats=out["stats"].data_ptr())
    ctx.wavefront_mtf_dev(sets, out["ys"].data_ptr(), 1, ny, out["xs"].data_ptr(), nx, freqs, sc, otf.data_ptr(),
                          status.data_ptr())
    torch.cuda.synchronize()
    o = otf.cpu().numpy()
    return o[..., 0] + 1j * o[..., 1], status.cpu().numpy()


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
    nu_c = 2.0 * sc * p["y_EP"]
    rng = np.random.default_rng(len(name))
    freqs = np.concatenate([np.linspace(0.0, nu_c, 32), rng.uniform(0.0, 1.1 * nu_c, 16)])
    got = _mtf_dev(ctx, out, ys.shape[1], len(xs), freqs, sc)
    assert np.all(got[1] == 0), got[1]
    _check(got, mr.sets_otf(opd, mask, stats, ys, xs, freqs, sc), (name, arith, vignette))
    # the host form runs the same sweep full grid and the same kernels: the same bytes, statistics included
    h = ctx.trace3d_mtf(flds, ys, xs, p["stop"], p["a_stop"], freqs, sc, arith=ar, ext=ext, opd_scale=-1.0 / LAM)
    assert h["stats"].tobytes() == stats.tobytes()
    assert h["otf"].tobytes() == got[0].tobytes() and h["status"].tobytes() == got[1].tobytes()
    if name == "COOKE":
        # mtf() is the host form (it leaves no apertures set behind it)
        f = ort.mtf(s.layout, s, (0.0, 0.7, 1.0), freqs=freqs, k_rays=k, vignette=vignette, backend=ctx, arith=ar)
        assert np.array_equal(np.stack([x.otf for x in f]), got[0])
    ctx.set_apertures(None)


def test_otf_is_the_transform_of_the_device_psf(ctx, ort):
    """the device MTF at lattice frequencies against the normalised DFT of the device PSF over one alias period
    (n_u = 4 nx - 3, n_v = 2 ny - 1 pixels of 1 / (s d n)); Cooke at H = 0.8, k_rays = 64"""
    P = ort.prescriptions.COOKE
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    k, H = 64, 0.8
    sc = 1.0 / (LAM * s.f)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [H], k, None, False, ctx, "test")
    ctx.set_apertures(None)
    dx, dy = mr.steps(ys[0], xs)
    nx, ny = len(xs), ys.shape[1]
    n_u, n_v = 4 * nx - 3, 2 * ny - 1
    x = ort.psf(s.layout, s, [H], n_pix=(n_u, n_v), pixel=(1 / (sc * dx * n_u), 1 / (sc * abs(dy) * n_v)), k_rays=k,
                backend=ctx)[0]
    ks, kt = np.arange(2 * nx - 1), np.arange(ny)
    nu_s, nu_t = ks * sc * dx, kt * sc * abs(dy)
    dft_s = (x.psf.sum(axis=0) @ np.exp(-2j * np.pi * nu_s[None, :] * x.u[:, None])) / x.psf.sum()
    dft_t = (x.psf.sum(axis=1) @ np.exp(-2j * np.pi * nu_t[None, :] * x.v[:, None])) / x.psf.sum()
    m = ort.mtf(s.layout, s, [H], freqs=np.concatenate([nu_s, nu_t]), k_rays=k, backend=ctx)[0]
    assert x.status == 0 and m.status == 0
    assert np.max(np.abs(m.otf[0][:len(ks)] - dft_s)) < 1e-10
    assert np.max(np.abs(m.otf[1][len(ks):] - dft_t)) < 1e-10


def test_bench_size(ctx, ort):
    """the bench grid: double-Gauss, 5792 x 2896 rays x 5 fields, FAST; the field H = 1 against the vectorised reference
    on the copied-back outputs at a handful of frequencies"""
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    s, p, xs, ys, flds, ext, out = _sweep(ctx, ort, "DOUBLE_GAUSS", ort.FAST, False, Hs, 5792)
    assert ys.shape[1] * len(xs) == 5792 * 2896
    sc = 1.0 / (LAM * s.f)
    nu_c = 2.0 * sc * p["y_EP"]
    freqs = np.array([0.0, 0.013 * nu_c, 0.25 * nu_c, 0.61 * nu_c, 0.97 * nu_c])
    got = _mtf_dev(ctx, out, ys.shape[1], len(xs), freqs, sc)
    assert np.all(got[1] == 0)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    f = len(Hs) - 1
    ref = mr.set_otf(out["opd"][f].cpu().numpy(), out["mask"][f].cpu().numpy(), int(stats[f]["n_kept"]), ys[f], xs,
                     freqs, sc)
    _check(tuple(g[f:f + 1] for g in got), tuple(np.array([r]) for r in ref), "bench", tol=1e-11)


# ---- determinism, enqueue only, validation ---------------------------------------------------------------------------
def _sets_for(ort, n_sets, ny, nx):
    rng = np.random.default_rng(n_sets + ny + nx)
    opd, mask, ys, xs = _synthetic(rng, n_sets, ny, nx, per_set_ys=False)
    t = dict(opd=_tensor(opd), mask=_tensor(mask), ys=_tensor(ys), xs=_tensor(xs),
             stats=_tensor(np.frombuffer(_stats(ort, (mask == 1).sum(axis=1)).tobytes(), dtype=np.uint8)))
    sets = dict(n_sets=n_sets, stride=ny * nx, opd=t["opd"].data_ptr(), mask=t["mask"].data_ptr(),
                stats=t["stats"].data_ptr())
    return sets, t


def _run(ctx, sets, t, ny, nx, freqs, stream=0, out=None):
    out = _outs(sets["n_sets"], len(freqs)) if out is None else out
    ctx.wavefront_mtf_dev(sets, t["ys"].data_ptr(), 0, ny, t["xs"].data_ptr(), nx, freqs, 1.5,
                          *[o.data_ptr() for o in out], stream=stream)
    return out


def test_determinism_and_launch_count(ctx, ort):
    import torch
    sets, t = _sets_for(ort, 5, 2000, 1000)
    freqs = np.linspace(0.0, 40.0, 32)
    runs = []
    for _ in range(2):
        out = _run(ctx, sets, t, 2000, 1000, freqs)
        torch.cuda.synchronize()
        runs.append(b"".join(o.cpu().numpy().tobytes() for o in out))
    assert runs[0] == runs[1]
    launches = set()
    for n_sets, ny, nx, nf in ((1, 2, 2, 1), (5, 2000, 1000, 1024), (32, 50, 40, 64), (3, 7, 900, 5)):
        sets, t = _sets_for(ort, n_sets, ny, nx)
        l0 = ctx.launch_count()
        _run(ctx, sets, t, ny, nx, np.linspace(0.0, 30.0, nf))
        launches.add(ctx.launch_count() - l0)
    torch.cuda.synchronize()
    assert launches == {4}, launches


def test_enqueue_only(ctx, ort):
    """ort_wavefront_mtf_dev returns while the stream is still busy.  The output tensors are allocated before the timed
    call: torch's first allocation on a new stream can need a cudaMalloc, and when its cache holds most of the device
    (as after the full-size tests) the allocator may free cached blocks first, which waits for the device -- a wait in
    the test, not in the library."""
    import torch
    sets, t = _sets_for(ort, 5, 2000, 1000)
    freqs = np.linspace(0.0, 40.0, 32)
    ref = _run(ctx, sets, t, 2000, 1000, freqs)
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        out = _outs(sets["n_sets"], len(freqs))
        torch.cuda._sleep(int(100e-3 * 2.0e9))           # ~100 ms at ~2 GHz
        t0 = time.perf_counter()
        _run(ctx, sets, t, 2000, 1000, freqs, stream=st.cuda_stream, out=out)
        dt = time.perf_counter() - t0
    st.synchronize()
    assert dt < 0.02, dt
    assert all(torch.equal(a, b) for a, b in zip(out, ref))        # and the enqueued work ran to the same result


def test_validation(ctx, ort):
    import torch
    L = ort._lib
    ny, nx = 20, 10
    sets, t = _sets_for(ort, 2, ny, nx)
    ws = lambda **kw: L.WaveSets(*[dict(sets, **kw).get(k) or 0 for k in L.WAVE_SETS_NAMES])
    out = [o.data_ptr() for o in _outs(2, 3)]
    good = dict(freqs=[0.0, 1.0, 2.0], scale=1.0, ys=t["ys"].data_ptr(), xs=t["xs"].data_ptr(), ny=ny, nx=nx,
                otf=out[0], status=out[1])
    cases = [(ws(), dict(freqs=[])), (ws(), dict(freqs=np.zeros(L.MTF_MAX_FREQS + 1))), (ws(), dict(freqs=[1.0, -1.0])),
             (ws(), dict(freqs=[np.inf])), (ws(), dict(freqs=[np.nan, 1.0])), (ws(), dict(freqs=None)),
             (ws(), dict(scale=0.0)), (ws(), dict(scale=-2.0)), (ws(), dict(scale=np.nan)), (ws(), dict(scale=np.inf)),
             (ws(n_sets=0), {}), (ws(n_sets=L.MAX_FIELDS + 1), {}), (ws(stride=ny * nx + 1), {}),
             (ws(stride=ny * 1), dict(nx=1)), (ws(stride=nx), dict(ny=1)), (ws(opd=0), {}), (ws(mask=0), {}),
             (ws(stats=0), {}), (ws(), dict(ys=0)), (ws(), dict(xs=0)), (ws(), dict(otf=0)), (ws(), dict(status=0))]
    for s_, kw in cases:
        a = dict(good, **kw)
        if a["freqs"] is None:
            req = L.MtfReq(3, 0, None, a["scale"])
        else:
            req, keep = L.mtf_req(a["freqs"], a["scale"])
        l0 = ctx.launch_count()
        rc = ctx.L.ort_wavefront_mtf_dev(ctx.h, C.byref(s_), C.c_void_p(a["ys"]), 0, a["ny"], C.c_void_p(a["xs"]),
                                         a["nx"], C.byref(req), C.c_void_p(a["otf"]), C.c_void_p(a["status"]), None)
        assert rc == L.ORT_EINVAL, (kw, rc)
        assert ctx.launch_count() == l0
    req, keep = L.mtf_req(good["freqs"], 1.0)
    assert ctx.L.ort_wavefront_mtf_dev(ctx.h, C.byref(ws()), C.c_void_p(good["ys"]), 0, ny, C.c_void_p(good["xs"]), nx,
                                       None, C.c_void_p(out[0]), C.c_void_p(out[1]), None) == L.ORT_EINVAL
    # the host form: ORT_EXT_OPD required, compaction invalid, gather_stats unsupported, the request checked first
    P = ort.prescriptions.COOKE
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [0.0], 16, None, False, ctx, "test")
    fa, nf = L.make_fields(flds)
    st = np.zeros(1, dtype=ort.STATS_DTYPE)
    ot, ss = np.zeros(12), np.zeros(1, dtype=np.int32)
    good, k1 = L.mtf_req([0.0, 1.0, 2.0], 1.0)
    neg, k2 = L.mtf_req([0.0, -1.0, 2.0], 1.0)
    zero, k3 = L.mtf_req([0.0, 1.0, 2.0], 0.0)
    for op, req, code, n_x in ((L._opts(ort.FAST, False, True, ext=0), good, L.ORT_EINVAL, len(xs)),
                               (L._opts(ort.FAST, False, True, ext=L.EXT_VIGNETTE), good, L.ORT_EINVAL, len(xs)),
                               (L._opts(ort.FAST, True, True, ext=L.EXT_OPD), good, L.ORT_EINVAL, len(xs)),
                               (L._opts(ort.FAST, False, True, ext=L.EXT_OPD, gather=True), good, L.ORT_EUNSUPPORTED,
                                len(xs)),
                               (L._opts(ort.FAST, False, True, ext=L.EXT_OPD), neg, L.ORT_EINVAL, len(xs)),
                               (L._opts(ort.FAST, False, True, ext=L.EXT_OPD), zero, L.ORT_EINVAL, len(xs)),
                               (L._opts(ort.FAST, False, True, ext=L.EXT_OPD), good, L.ORT_EINVAL, 1)):
        l0 = ctx.launch_count()
        rc = ctx.L.ort_trace3d_mtf(ctx.h, fa, nf, L._vp(ys), ys.shape[1], L._vp(xs), n_x, p["stop"], p["a_stop"],
                                   C.byref(op), C.byref(req), st.ctypes.data, ot.ctypes.data, ss.ctypes.data)
        assert rc == code and ctx.launch_count() == l0, (rc, code)
    ctx.set_apertures(None)
    torch.cuda.synchronize()


def test_abi_struct_sizes(ort):
    assert C.sizeof(ort._lib.MtfReq) == 24


@pytest.mark.skipif(os.environ.get("ORT_POISON_SCRATCH") == "1", reason="already inside the poisoned run")
def test_parity_with_poisoned_scratch():
    env = dict(os.environ, ORT_POISON_SCRATCH="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_mtf.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", "synthetic or statuses or traced or determinism"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
