"""Zernike fit of the wavefront on the device (ort_wavefront_zernike_dev, ort_trace3d_zernike) against tests/zernike_ref.py:
synthetic sets of known coefficients at every order, the statuses, the outputs of traced OPD sweeps, the bench-size grid,
and determinism, enqueue-only behaviour, launch counts and validation."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import zernike_ref as zr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAM = 587.5618e-6


def _tensor(a):
    import torch
    return torch.from_numpy(np.array(a, copy=True)).cuda()


def _stats(ort, n_kept, r_max):
    st = np.zeros(len(n_kept), dtype=ort.STATS_DTYPE)
    st["n_kept"], st["r_max"] = n_kept, r_max
    return st


def _dev(ctx, ort, opd, r, th, mask, stats, n_max, r_norm, stream=0):
    """ort_wavefront_zernike_dev on torch copies of [n_sets][stride] arrays -> (coef, resid, status) numpy"""
    import torch
    n_sets, stride = opd.shape
    t = [_tensor(a) for a in (opd, r, th)]
    t_mask = None if mask is None else _tensor(mask.astype(np.uint8))
    t_st = _tensor(np.frombuffer(stats.tobytes(), dtype=np.uint8))
    coef = torch.full((n_sets, zr.n_terms(n_max)), -5.0, dtype=torch.float64, device="cuda")
    resid = torch.full((n_sets, 2), -5.0, dtype=torch.float64, device="cuda")
    status = torch.full((n_sets,), -5, dtype=torch.int32, device="cuda")
    sets = dict(n_sets=n_sets, stride=stride, opd=t[0].data_ptr(), r=t[1].data_ptr(), theta=t[2].data_ptr(),
                mask=0 if t_mask is None else t_mask.data_ptr(), stats=t_st.data_ptr())
    ctx.wavefront_zernike_dev(sets, n_max, r_norm, coef.data_ptr(), resid.data_ptr(), status.data_ptr(), stream)
    torch.cuda.synchronize()
    return coef.cpu().numpy(), resid.cpu().numpy(), status.cpu().numpy()


def _synthetic(rng, n_max, stride, masked, antisym, r_pupil=2.5):
    """one set: rays uniform over a disk of radius r_pupil, W = sum c_j Z_j in longdouble from random c (symmetric terms,
    plus the antisymmetric ones if antisym); -> opd, r, theta, mask, n_kept, r_max, c"""
    r = r_pupil * np.sqrt(rng.uniform(0, 1, stride))
    th = rng.uniform(-np.pi, np.pi, stride)
    mask = (rng.random(stride) < 0.8).astype(np.uint8) if masked else None
    keep = mask == 1 if masked else np.arange(stride) < stride - 37
    n_kept = int(keep.sum())
    r_max = float(r[keep].max())
    c = rng.standard_normal(zr.n_terms(n_max)) * 0.3
    if not antisym:
        c[~zr.symmetric(n_max)] = 0.0
    return r, th, mask, n_kept, r_max, c


def _opd(c, n_max, rho, th):
    return (zr.basis(n_max, rho, th, np.longdouble) @ np.asarray(c, dtype=np.longdouble)).astype(np.float64)


@pytest.mark.parametrize("r_norm", ["explicit", "rmax"])
@pytest.mark.parametrize("masked", [True, False])
@pytest.mark.parametrize("n_max", list(range(13)))
def test_synthetic_sets(ctx, ort, n_max, masked, r_norm):
    """set 0: symmetric terms only, recovered to 1e-11 relative with a residual at rounding level; set 1: antisymmetric
    terms too, equal to the full-basis lstsq of the mirrored set within the tolerance cond(G) gives"""
    rng = np.random.default_rng(100 * n_max + 10 * masked + (r_norm == "rmax"))
    stride = 20011
    sets = [_synthetic(rng, n_max, stride, masked, anti) for anti in (False, True)]
    rn = 2.5 if r_norm == "explicit" else 0.0
    opd = np.zeros((2, stride)); R = np.zeros((2, stride)); TH = np.zeros((2, stride))
    mask = np.zeros((2, stride), dtype=np.uint8) if masked else None
    for s, (r, th, m, n_kept, r_max, c) in enumerate(sets):
        rho = r / (rn if rn > 0 else r_max)
        opd[s], R[s], TH[s] = _opd(c, n_max, rho, th), r, th
        if masked:
            mask[s] = m
    st = _stats(ort, [x[3] for x in sets], [x[4] for x in sets])
    coef, resid, status = _dev(ctx, ort, opd, R, TH, mask, st, n_max, rn)
    assert np.all(status == 0), status
    sym = zr.symmetric(n_max)
    for s, (r, th, m, n_kept, r_max, c) in enumerate(sets):
        assert np.all(coef[s][~sym] == 0.0)
        o, rr, tt = zr.kept(opd[s], R[s], TH[s], None if mask is None else mask[s], n_kept)
        rho = rr / (rn if rn > 0 else r_max)
        if s == 0:
            assert np.max(np.abs(coef[s] - c)) <= 1e-11 * np.max(np.abs(c)), (n_max, coef[s] - c)
            assert resid[s][0] < 1e-13 * np.max(np.abs(c)) * np.sqrt(len(c)) and resid[s][1] < 1e-12 * np.max(np.abs(c)) * len(c)
        else:
            ref = zr.lstsq_mirrored(o, rho, tt, n_max)
            _, G = zr.normal_fit(o, rho, tt, n_max)
            scale = np.sqrt(np.mean(o ** 2))
            tol = zr.cond_tol(G, len(o)) * scale
            assert np.max(np.abs(coef[s] - ref)) <= tol, (n_max, np.max(np.abs(coef[s] - ref)), tol)
            e = o - zr.basis(n_max, rho, tt) @ ref
            assert abs(resid[s][0] - np.sqrt(np.mean(e ** 2))) <= tol * np.sqrt(len(ref))
            assert abs(resid[s][1] - (e.max() - e.min())) <= 4 * tol * len(ref)


def test_statuses(ctx, ort):
    """n_kept of 0, 1 and J_s - 1: status 1; all rays at one radius: 2; a NaN opd on a kept ray: 3 (on a dropped ray: 0)"""
    rng = np.random.default_rng(7)
    n_max, stride = 8, 4000
    Js = int(zr.symmetric(n_max).sum())
    r = np.sqrt(rng.uniform(0, 1, (6, stride)))
    th = rng.uniform(-np.pi, np.pi, (6, stride))
    opd = rng.standard_normal((6, stride))
    r[3] = 0.7                                           # one radius: Z_4 is a multiple of Z_0
    opd[4, 10] = np.nan
    n_kept = [0, 1, Js - 1, stride, stride, stride]
    st = _stats(ort, n_kept, 1.0)
    coef, resid, status = _dev(ctx, ort, opd, r, th, None, st, n_max, 1.0)
    assert list(status) == [1, 1, 1, 2, 3, 0]
    assert np.all(np.isnan(coef[:5])) and np.all(np.isnan(resid[:5]))
    assert np.all(np.isfinite(coef[5])) and np.all(np.isfinite(resid[5]))
    mask = np.ones((6, stride), dtype=np.uint8)
    mask[4, 10] = 0                                       # the NaN is dropped: the set fits
    mask[0], mask[1, 1:], mask[2, Js - 1:] = 0, 0, 0
    st = _stats(ort, mask.sum(axis=1), 1.0)
    _, _, status = _dev(ctx, ort, opd, r, th, mask, st, n_max, 1.0)
    assert list(status) == [1, 1, 1, 2, 0, 0]
    # n_max = 0 fits the mean: one ray is enough, one radius is no obstacle
    coef, resid, status = _dev(ctx, ort, opd[3:4], r[3:4], th[3:4], None, _stats(ort, [1], 1.0), 0, 0.0)
    assert status[0] == 0 and coef[0][0] == opd[3, 0] and resid[0][0] == 0.0


# ---- traced OPD sweeps -----------------------------------------------------------------------------------------------
SYSTEMS = ("COOKE", "DOUBLE_GAUSS", "REFLECTIVE", "PARABOLA")


def _sweep(ctx, ort, name, arith, compact, vignette, Hs=(0.0, 0.7, 1.0), k_rays=96):
    """the OPD sweep of zernike() on the device into torch buffers -> (p, xs, ys, flds, ext, tensors)"""
    import torch
    P = getattr(ort.prescriptions, name)
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, k_rays, None, vignette, ctx, "test")
    nf, NN = len(flds), ys.shape[1] * len(xs)
    out = {k: torch.full((nf, NN), -7.0, dtype=torch.float64, device="cuda") for k in ("opd", "r", "theta")}
    out["mask"] = torch.zeros((nf, NN), dtype=torch.uint8, device="cuda")
    out["stats"] = torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device="cuda")
    d_ys, d_xs = _tensor(ys), _tensor(xs)
    ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), ys.shape[1], d_xs.data_ptr(), len(xs), p["stop"], p["a_stop"],
                         {k: v.data_ptr() for k, v in out.items()}, arith=arith, compact=compact, ys_per_field=True,
                         ext=ext, opd_scale=-1.0 / LAM)
    torch.cuda.synchronize()
    return s, p, xs, ys, flds, ext, out


def _fit_dev(ctx, ort, out, n_max, r_norm, masked):
    import torch
    nf, NN = out["opd"].shape
    coef = torch.zeros((nf, zr.n_terms(n_max)), dtype=torch.float64, device="cuda")
    resid = torch.zeros((nf, 2), dtype=torch.float64, device="cuda")
    status = torch.zeros(nf, dtype=torch.int32, device="cuda")
    sets = dict(n_sets=nf, stride=NN, opd=out["opd"].data_ptr(), r=out["r"].data_ptr(), theta=out["theta"].data_ptr(),
                mask=out["mask"].data_ptr() if masked else 0, stats=out["stats"].data_ptr())
    ctx.wavefront_zernike_dev(sets, n_max, r_norm, coef.data_ptr(), resid.data_ptr(), status.data_ptr())
    torch.cuda.synchronize()
    return coef.cpu().numpy(), resid.cpu().numpy(), status.cpu().numpy()


@pytest.mark.parametrize("vignette", [False, True])
@pytest.mark.parametrize("compact", [False, True])
@pytest.mark.parametrize("arith", ["FAST", "STRICT"])
@pytest.mark.parametrize("name", SYSTEMS)
def test_traced_sweeps(ctx, ort, name, arith, compact, vignette):
    ar = getattr(ort, arith)
    s, p, xs, ys, flds, ext, out = _sweep(ctx, ort, name, ar, compact, vignette)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    arr = {k: out[k].cpu().numpy() for k in ("opd", "r", "theta", "mask")}
    for n_max, r_norm in ((8, p["a_stop"]), (12, 0.0)):
        coef, resid, status = _fit_dev(ctx, ort, out, n_max, r_norm, not compact)
        for f in range(len(flds)):
            st = stats[f]
            o, rr, tt = zr.kept(arr["opd"][f], arr["r"][f], arr["theta"][f], None if compact else arr["mask"][f],
                                int(st["n_kept"]))
            rho = rr / (r_norm if r_norm > 0 else float(st["r_max"]))
            ref, G = zr.normal_fit(o, rho, tt, n_max)
            assert ref is not None and status[f] == 0, (name, f, status)
            scale = max(np.sqrt(np.mean(o ** 2)), 1e-12)
            tol = zr.cond_tol(G, len(o)) * scale
            assert np.max(np.abs(coef[f] - ref)) <= tol, (name, n_max, f, np.max(np.abs(coef[f] - ref)), tol)
            rms, pv = zr.residual(o, rho, tt, n_max, ref)
            assert abs(resid[f][0] - rms) <= tol * np.sqrt(len(ref)) and abs(resid[f][1] - pv) <= 4 * tol * len(ref)
        if compact:
            continue
        # the host form runs the same sweep full grid and the same kernels: the same bytes, statistics included
        h = ctx.trace3d_zernike(flds, ys, xs, p["stop"], p["a_stop"], n_max, r_norm, arith=ar, ext=ext,
                                opd_scale=-1.0 / LAM)
        assert h["stats"].tobytes() == stats.tobytes()
        assert h["coef"].tobytes() == coef.tobytes() and h["resid"].tobytes() == resid.tobytes()
        assert h["status"].tobytes() == status.tobytes()
    if name == "COOKE" and not compact:
        # zernike() is the host form at norm "rmax" (it leaves no apertures set behind it)
        z = ort.zernike(s.layout, s, (0.0, 0.7, 1.0), n_max=12, k_rays=96, vignette=vignette, norm="rmax", backend=ctx,
                        arith=ar)
        assert np.array_equal(np.stack([x.coef for x in z]), coef)
        assert np.array_equal(np.array([[x.rms_resid, x.pv_resid] for x in z]), resid)
        assert [x.status for x in z] == list(status) and [x.n_kept for x in z] == list(stats["n_kept"])
    ctx.set_apertures(None)


def test_bench_size(ctx, ort):
    """the bench grid: double-Gauss, 5792 x 2896 rays x 5 fields, FAST, n_max 8 and 12 against the longdouble
    normal equations of the copied-back outputs (the n_max 8 system is the leading block of the n_max 12 one), and the
    residual of a second pass over them (the quadratic form sum W^2 - 2 c^T b + c^T G c cancels to noise here: the
    piston is ~4.5 waves, the residual ~6e-8)"""
    import torch
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    s, p, xs, ys, flds, ext, out = _sweep(ctx, ort, "DOUBLE_GAUSS", ort.FAST, False, False, Hs, 5792)
    assert ys.shape[1] * len(xs) == 5792 * 2896
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    fits = {n: _fit_dev(ctx, ort, out, n, p["a_stop"], True) for n in (8, 12)}
    for f in range(len(Hs)):
        m = out["mask"][f].cpu().numpy() == 1
        o = out["opd"][f].cpu().numpy()[m]
        rho = out["r"][f].cpu().numpy()[m] / p["a_stop"]
        tt = out["theta"][f].cpu().numpy()[m]
        G, b = zr.normal_equations(o, rho, tt, 12, chunk=1 << 17, basis_dtype=np.float64)
        for n_max, (coef, resid, status) in fits.items():
            Js = int(zr.symmetric(n_max).sum())
            ref = zr.solve_normal(G, b, n_max)
            assert status[f] == 0 and ref is not None
            scale = np.sqrt(np.mean(o ** 2))
            tol = zr.cond_tol(G[:Js, :Js].astype(np.float64), len(o)) * scale
            assert np.max(np.abs(coef[f] - ref)) <= tol, (f, n_max, np.max(np.abs(coef[f] - ref)), tol)
            rms, pv = zr.residual(o, rho, tt, n_max, ref, chunk=1 << 17, dtype=np.float64)
            assert abs(resid[f][0] - rms) <= tol * np.sqrt(Js) and abs(resid[f][1] - pv) <= 4 * tol * Js, (f, n_max)


# ---- determinism, enqueue only, validation ---------------------------------------------------------------------------
def _sets_for(ort, n_sets, stride, n_max=8):
    import torch
    rng = np.random.default_rng(n_sets + stride)
    t = [_tensor(a) for a in (rng.standard_normal((n_sets, stride)), np.sqrt(rng.uniform(0, 1, (n_sets, stride))),
                              rng.uniform(-np.pi, np.pi, (n_sets, stride)))]
    st = _tensor(np.frombuffer(_stats(ort, [stride] * n_sets, [1.0] * n_sets).tobytes(), dtype=np.uint8))
    J = zr.n_terms(ort._lib.ZERN_MAX_ORDER)
    out = (torch.zeros((n_sets, J), dtype=torch.float64, device="cuda"),
           torch.zeros((n_sets, 2), dtype=torch.float64, device="cuda"), torch.zeros(n_sets, dtype=torch.int32, device="cuda"))
    sets = dict(n_sets=n_sets, stride=stride, opd=t[0].data_ptr(), r=t[1].data_ptr(), theta=t[2].data_ptr(), mask=0,
                stats=st.data_ptr())
    return sets, out, (t, st)


def test_determinism_and_launch_count(ctx, ort):
    import torch
    sets, out, _keep = _sets_for(ort, 5, 1 << 21)
    runs = []
    for _ in range(2):
        ctx.wavefront_zernike_dev(sets, 12, 0.0, *[o.data_ptr() for o in out])
        torch.cuda.synchronize()
        runs.append(b"".join(o.cpu().numpy().tobytes() for o in out))
    assert runs[0] == runs[1]
    launches = set()
    for n_sets, stride, n_max in ((1, 10, 0), (5, 1 << 21, 12), (32, 5000, 8), (3, 100, 3)):
        sets, out, _keep = _sets_for(ort, n_sets, stride)
        l0 = ctx.launch_count()
        ctx.wavefront_zernike_dev(sets, n_max, 1.0, *[o.data_ptr() for o in out])
        launches.add(ctx.launch_count() - l0)
    torch.cuda.synchronize()
    assert launches == {4}, launches


def test_enqueue_only(ctx, ort):
    import torch
    sets, out, _keep = _sets_for(ort, 5, 1 << 22)
    ctx.wavefront_zernike_dev(sets, 8, 0.0, *[o.data_ptr() for o in out])
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        torch.cuda._sleep(int(100e-3 * 2.0e9))           # ~100 ms at ~2 GHz
        t0 = time.perf_counter()
        ctx.wavefront_zernike_dev(sets, 8, 0.0, *[o.data_ptr() for o in out], stream=st.cuda_stream)
        dt = time.perf_counter() - t0
    st.synchronize()
    assert dt < 0.02, dt


def test_validation(ctx, ort):
    import torch
    L = ort._lib
    sets, out, _keep = _sets_for(ort, 2, 1000)
    ws = lambda **kw: L.WaveSets(*[dict(sets, **kw).get(k) or 0 for k in L.WAVE_SETS_NAMES])
    ptrs = [o.data_ptr() for o in out]
    cases = [(ws(), dict(n_max=13)), (ws(), dict(n_max=-1)), (ws(), dict(r_norm=-1.0)), (ws(), dict(r_norm=np.inf)),
             (ws(), dict(r_norm=np.nan)), (ws(n_sets=0), {}), (ws(n_sets=L.MAX_FIELDS + 1), {}), (ws(stride=0), {}),
             (ws(stride=-3), {}), (ws(stride=1 << 31), {}), (ws(opd=0), {}), (ws(r=0), {}), (ws(theta=0), {}),
             (ws(stats=0), {}), (ws(), dict(coef=0)), (ws(), dict(resid=0)), (ws(), dict(status=0))]
    for s_, kw in cases:
        a = dict(n_max=8, r_norm=1.0, coef=ptrs[0], resid=ptrs[1], status=ptrs[2])
        a.update(kw)
        req = L.ZernikeReq(a["n_max"], 0, a["r_norm"])
        l0 = ctx.launch_count()
        rc = ctx.L.ort_wavefront_zernike_dev(ctx.h, C.byref(s_), C.byref(req), C.c_void_p(a["coef"]),
                                             C.c_void_p(a["resid"]), C.c_void_p(a["status"]), None)
        assert rc == L.ORT_EINVAL, (kw, rc)
        assert ctx.launch_count() == l0
    # the host form: ORT_EXT_OPD required, compaction invalid, gather_stats unsupported, the request checked first
    P = ort.prescriptions.COOKE
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, [0.0], 16, None, False, ctx, "test")
    fa, nf = L.make_fields(flds)
    st = np.zeros(1, dtype=ort.STATS_DTYPE)
    cf, rs, ss = np.zeros(zr.n_terms(12)), np.zeros(2), np.zeros(1, dtype=np.int32)
    good = L.ZernikeReq(8, 0, 1.0)
    for op, req, code in ((L._opts(ort.FAST, False, True, ext=0), good, L.ORT_EINVAL),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_VIGNETTE), good, L.ORT_EINVAL),
                          (L._opts(ort.FAST, True, True, ext=L.EXT_OPD), good, L.ORT_EINVAL),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_OPD, gather=True), good, L.ORT_EUNSUPPORTED),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_OPD), L.ZernikeReq(13, 0, 1.0), L.ORT_EINVAL)):
        l0 = ctx.launch_count()
        rc = ctx.L.ort_trace3d_zernike(ctx.h, fa, nf, L._vp(ys), ys.shape[1], L._vp(xs), len(xs), p["stop"], p["a_stop"],
                                       C.byref(op), C.byref(req), st.ctypes.data, cf.ctypes.data, rs.ctypes.data,
                                       ss.ctypes.data)
        assert rc == code and ctx.launch_count() == l0, (rc, code)
    ctx.set_apertures(None)
    torch.cuda.synchronize()


def test_abi_struct_sizes(ort):
    assert C.sizeof(ort._lib.ZernikeReq) == 16
    assert C.sizeof(ort._lib.WaveSets) == 56


@pytest.mark.skipif(os.environ.get("ORT_POISON_SCRATCH") == "1", reason="already inside the poisoned run")
def test_parity_with_poisoned_scratch():
    env = dict(os.environ, ORT_POISON_SCRATCH="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_zernike.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", "synthetic or statuses or traced or determinism"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
