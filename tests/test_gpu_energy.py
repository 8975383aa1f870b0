"""Encircled / ensquared energy on the device (ort_spot_energy_dev, ort_trace3d_energy) bit for bit against numpy sort /
searchsorted on the same arrays (tests/energy_ref.py): adversarial synthetic sets through torch arrays, the outputs of
traced grid and through-focus sweeps, the bench-size grid, determinism, enqueue-only behaviour and validation."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from energy_ref import distances, set_energy

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stats(ort, n_kept, mean_y):
    st = np.zeros(len(n_kept), dtype=ort.STATS_DTYPE)
    st["n_kept"], st["mean_y"] = n_kept, mean_y
    return st


def _tensor(a):
    import torch
    return torch.from_numpy(np.array(a, copy=True)).cuda()


def _dev(ctx, ort, ex, ey, mask, stats, spm, radii, fracs, metric="circle", center="centroid"):
    """ort_spot_energy_dev on torch copies of ex, ey [n_sets][stride], mask [n_sets / spm][stride] (or None), stats"""
    import torch
    n_sets, stride = ex.shape
    t_ex, t_ey = _tensor(ex), _tensor(ey)
    t_mask = None if mask is None else _tensor(mask.astype(np.uint8))
    t_st = _tensor(np.frombuffer(stats.tobytes(), dtype=np.uint8))
    cnt = torch.full((n_sets, len(radii)), -5, dtype=torch.int64, device="cuda")
    rad = torch.full((n_sets, len(fracs)), -5.0, dtype=torch.float64, device="cuda")
    sets = dict(n_sets=n_sets, sets_per_mask=spm, stride=stride, ex=t_ex.data_ptr(), ey=t_ey.data_ptr(),
                mask=0 if t_mask is None else t_mask.data_ptr(), stats=t_st.data_ptr())
    ctx.spot_energy_dev(sets, radii, fracs, metric, center, cnt.data_ptr() if len(radii) else 0,
                        rad.data_ptr() if len(fracs) else 0)
    torch.cuda.synchronize()
    return cnt.cpu().numpy(), rad.cpu().numpy()


def _ref(ex, ey, mask, stats, spm, radii, fracs, metric, center):
    out = [set_energy(ex[s], ey[s], None if mask is None else mask[s // spm], int(stats[s]["n_kept"]),
                      float(stats[s]["mean_y"]), radii, fracs, metric, center) for s in range(ex.shape[0])]
    return (np.array([o[0] for o in out]).reshape(ex.shape[0], len(radii)),
            np.array([o[1] for o in out]).reshape(ex.shape[0], len(fracs)))


def _same_bits(a, b):
    """the same doubles bit for bit; any NaN equals any NaN"""
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def _check(ctx, ort, ex, ey, mask, stats, spm, radii, fracs, metric, center):
    c, r = _dev(ctx, ort, ex, ey, mask, stats, spm, radii, fracs, metric, center)
    rc, rr = _ref(ex, ey, mask, stats, spm, radii, fracs, metric, center)
    assert np.array_equal(c, rc), (metric, center, np.argwhere(c != rc)[:5])
    assert _same_bits(r, rr), (metric, center, r, rr)
    return c, r


def _synthetic(rng, n_sets, stride, spm, masked, special):
    """random spots of varied scale; `special` adds the adversarial values to set 0"""
    scale = 10.0 ** rng.uniform(-4, 1, size=(n_sets, 1))
    ex = rng.standard_normal((n_sets, stride)) * scale
    ey = rng.standard_normal((n_sets, stride)) * scale + rng.uniform(-1, 1, size=(n_sets, 1)) * scale
    if special:
        ex[0, :7], ey[0, :7] = [0.0, 0.0, np.inf, 0.0, -0.0, 1e200, 0.0], [0.0, -0.0, 1.0, np.inf, 0.0, 1e200, -np.inf]
    if masked:
        mask = (rng.random((n_sets // spm, stride)) < 0.7).astype(np.uint8)
        mask[0, :7] = 1
        n = np.array([int((mask[s // spm] == 1).sum()) for s in range(n_sets)])
    else:
        mask = None
        n = rng.integers(0, stride + 1, size=n_sets)
        n[0] = max(n[0], 7)
    return ex, ey, mask, n


@pytest.mark.parametrize("center", ["centroid", "paraxial"])
@pytest.mark.parametrize("metric", ["circle", "square"])
@pytest.mark.parametrize("masked", [True, False])
@pytest.mark.parametrize("spm", [1, 3])
def test_synthetic_random_sets(ctx, ort, metric, center, masked, spm):
    rng = np.random.default_rng(11 + spm + 2 * masked)
    ex, ey, mask, n = _synthetic(rng, 6, 3001, spm, masked, special=True)
    ex[2, :3] = np.nan                                   # a NaN distance sorts after +Inf and lies within no radius
    st = _stats(ort, n, np.where(np.isfinite(ey), ey, 0.0).mean(axis=1))
    st["mean_y"][1] = np.nan                             # every distance of set 1 NaN under the centroid centre
    radii = np.concatenate([[0.0], np.geomspace(1e-6, 30.0, 200)])
    fracs = (1e-9, 0.1, 0.5, 0.8, 0.9, 0.95, 0.999, 1.0)
    _check(ctx, ort, ex, ey, mask, st, spm, radii, fracs, metric, center)


@pytest.mark.parametrize("metric", ["circle", "square"])
def test_all_equal_and_ulp_edges(ctx, ort, metric):
    n = 4000
    ex, ey = np.full((1, n), 0.3), np.full((1, n), 0.4)
    st = _stats(ort, [n], [0.0])
    d0 = float(distances(ex[0, :1], ey[0, :1], 0.0, metric)[0])
    radii = np.array([np.nextafter(d0, 0.0), d0, np.nextafter(d0, 1.0)])
    c, r = _check(ctx, ort, ex, ey, None, st, 1, radii, (1e-9, 0.5, 1.0), metric, "paraxial")
    assert list(c[0]) == [0, n, n] and np.all(r == d0)
    # distances 1 ulp either side of each radius and on it (<= is inclusive); square metric: d = |ey| exactly
    base = np.array([1e-3, 0.25, 1.0, 7.5])
    vals = np.concatenate([base, np.nextafter(base, 0.0), np.nextafter(base, np.inf)])
    ey2 = np.tile(vals, 50)[None]
    ex2 = np.zeros_like(ey2)
    st2 = _stats(ort, [ey2.shape[1]], [0.0])
    c2, _ = _check(ctx, ort, ex2, ey2, None, st2, 1, base, (0.5,), "square", "paraxial")
    assert list(c2[0]) == [100, 250, 400, 550]
    _check(ctx, ort, ex2, ey2, None, st2, 1, base, (0.25, 0.75), metric, "paraxial")


def test_small_n_and_rank_rounding(ctx, ort):
    rng = np.random.default_rng(5)
    stride = 1000
    ex, ey = rng.standard_normal((4, stride)), rng.standard_normal((4, stride))
    st = _stats(ort, [0, 1, 1000, 999], [0.1, 0.2, 0.0, -0.3])
    fracs = (1e-12, 0.001, 0.5, 0.25, 1.0)               # q n integer at n = 1000 (k = 500, 250, 1000)
    c, r = _check(ctx, ort, ex, ey, None, st, 1, np.linspace(0, 3, 7), fracs, "circle", "centroid")
    assert np.all(np.isnan(r[0])) and np.all(c[0] == 0)
    assert np.all(r[1] == r[1][0])


def test_max_radii_and_fracs(ctx, ort):
    rng = np.random.default_rng(9)
    ex, ey = rng.standard_normal((2, 70000)) * 1e-2, rng.standard_normal((2, 70000)) * 1e-2
    st = _stats(ort, [70000, 12345], ey.mean(axis=1))
    radii = np.linspace(0.0, 0.05, ort._lib.MAX_RADII)
    fracs = np.linspace(0.05, 1.0, ort._lib.MAX_FRACS)
    _check(ctx, ort, ex, ey, None, st, 1, radii, fracs, "circle", "centroid")
    _check(ctx, ort, ex, ey, None, st, 1, radii, (), "square", "centroid")
    _check(ctx, ort, ex, ey, None, st, 1, (), fracs, "square", "paraxial")


@pytest.mark.parametrize("kind", ["spread", "equal"])
def test_set_above_2_24_rays(ctx, ort, kind):
    """a set above 2^24 rays: pass 0 cannot keep all keys, later passes read the sweep outputs again and then, for a spread
    spot, a candidate list; for equal distances every pass reads the sweep outputs.  A small second set keeps its keys from
    pass 0 on."""
    rng = np.random.default_rng(3)
    stride = (1 << 24) + 4097
    if kind == "spread":
        ex = rng.standard_normal((2, stride)) * 1e-2
        ey = rng.standard_normal((2, stride)) * 1e-2
    else:
        ex, ey = np.full((2, stride), 1e-3), np.full((2, stride), -2e-3)
    mask = np.ones((2, stride), dtype=np.uint8)
    mask[1, 5000:] = 0
    mask[0, ::1000] = 0
    n = mask.sum(axis=1)
    st = _stats(ort, n, [float(ey[0][mask[0] == 1].mean()), float(ey[1, :5000].mean())])
    _check(ctx, ort, ex, ey, mask, st, 1, np.linspace(0.0, 0.05, 256), (1e-9, 0.5, 0.8, 0.9, 0.95, 1.0), "circle", "centroid")


# ---- traced sweeps ---------------------------------------------------------------------------------------------------
SYSTEMS = ("COOKE", "DOUBLE_GAUSS", "REFLECTIVE", "PARABOLA")


def _setup(ort, ctx, name, Hs=(0.0, 0.7, 1.0), ny=96, nx=48):
    P = getattr(ort.prescriptions, name)
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], ny) for j in range(len(Hs))])
    xs = ort.host.jl_range(0.0, p["y_EP"], nx)
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    ctx.set_layout(p["ext"], p["K"])
    return p, ys, xs, flds


def _sweep_dev(ctx, ort, p, ys, xs, flds, foci, arith, compact):
    """device sweep into torch buffers -> (ex, ey, mask, stats tensors, M)"""
    import torch
    nf, NN = len(flds), ys.shape[1] * len(xs)
    M = 1 if foci is None else len(foci)
    ex = torch.full((nf * M, NN), -7.0, dtype=torch.float64, device="cuda")
    ey = torch.full((nf * M, NN), -7.0, dtype=torch.float64, device="cuda")
    mask = torch.zeros((nf, NN), dtype=torch.uint8, device="cuda")
    st = torch.zeros(nf * M * ort.STATS_BYTES, dtype=torch.uint8, device="cuda")
    ptrs = dict(ex=ex.data_ptr(), ey=ey.data_ptr(), mask=mask.data_ptr(), stats=st.data_ptr())
    d_ys, d_xs = _tensor(ys), _tensor(xs)
    if foci is None:
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), ys.shape[1], d_xs.data_ptr(), len(xs), p["stop"], p["a_stop"], ptrs,
                             arith=arith, compact=compact, ys_per_field=True)
    else:
        ctx.trace3d_focus_dev(flds, d_ys.data_ptr(), ys.shape[1], d_xs.data_ptr(), len(xs), p["stop"], p["a_stop"], foci,
                              ptrs, arith=arith, compact=compact, ys_per_field=True)
    torch.cuda.synchronize()
    return ex, ey, mask, st, M, (d_ys, d_xs)


@pytest.mark.parametrize("sweep", ["grid", "focus"])
@pytest.mark.parametrize("compact", [False, True])
@pytest.mark.parametrize("arith", ["FAST", "STRICT"])
@pytest.mark.parametrize("name", SYSTEMS)
def test_traced_sweeps(ctx, ort, name, arith, compact, sweep):
    import torch
    p, ys, xs, flds = _setup(ort, ctx, name)
    foci = None if sweep == "grid" else p["focus"] + np.array([-0.3, 0.0, 0.2]) * max(abs(p["focus"]), 1.0) * 1e-2
    ar = getattr(ort, arith)
    ex, ey, mask, st, M, _keep = _sweep_dev(ctx, ort, p, ys, xs, flds, foci, ar, compact)
    stats = np.frombuffer(st.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    assert stats["n_kept"].min() > 0
    radii = np.linspace(0.0, 0.2, 257)
    fracs = (0.5, 0.8, 0.9, 0.95)
    nset = len(flds) * M
    for metric, center in (("circle", "centroid"), ("square", "paraxial")):
        cnt = torch.zeros((nset, len(radii)), dtype=torch.int64, device="cuda")
        rad = torch.zeros((nset, len(fracs)), dtype=torch.float64, device="cuda")
        sets = dict(n_sets=nset, sets_per_mask=M, stride=ex.shape[1], ex=ex.data_ptr(), ey=ey.data_ptr(),
                    mask=0 if compact else mask.data_ptr(), stats=st.data_ptr())
        ctx.spot_energy_dev(sets, radii, fracs, metric, center, cnt.data_ptr(), rad.data_ptr())
        torch.cuda.synchronize()
        rc, rr = _ref(ex.cpu().numpy(), ey.cpu().numpy(), None if compact else mask.cpu().numpy(), stats, M, radii, fracs,
                      metric, center)
        assert np.array_equal(cnt.cpu().numpy(), rc), (name, metric)
        assert rad.cpu().numpy().tobytes() == rr.tobytes(), (name, metric)
        if compact:
            continue
        # the host form runs the same sweep full-grid and the same kernels: the same bytes, statistics included
        h = ctx.trace3d_energy(flds, ys, xs, p["stop"], p["a_stop"], radii, fracs, foci=foci, arith=ar, metric=metric,
                               center=center)
        assert h["stats"].tobytes() == stats.tobytes()
        assert h["counts"].tobytes() == cnt.cpu().numpy().tobytes()
        assert h["radius"].tobytes() == rad.cpu().numpy().tobytes()


def test_encircled_energy_api_equals_host_form(ctx, ort):
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    radii = np.linspace(0.0, 0.1, 33)
    ee = ort.encircled_energy(s.layout, s, (0.0, 0.7, 1.0), radii=radii, fractions=(0.5, 0.8), k_rays=64, backend=ctx)
    for e in ee:
        rre = ort.full_trace(s.layout, s, e.H, 64, backend=ctx)
        d = np.sort(distances(rre.x, rre.y, float(rre.stats[0]["mean_y"]), "circle"))
        assert np.array_equal(e.fraction[0], np.searchsorted(d, radii, side="right") / len(d))
        assert e.radius[0].tobytes() == np.array([d[int(np.ceil(q * len(d))) - 1] for q in (0.5, 0.8)]).tobytes()


def test_bench_size(ctx, ort):
    """the bench grid: double-Gauss, 5792 x 2896 rays x 5 fields, FAST, against numpy on the copied-back outputs"""
    import torch
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p, ys, xs, flds = _setup(ort, ctx, "DOUBLE_GAUSS", Hs, 5792, 2896)
    ex, ey, mask, st, M, _keep = _sweep_dev(ctx, ort, p, ys, xs, flds, None, ort.FAST, False)
    stats = np.frombuffer(st.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    radii = np.linspace(0.0, 0.05, 256)
    fracs = (0.5, 0.8, 0.9, 0.95)
    cnt = torch.zeros((5, 256), dtype=torch.int64, device="cuda")
    rad = torch.zeros((5, 4), dtype=torch.float64, device="cuda")
    sets = dict(n_sets=5, sets_per_mask=1, stride=ex.shape[1], ex=ex.data_ptr(), ey=ey.data_ptr(), mask=mask.data_ptr(),
                stats=st.data_ptr())
    ctx.spot_energy_dev(sets, radii, fracs, "circle", "centroid", cnt.data_ptr(), rad.data_ptr())
    torch.cuda.synchronize()
    c, r = cnt.cpu().numpy(), rad.cpu().numpy()
    m = mask.cpu().numpy()
    for f in range(5):
        keep = m[f] == 1
        rc, rr = set_energy(ex[f].cpu().numpy()[keep], ey[f].cpu().numpy()[keep], None, int(stats[f]["n_kept"]),
                            float(stats[f]["mean_y"]), radii, fracs)
        assert np.array_equal(c[f], rc) and r[f].tobytes() == rr.tobytes(), f


# ---- determinism, enqueue only, validation ---------------------------------------------------------------------------
def _sets_for(ort, n_sets, stride, n):
    import torch
    rng = np.random.default_rng(n_sets + stride)
    ex = _tensor(rng.standard_normal((n_sets, stride)))
    ey = _tensor(rng.standard_normal((n_sets, stride)))
    st = _tensor(np.frombuffer(_stats(ort, [n] * n_sets, [0.0] * n_sets).tobytes(), dtype=np.uint8))
    cnt = torch.zeros((n_sets, ort._lib.MAX_RADII), dtype=torch.int64, device="cuda")
    rad = torch.zeros((n_sets, ort._lib.MAX_FRACS), dtype=torch.float64, device="cuda")
    sets = dict(n_sets=n_sets, sets_per_mask=1, stride=stride, ex=ex.data_ptr(), ey=ey.data_ptr(), mask=0,
                stats=st.data_ptr())
    return sets, cnt, rad, (ex, ey, st)


def test_determinism_and_launch_count(ctx, ort):
    import torch
    sets, cnt, rad, _keep = _sets_for(ort, 3, 1 << 20, 1 << 20)
    radii, fracs = np.linspace(0, 3, 100), (0.1, 0.5, 0.9)
    outs = []
    for _ in range(2):
        ctx.spot_energy_dev(sets, radii, fracs, "circle", "centroid", cnt.data_ptr(), rad.data_ptr())
        torch.cuda.synchronize()
        outs.append((cnt.cpu().numpy().tobytes(), rad.cpu().numpy().tobytes()))
    assert outs[0] == outs[1]
    launches = set()
    for n_sets, stride, n, R, Q in ((1, 10, 0, 1, 0), (3, 1 << 20, 1 << 20, 100, 3), (40, 5000, 4000, 1024, 8),
                                    (2, 3000, 1, 0, 1)):
        sets, cnt, rad, _keep = _sets_for(ort, n_sets, stride, n)
        l0 = ctx.launch_count()
        ctx.spot_energy_dev(sets, np.linspace(0, 3, R), np.linspace(0.1, 1, Q), "square", "paraxial",
                            cnt.data_ptr() if R else 0, rad.data_ptr() if Q else 0)
        launches.add(ctx.launch_count() - l0)
    torch.cuda.synchronize()
    assert len(launches) == 1, launches


def test_enqueue_only(ctx, ort):
    import torch
    sets, cnt, rad, _keep = _sets_for(ort, 5, 1 << 22, 1 << 22)
    ctx.spot_energy_dev(sets, np.linspace(0, 3, 256), (0.5, 0.9), "circle", "centroid", cnt.data_ptr(), rad.data_ptr())
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        torch.cuda._sleep(int(100e-3 * 2.0e9))           # ~100 ms at ~2 GHz
        t0 = time.perf_counter()
        ctx.spot_energy_dev(sets, np.linspace(0, 3, 256), (0.5, 0.9), "circle", "centroid", cnt.data_ptr(), rad.data_ptr(),
                            stream=st.cuda_stream)
        dt = time.perf_counter() - t0
    st.synchronize()
    assert dt < 0.02, dt


def test_validation(ctx, ort):
    import torch
    L = ort._lib
    sets, cnt, rad, _keep = _sets_for(ort, 2, 1000, 1000)
    good = dict(radii=np.linspace(0, 1, 5), fracs=(0.5,))
    ss = lambda **kw: L.SpotSets(*[dict(sets, **kw).get(k) or 0 for k in L.SPOT_SETS_NAMES])
    cases = [
        (ss(), dict(radii=[0.1, 0.1]), L.ORT_EINVAL), (ss(), dict(radii=[0.2, 0.1]), L.ORT_EINVAL),
        (ss(), dict(radii=[np.inf]), L.ORT_EINVAL), (ss(), dict(radii=[np.nan]), L.ORT_EINVAL),
        (ss(), dict(radii=[-1.0, 0.0]), L.ORT_EINVAL), (ss(), dict(fracs=(0.0,)), L.ORT_EINVAL),
        (ss(), dict(fracs=(1.0000001,)), L.ORT_EINVAL), (ss(), dict(fracs=(np.nan,)), L.ORT_EINVAL),
        (ss(), dict(radii=np.linspace(0, 1, L.MAX_RADII + 1)), L.ORT_EINVAL),
        (ss(), dict(fracs=np.linspace(0.1, 1, L.MAX_FRACS + 1)), L.ORT_EINVAL),
        (ss(), dict(radii=(), fracs=()), L.ORT_EINVAL), (ss(), dict(metric=2), L.ORT_EINVAL),
        (ss(), dict(center=-1), L.ORT_EINVAL),
        (ss(n_sets=L.MAX_FIELDS * L.MAX_FOCI + 1), {}, L.ORT_EINVAL), (ss(n_sets=0), {}, L.ORT_EINVAL),
        (ss(stride=0), {}, L.ORT_EINVAL), (ss(stride=-5), {}, L.ORT_EINVAL), (ss(sets_per_mask=0), {}, L.ORT_EINVAL),
        (ss(ex=0), {}, L.ORT_EINVAL), (ss(stats=0), {}, L.ORT_EINVAL),
        (ss(), dict(counts=0), L.ORT_EINVAL), (ss(), dict(radius=0), L.ORT_EINVAL),
    ]
    for s_, kw, code in cases:
        a = dict(good, metric=0, center=0, counts=cnt.data_ptr(), radius=rad.data_ptr())
        a.update(kw)
        req, _r, _q = L._energy_req(a["radii"], a["fracs"], a["metric"], a["center"])
        l0 = ctx.launch_count()
        rc = ctx.L.ort_spot_energy_dev(ctx.h, C.byref(s_), C.byref(req), C.c_void_p(a["counts"]), C.c_void_p(a["radius"]),
                                       None)
        assert rc == code, (kw, rc)
        assert ctx.launch_count() == l0
    # the host form: compaction is invalid, gather_stats unsupported, the focus sweep rejects opts.ext
    p, ys, xs, flds = _setup(ort, ctx, "COOKE", (0.0,), 16, 8)
    req, _r, _q = L._energy_req(good["radii"], good["fracs"], 0, 0)
    st = np.zeros(1, dtype=ort.STATS_DTYPE)
    cn, rd = np.zeros(5, dtype=np.int64), np.zeros(1)
    fa, nf = L.make_fields(flds)
    fo = np.array([float(p["focus"])])
    for op, foc, code in ((L._opts(ort.FAST, True, True), None, L.ORT_EINVAL),
                          (L._opts(ort.FAST, False, True, gather=True), None, L.ORT_EUNSUPPORTED),
                          (L._opts(ort.FAST, False, True, ext=L.EXT_VIGNETTE), fo, L.ORT_EUNSUPPORTED)):
        l0 = ctx.launch_count()
        rc = ctx.L.ort_trace3d_energy(ctx.h, fa, nf, L._vp(ys), ys.shape[1], L._vp(xs), len(xs), p["stop"], p["a_stop"],
                                      L._p(foc), 0 if foc is None else 1, C.byref(op), C.byref(req), st.ctypes.data,
                                      cn.ctypes.data, rd.ctypes.data)
        assert rc == code and ctx.launch_count() == l0
    torch.cuda.synchronize()


def test_abi_struct_sizes(ort):
    assert C.sizeof(ort._lib.EnergyReq) == 32
    assert C.sizeof(ort._lib.SpotSets) == 48


@pytest.mark.skipif(os.environ.get("ORT_POISON_SCRATCH") == "1", reason="already inside the poisoned run")
def test_parity_with_poisoned_scratch():
    env = dict(os.environ, ORT_POISON_SCRATCH="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_energy.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", "synthetic or ulp or small_n or max_radii or traced or determinism"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
