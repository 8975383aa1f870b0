"""Through-focus sweep on the device (ort_trace3d_focus): every focus against a k_grid sweep of the layout with
t[rows-2] = that focus, in the same arithmetic -- per-ray outputs bit for bit, counts exact, moments to 1e-12."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = ("ex", "ey", "r", "theta", "mask", "flags", "stats")
COUNTS = ("n_kept", "n_miss", "n_tir", "n_domain", "n_clip", "n_strict")


def _setup(ort, ctx, name, Hs, k=64):
    P = getattr(ort.prescriptions, name)
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    p = ort.host._full_trace_setup(s.layout, s, Hs, k, None, ctx)
    xs = ort.host.jl_range(0.0, p["y_EP"], k // 2)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], k) for j in range(len(Hs))])
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    return s, p, ys, xs, flds


def _foci(s, p):
    """7 foci over BFD +- 3 depths of focus (2 lambda N^2 each, lambda = 0.55 um), BFD itself in the middle"""
    N = abs(s.f) / (2.0 * p["y_EP"])
    dof = max(2.0 * 0.55e-3 * N * N, 1e-3)
    return p["focus"] + dof * np.arange(-3.0, 4.0)


def _close(a, b, scale):
    return abs(a - b) <= 1e-12 * (abs(b) + scale)


def _rms(ort, st):
    return ort.rms_from_stats(st)


def _variant_run(fn):
    """(ARITH, rays per thread, MIRROR, SIMPLE) of every k_focus launch inside fn(), from the kernel names torch.profiler
    records (demangled "k_focus<1, 3, false, 1>" or mangled "_Z7k_focusILi1ELi3ELb0ELi1EE...")"""
    import re
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    got = set()
    for e in prof.events():
        m = re.search(r"k_focus<(\d+), ?(\d+), ?(true|false), ?(\d+)>", e.name)
        if m:
            got.add((int(m[1]), int(m[2]), m[3] == "true", int(m[4])))
        m = re.search(r"k_focusILi(\d+)ELi(\d+)ELb(\d)ELi(\d+)E", e.name)
        if m:
            got.add((int(m[1]), int(m[2]), m[3] == "1", int(m[4])))
    return got


STRICT_K = (0, 1, True, 0)          # k_focus<STRICT, 1 ray per thread>
SIMPLE_K = (1, 3, False, 1)         # FAST, refracting spheres (|R| <= 64 L) and planes
CONIC_K = (1, 2, False, 2)          # FAST, refracting conics / spheres and planes
GENERAL_K = (1, 2, False, 0)        # FAST, anything else without a mirror (weak or dummy spheres ...)
MIRROR_K = (1, 2, True, 0)          # FAST with mirrors


def _compare(ctx, ort, ext, K, fld, ys, xs, stop, a_stop, foci, ar, expect):
    """k_focus against k_grid on the layout with t[rows-2] = foci[j], every focus, same arithmetic"""
    ctx.set_layout(ext, K)
    got = _variant_run(lambda: ctx.trace3d_focus([fld], ys, xs, stop, a_stop, foci, arith=ar))
    assert got == {expect}, (got, expect)
    with np.errstate(all="ignore"):
        r = ctx.trace3d_focus([fld], ys, xs, stop, a_stop, foci, arith=ar, want=ALL)
        rc = ctx.trace3d_focus([fld], ys, xs, stop, a_stop, foci, arith=ar, compact=True, want=ALL)
    assert r["stats"].shape == (1, len(foci)) and r["ex"].shape == (1, len(foci), len(ys) * len(xs))
    for m, f in enumerate(foci):
        e2 = ext.copy()
        e2[-2, 1] = f
        ctx.set_layout(e2, K)
        with np.errstate(all="ignore"):
            g = ctx.trace3d_grid([fld], ys, xs, stop, a_stop, arith=ar, want=ALL)
            gc = ctx.trace3d_grid([fld], ys, xs, stop, a_stop, arith=ar, compact=True, want=ALL)
        st, sg = r["stats"][0, m], g["stats"][0]
        for k in COUNTS:
            assert st[k] == sg[k], (f, k, st[k], sg[k])
        assert st["r_max"] == sg["r_max"]
        n = int(sg["n_kept"])
        assert n > 0
        for k in ("mask", "flags", "r", "theta"):
            assert np.array_equal(r[k][0], g[k][0], equal_nan=True), (f, k)
        assert np.array_equal(r["ex"][0, m], g["ex"][0], equal_nan=True), f
        assert np.array_equal(r["ey"][0, m], g["ey"][0], equal_nan=True), f
        assert rc["stats"][0, m]["n_kept"] == n
        assert np.array_equal(rc["ex"][0, m, :n], gc["ex"][0, :n]) and np.array_equal(rc["ey"][0, m, :n], gc["ey"][0, :n])
        assert np.array_equal(rc["r"][0, :n], gc["r"][0, :n]) and np.array_equal(rc["theta"][0, :n], gc["theta"][0, :n])
        rms = _rms(ort, sg)
        assert math.isclose(_rms(ort, st), rms, rel_tol=1e-12)
        assert _close(st["mean_x"], sg["mean_x"], rms) and _close(st["mean_y"], sg["mean_y"], rms)
    ctx.set_layout(ext, K)


CASES = [("COOKE", 0.0), ("COOKE", 0.7), ("COOKE", 1.0), ("SINGLET", 1.0), ("DOUBLE_GAUSS", 0.5), ("TESSAR", 1.0),
         ("COOKE_RAYBASIS", 0.7)]


@pytest.mark.parametrize("arith", ["STRICT", "FAST"])
@pytest.mark.parametrize("name,H", CASES)
def test_focus_bit_identical_to_grid(ctx, ort, name, H, arith):
    ar = getattr(ort, arith)
    s, p, ys, xs, flds = _setup(ort, ctx, name.replace("_RAYBASIS", ""), [H])
    fld = flds[0]
    if name.endswith("_RAYBASIS"):
        fld = dict(mode=1, ybar=12.0, z0=-500.0, h_prime=0.3)
    _compare(ctx, ort, p["ext"], p["K"], fld, ys[0], xs, p["stop"], p["a_stop"], _foci(s, p), ar,
             STRICT_K if ar == ort.STRICT else SIMPLE_K)


def _cooke_variant(ort, ctx, which):
    """the Cooke triplet's prelude grid on a changed layout: one surface made a conic (SIMPLE-conic class) or one sphere
    made weak, |R| far above 64 L (general class without mirrors)"""
    s, p, ys, xs, flds = _setup(ort, ctx, "COOKE", [0.7])
    ext, K = p["ext"].copy(), p["K"].copy()
    if which == "conic":
        K[3] = -0.6
    else:
        ext[2, 0] = -2.0e4
    return ext, K, flds[0], ys[0], xs, p["stop"], p["a_stop"], _foci(s, p)


def _mirror_system(ort, ctx, name):
    """a reflecting prescription with an explicit grid over its stop; the image plane [Inf 0 1] sits behind the last
    medium n = -1, so it is a refracting plane (n -1 -> 1) in both arithmetics"""
    P = getattr(ort.prescriptions, name)
    S = P["surfaces"]
    s = ort.solve(S[:, :3], P["a"], P["h"], backend=ctx)
    K = np.append(S[:, 3] if S.shape[1] > 3 else np.zeros(len(S)), 0.0)
    ext = np.vstack([S[:, :3], [np.inf, 0.0, 1.0]])
    focus = float(s.marginal.z[-1] - s.marginal.z[-2])
    ext[-2, 1] = focus
    a_stop = abs(P["a"][s.stop - 1])
    ys = np.linspace(-0.98 * a_stop, 0.98 * a_stop, 48)
    xs = np.linspace(0.0, 0.98 * a_stop, 24)
    fld = dict(mode=0, u=0.02, v=0.0, h_prime=0.02 * s.f)
    foci = focus + 0.02 * abs(focus) * np.arange(-3.0, 4.0)
    return ext, K, fld, ys, xs, s.stop, a_stop, foci


@pytest.mark.parametrize("arith", ["STRICT", "FAST"])
@pytest.mark.parametrize("case", ["COOKE_CONIC", "COOKE_WEAK_SPHERE", "REFLECTIVE", "PARABOLA"])
def test_focus_bit_identical_other_variants(ctx, ort, case, arith):
    """the FAST instantiations the refracting fixtures above do not reach: SIMPLE-conic, general, general with mirrors
    (incl. the refracting image plane behind a mirror and the conic mirror body)"""
    ar = getattr(ort, arith)
    if case.startswith("COOKE"):
        args = _cooke_variant(ort, ctx, "conic" if case == "COOKE_CONIC" else "weak")
        fast_k = CONIC_K if case == "COOKE_CONIC" else GENERAL_K
    else:
        args = _mirror_system(ort, ctx, case)
        fast_k = MIRROR_K
    _compare(ctx, ort, *args, ar, STRICT_K if ar == ort.STRICT else fast_k)


def test_multi_field_ys_per_field(ctx, ort):
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = (0.0, 0.7, 1.0)
    foci = s.marginal.z[-1] - s.marginal.z[-2] + np.linspace(-0.3, 0.3, 5)
    tf = ort.through_focus(s.layout, s, Hs, foci, 64, spots=True, backend=ctx)
    for m, f in enumerate(foci):
        errs = ort.full_trace_fields(s.layout, s, Hs, 64, focus=float(f), backend=ctx)
        for t, e in zip(tf, errs):
            assert t.n_kept == int(e.stats[0]["n_kept"])
            assert math.isclose(t.rms[m], e.RMS, rel_tol=1e-12), (t.H, f, t.rms[m], e.RMS)
            assert np.array_equal(t.spots[m][0], e.x) and np.array_equal(t.spots[m][1], e.y)
    for t in tf:
        assert t.bracketed and t.best_rms <= t.rms.min() * (1 + 1e-12)


def test_launch_count_stats_only(ctx, ort):
    s, p, ys, xs, flds = _setup(ort, ctx, "COOKE", [0.0, 0.7, 1.0])
    ctx.set_layout(p["ext"], p["K"])
    for M in (1, 16, 64):
        foci = p["focus"] + np.linspace(-1.0, 1.0, M)
        l0 = ctx.launch_count()
        ctx.trace3d_focus(flds, ys, xs, p["stop"], p["a_stop"], foci)
        assert ctx.launch_count() - l0 == 2, M
        l0 = ctx.launch_count()
        ctx.trace3d_focus(flds, ys, xs, p["stop"], p["a_stop"], foci, compact=True, want=("ex", "ey", "stats"))
        assert ctx.launch_count() - l0 == 5, M


def test_deterministic(ctx, ort):
    s, p, ys, xs, flds = _setup(ort, ctx, "DOUBLE_GAUSS", [0.0, 0.5, 1.0], k=512)
    ctx.set_layout(p["ext"], p["K"])
    foci = p["focus"] + np.linspace(-0.5, 0.5, 16)
    for ar in (ort.FAST, ort.STRICT):
        a = ctx.trace3d_focus(flds, ys, xs, p["stop"], p["a_stop"], foci, arith=ar)["stats"]
        b = ctx.trace3d_focus(flds, ys, xs, p["stop"], p["a_stop"], foci, arith=ar)["stats"]
        assert a.tobytes() == b.tobytes()


def _raw(ctx, ort, flds, ys, xs, stop, a_stop, foci, opts=None, out=None):
    """ort_trace3d_focus with explicit ort_opts / ort_grid_out fields -> status code"""
    farr, nf = ort._lib.make_fields(flds)
    ys, xs, foci = (np.ascontiguousarray(a, dtype=np.float64) for a in (ys, xs, foci))
    stats = np.zeros((nf, max(len(foci), 1)), dtype=ort.STATS_DTYPE)
    spare = np.zeros(nf * len(ys) * len(xs) * max(len(foci), 1))
    o = dict(arith=1, compact=0, ys_per_field=0, ext=0, wg_nu=0.0, wg_lambda=1.0, opd_scale=1.0, gather_stats=0, reserved=0)
    o.update(opts or {})
    op = ort._lib.Opts(**o)
    go = ort._lib.GridOut(stats=stats.ctypes.data)
    for k in (out or ()):
        setattr(go, k, spare.ctypes.data)
    return ctx.L.ort_trace3d_focus(ctx.h, farr, nf, ys.ctypes.data, len(ys), xs.ctypes.data, len(xs), int(stop),
                                   float(a_stop), foci.ctypes.data_as(C.POINTER(C.c_double)), len(foci), C.byref(op),
                                   C.byref(go))


def test_error_paths_leave_context_usable(ctx, ort):
    s, p, ys, xs, flds = _setup(ort, ctx, "COOKE", [0.7], k=32)
    ext, K = p["ext"], p["K"]
    stop, a_stop = p["stop"], p["a_stop"]
    foci = p["focus"] + np.array([-0.5, 0.0, 0.5])
    EINVAL, EUNSUP = ort._lib.ORT_EINVAL, ort._lib.ORT_EUNSUPPORTED

    def usable():
        ctx.set_layout(ext, K)
        g = ctx.trace3d_grid(flds, ys[0], xs, stop, a_stop)
        assert g["stats"][0]["n_kept"] > 0

    ctx.set_layout(ext, K)
    cases = [
        (EINVAL, dict(foci=np.array([]))),
        (EINVAL, dict(foci=p["focus"] + np.arange(ort._lib.MAX_FOCI + 1) * 1e-3)),
        (EINVAL, dict(foci=np.array([p["focus"], np.nan]))),
        (EINVAL, dict(foci=np.array([np.inf]))),
        (EINVAL, dict(stop=len(ext) - 1)),                           # the image plane itself
        (EINVAL, dict(out=("wx",))), (EINVAL, dict(out=("wy",))), (EINVAL, dict(out=("opd",))),
        (EINVAL, dict(out=("stats_local",))),
        (EINVAL, dict(flds=[])), (EINVAL, dict(flds=[dict(flds[0], mode=2)])), (EINVAL, dict(stop=0)),
        (EINVAL, dict(opts=dict(arith=7))),
        (EUNSUP, dict(opts=dict(ext=ort.EXT_OPD))), (EUNSUP, dict(opts=dict(ext=ort.EXT_VIGNETTE))),
        (EUNSUP, dict(opts=dict(gather_stats=1))),
    ]
    for code, kw in cases:
        a = dict(flds=flds, ys=ys[0], xs=xs, stop=stop, a_stop=a_stop, foci=foci)
        a.update(kw)
        assert _raw(ctx, ort, **a) == code, kw
        usable()
    for last in ([1000.0, 0.0, 1.0], [np.inf, 0.0, 1.0, 0.5]):        # a curved last row; a plane with K != 0
        e2 = ext.copy()
        K2 = K.copy()
        e2[-1, 0] = last[0]
        if len(last) > 3:
            K2[-1] = last[3]
        ctx.set_layout(e2, K2)
        assert _raw(ctx, ort, flds, ys[0], xs, stop, a_stop, foci) == EINVAL
        usable()
    ctx.set_layout(ext, K)
    coef = np.zeros((len(ext), 3))
    coef[2, 2] = 1e-6
    ctx.set_polynomials(coef)
    assert _raw(ctx, ort, flds, ys[0], xs, stop, a_stop, foci) == EUNSUP
    ctx.set_polynomials(None)
    usable()


def test_full_size_double_gauss_dev(ctx, ort):
    """the bench grid: 5792 x 2896 x 5 fields, FAST, 16 foci, stats only through _dev, against 16 separate sweeps"""
    import torch
    NY, NX = 5792, 2896
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], NY) for j in range(len(Hs))])
    xs = ort.host.jl_range(0.0, p["y_EP"], NX)
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    foci = p["focus"] + np.linspace(-0.4, 0.4, 16)
    dev = torch.device("cuda", ctx.device)
    d_ys = torch.from_numpy(ys).to(dev)
    d_xs = torch.from_numpy(xs).to(dev)
    nf, M = len(Hs), len(foci)
    d_st = torch.zeros(nf * M * ort.STATS_BYTES, dtype=torch.uint8, device=dev)
    d_sg = torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device=dev)
    ext, K = p["ext"], p["K"]
    ctx.set_layout(ext, K)
    ctx.trace3d_focus_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"], foci,
                          {"stats": d_st.data_ptr()}, ys_per_field=True)
    ctx.sync()
    st = np.frombuffer(d_st.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE).reshape(nf, M)
    for m, f in enumerate(foci):
        e2 = ext.copy()
        e2[-2, 1] = f
        ctx.set_layout(e2, K)
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"],
                             {"stats": d_sg.data_ptr()}, ys_per_field=True)
        ctx.sync()
        sg = np.frombuffer(d_sg.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
        for j in range(nf):
            assert st[j, m]["n_kept"] == sg[j]["n_kept"] > 0
            assert math.isclose(_rms(ort, st[j, m]), _rms(ort, sg[j]), rel_tol=1e-12), (j, f)
    ctx.set_layout(ext, K)


@pytest.mark.skipif(os.environ.get("ORT_POISON_SCRATCH") == "1", reason="already inside the poisoned run")
def test_focus_suite_with_poisoned_scratch():
    """this file once more with every scratch slot filled with 0xFF bytes each time an entry point asks for it"""
    env = dict(os.environ, ORT_POISON_SCRATCH="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_focus.py", "-m", "gpu", "-x", "-q", "-p",
                        "no:cacheprovider", "-k", "not full_size"], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
