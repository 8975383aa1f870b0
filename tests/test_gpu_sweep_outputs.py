"""Host-pointer sweeps (ort_trace3d_grid, ort_trace3d_focus: outputs staged through the library's scratch and copied back)
against device-pointer sweeps (ort_trace3d_grid_dev, ort_trace3d_focus_dev: outputs written into the caller's arrays): the
same bytes for every output member each sweep accepts, with and without compaction.  Two sizes: a small ragged grid (one
launch sequence for all fields) and 2 fields x 1.1 M rays (ort_trace3d_grid's launch sequence per field, with the copies
of field f behind the trace of field f + 1)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GRID = ("ex", "ey", "r", "theta", "wx", "wy", "opd", "mask", "flags")
FOCUS = ("ex", "ey", "r", "theta", "mask", "flags")
SIZES = {"ragged": ((0.0, 0.7, 1.0), 37, 23), "per_field": ((0.0, 1.0), 1100, 1001)}


@pytest.mark.parametrize("compact", [False, True])
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("sweep", ["grid", "focus"])
def test_host_equals_dev(ctx, ort, sweep, size, compact):
    import torch
    Hs, ny, nx = SIZES[size]
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], ny) for j in range(len(Hs))])
    xs = ort.host.jl_range(0.0, p["y_EP"], nx)
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    ctx.set_layout(p["ext"], p["K"])
    if sweep == "grid":
        names, foci, kw = GRID, (), dict(compact=compact, wavegrad=(0.25, 0.55e-3), opd_scale=1.0 / 0.55e-3)
        host_sweep, dev_sweep = ctx.trace3d_grid, ctx.trace3d_grid_dev
    else:
        names, foci, kw = FOCUS, (p["focus"] + np.array([-0.2, 0.0, 0.3]),), dict(compact=compact)
        host_sweep, dev_sweep = ctx.trace3d_focus, ctx.trace3d_focus_dev
    with np.errstate(all="ignore"):
        host = host_sweep(flds, ys, xs, p["stop"], p["a_stop"], *foci, want=names + ("stats",), **kw)
    kept = host["stats"]["n_kept"].reshape(len(Hs), -1)                   # [field][focus]
    assert kept.min() > 0
    # ort_trace3d_grid launches each field of a large sweep alone, with the CTAs of a one-field launch; the device form
    # launches all fields at once, so its moments are summed over other CTA partials
    per_field_launches = sweep == "grid" and size == "per_field"
    d_ys, d_xs = torch.from_numpy(ys).cuda(), torch.from_numpy(xs).cuda()
    for with_mask in ((True, False) if compact else (True,)):            # without one the library traces its own
        dev = {k: torch.full(host[k].shape, 0xA5, dtype=torch.uint8, device="cuda") if host[k].dtype == np.uint8 else
               torch.full(host[k].shape, -7.0, dtype=torch.float64, device="cuda") for k in names}
        if not with_mask:
            del dev["mask"]
        d_stats = torch.zeros(host["stats"].nbytes, dtype=torch.uint8, device="cuda")
        ptrs = dict({k: v.data_ptr() for k, v in dev.items()}, stats=d_stats.data_ptr())
        dev_sweep(flds, d_ys.data_ptr(), ny, d_xs.data_ptr(), nx, p["stop"], p["a_stop"], *foci, ptrs, ys_per_field=True, **kw)
        torch.cuda.synchronize()
        d_st = np.frombuffer(d_stats.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE).reshape(host["stats"].shape)
        for k in ort.STATS_DTYPE.names:
            if per_field_launches and k.startswith(("mean", "m2")):           # other CTA partial sums: other rounding
                np.testing.assert_allclose(d_st[k], host["stats"][k], rtol=1e-12, atol=1e-12 * np.abs(host["stats"][k]).max())
            else:
                assert d_st[k].tobytes() == host["stats"][k].tobytes(), k
        for k, d in dev.items():
            h, d = host[k], d.cpu().numpy()
            if not compact or k in ("mask", "flags"):
                assert h.tobytes() == d.tobytes(), k
                continue
            for f in range(len(Hs)):
                for j in range(kept.shape[1] if h.ndim == 3 else 1):       # ex, ey of a focus sweep: one block per focus
                    hb, db = (h[f, j], d[f, j]) if h.ndim == 3 else (h[f], d[f])
                    assert hb[:kept[f, j]].tobytes() == db[:kept[f, j]].tobytes(), (k, f, j)
