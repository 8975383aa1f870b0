"""Encircled energy on the device (ort_spot_energy_dev, ort_trace3d_energy) against copying the spot back and sorting it.

1. Bench grid (double-Gauss, 5792 x 2896 rays x 5 fields, FAST), swept full-grid with trace3d_grid_dev into caller
   buffers; ort_spot_energy_dev with 256 radii and q = (0.5, 0.8, 0.9, 0.95), kernel time from the library's profile
   events (one event pair around all its launches), alternated with the sweep, median over --reps.  Bytes per call from
   the pass structure (csrc/kern_energy.cu), replayed in numpy on the copied-back outputs, and their share of the measured
   HBM bandwidth DESIGN.md uses (6.54 TB/s: k_paraxial_final's 5928 GB/s = 90.6 %).
2. ort_trace3d_energy end to end on the host clock, against trace3d_grid with the compacted spots copied back, and
   against numpy.sort of those spots on this host.
3. Cooke triplet, 64 x 32 grid, 3 fields x 21 foci: the EE80 radius through focus (encircled_energy with foci).

    python tools/bench_energy.py [--reps 7] [--out FILE]
Prints one JSON document (and writes it to FILE).  Needs a B200: there is no CPU path."""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench_focus import gpu_info  # noqa: E402  (tools/ is on sys.path when run as a script)

HBM_GBS = 5928.0 / 0.906
LO, HI = [51, 40, 29, 18, 7, 0], [63, 51, 40, 29, 18, 7]
CAND = 1 << 22


def pass_bytes(keys, fracs, stride, n_sets):
    """replay of kern_energy.cu's pass structure for one set: bytes read and written per pass.  A pass over the sweep
    outputs reads the mask and ex, ey: counted as 17 B per ray of the grid."""
    cap = min(stride, CAND, (1 << 26) // n_sets)
    ks = np.sort(keys)
    n = len(ks)
    tgt = [int(ks[min(max(math.ceil(q * n), 1), n) - 1]) for q in fracs]

    def matching(sh):                    # keys that carry any fraction's prefix key >> sh, each counted once
        tot = 0
        for t in set(x >> sh for x in tgt):
            lo, hi = np.uint64(t << sh), np.uint64(((t + 1) << sh) - 1) if sh < 64 else np.uint64(2 ** 64 - 1)
            tot += int(np.searchsorted(ks, hi, side="right") - np.searchsorted(ks, lo, side="left"))
        return tot

    src_n, dst, out = None, n <= cap, []
    for p in range(6):
        rd = 17 * stride if src_n is None else 8 * src_n
        wr = 8 * (n if p == 0 else matching(HI[p])) if dst else 0
        out.append(dict(reads="sweep outputs" if src_n is None else "candidates", read_bytes=rd, write_bytes=wr))
        if dst:
            src_n = wr // 8
        dst = p < 5 and matching(LO[p]) <= cap
    return out


def large(ort, ctx, reps):
    import torch
    from energy_ref import distances
    NY, NX = 5792, 2896
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], NY) for j in range(len(Hs))])
    xs = ort.host.jl_range(0.0, p["y_EP"], NX)
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    ctx.set_layout(p["ext"], p["K"])
    nf, NN = len(Hs), NY * NX
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys).to(dev), torch.from_numpy(xs).to(dev)
    ex = torch.empty((nf, NN), dtype=torch.float64, device=dev)
    ey = torch.empty((nf, NN), dtype=torch.float64, device=dev)
    mask = torch.empty((nf, NN), dtype=torch.uint8, device=dev)
    st = torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device=dev)
    radii, fracs = np.linspace(0.0, 0.05, 256), (0.5, 0.8, 0.9, 0.95)
    cnt = torch.zeros((nf, 256), dtype=torch.int64, device=dev)
    rad = torch.zeros((nf, 4), dtype=torch.float64, device=dev)
    ptrs = dict(ex=ex.data_ptr(), ey=ey.data_ptr(), mask=mask.data_ptr(), stats=st.data_ptr())
    sets = dict(n_sets=nf, sets_per_mask=1, stride=NN, ex=ex.data_ptr(), ey=ey.data_ptr(), mask=mask.data_ptr(),
                stats=st.data_ptr())
    ctx.profile_enable(True)

    def sweep():
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"], ptrs, ys_per_field=True)
        ctx.sync()
        return float(np.sum(ctx.profile_read()))

    def energy():
        ctx.spot_energy_dev(sets, radii, fracs, "circle", "centroid", cnt.data_ptr(), rad.data_ptr())
        ctx.sync()
        t = ctx.profile_read()
        assert len(t) == 1
        return float(t[0])

    sweep(), energy()
    tsw, ten = [], []
    for _ in range(reps):
        tsw.append(sweep())
        ten.append(energy())
    launches0 = ctx.launch_count()
    energy()
    launches = ctx.launch_count() - launches0
    ctx.profile_enable(False)
    # bytes per call, replayed on the copied-back outputs
    stats = np.frombuffer(st.cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    m, exh, eyh = mask.cpu().numpy(), ex.cpu().numpy(), ey.cpu().numpy()
    passes, total = [], 0
    for f in range(nf):
        keep = m[f] == 1
        d = distances(exh[f][keep], eyh[f][keep], float(stats[f]["mean_y"]), "circle")
        pb = pass_bytes(d.view(np.uint64) & np.uint64(0x7fffffffffffffff), fracs, NN, nf)
        passes.append(pb)
        total += sum(x["read_bytes"] + x["write_bytes"] for x in pb)
    me = float(np.median(ten))
    per_pass = [dict(pass_=j, sets_reading_sweep_outputs=sum(pb[j]["reads"] == "sweep outputs" for pb in passes),
                     read_bytes=sum(pb[j]["read_bytes"] for pb in passes),
                     write_bytes=sum(pb[j]["write_bytes"] for pb in passes)) for j in range(6)]
    return dict(grid=[NY, NX], fields=nf, rays_per_call=NN * nf, arith="FAST", n_radii=256, fracs=list(fracs),
                timer="ort_profile events (one pair around all energy launches), alternated with the sweep",
                launches_per_call=launches, energy_kernel_ms=me, sweep_kernel_ms=float(np.median(tsw)),
                energy_vs_sweep=me / float(np.median(tsw)), bytes_per_call=total, passes=per_pass,
                achieved_gbs=total / (me * 1e-3) / 1e9, hbm_share=total / (me * 1e-3) / 1e9 / HBM_GBS,
                hbm_reference_gbs=HBM_GBS, energy_ms_all=ten, sweep_ms_all=tsw,
                radius_ee80=rad.cpu().numpy()[:, 1].tolist())


def end_to_end(ort, ctx, reps):
    NY, NX = 5792, 2896
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], NY) for j in range(len(Hs))])
    xs = ort.host.jl_range(0.0, p["y_EP"], NX)
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    ctx.set_layout(p["ext"], p["K"])
    radii, fracs = np.linspace(0.0, 0.05, 256), (0.5, 0.8, 0.9, 0.95)
    nf, NN = len(Hs), NY * NX
    pin = {k: ort.PinnedArray((nf, NN)) for k in ("ex", "ey")}
    out = {k: v.array for k, v in pin.items()}

    def on_device():
        t = time.perf_counter()
        r = ctx.trace3d_energy(flds, ys, xs, p["stop"], p["a_stop"], radii, fracs)
        return (time.perf_counter() - t) * 1e3, r

    def copied():
        t = time.perf_counter()
        r = ctx.trace3d_grid(flds, ys, xs, p["stop"], p["a_stop"], compact=True, want=("ex", "ey", "stats"), out=out)
        return (time.perf_counter() - t) * 1e3, r

    on_device(), copied()
    td, tc = [], []
    for _ in range(reps):
        td.append(on_device()[0])
        tc.append(copied()[0])
    _, r = copied()
    tsort = []
    for f in range(nf):                              # what a user does next on the host: one sort per field
        n = int(r["stats"][f]["n_kept"])
        dy = r["ey"][f][:n] - r["stats"][f]["mean_y"]
        d = np.sqrt(r["ex"][f][:n] * r["ex"][f][:n] + dy * dy)
        t = time.perf_counter()
        np.sort(d)
        tsort.append((time.perf_counter() - t) * 1e3)
    for v in pin.values():
        v.free()
    return dict(grid=[NY, NX], fields=nf, timer="host clock, end to end", trace3d_energy_ms=float(np.median(td)),
                trace3d_grid_compact_copy_ms=float(np.median(tc)), numpy_sort_ms_all_fields=float(np.sum(tsort)),
                host_cpus=os.cpu_count(), trace3d_energy_ms_all=td, trace3d_grid_compact_copy_ms_all=tc,
                numpy_sort_ms_per_field=tsort)


def focus_curve(ort, ctx):
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = (0.0, 0.7, 1.0)
    bfd = float(s.marginal.z[-1] - s.marginal.z[-2])
    foci = bfd + np.linspace(-1.0, 1.0, 21)
    ort.encircled_energy(s.layout, s, Hs, fractions=(0.8,), k_rays=64, foci=foci, backend=ctx)
    t = time.perf_counter()
    ee = ort.encircled_energy(s.layout, s, Hs, fractions=(0.8,), k_rays=64, foci=foci, backend=ctx)
    ms = (time.perf_counter() - t) * 1e3
    return dict(system="COOKE", grid=[64, 32], fields=list(Hs), foci=foci.tolist(), call_ms=ms,
                ee80_radius_mm={str(e.H): e.radius[:, 0].tolist() for e in ee},
                best_focus_ee80={str(e.H): float(foci[int(np.argmin(e.radius[:, 0]))]) for e in ee})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ort_b200 as ort
    ctx = ort.Context(0)
    res = dict(gpu=gpu_info(), device=ctx.device_info()["name"], large=large(ort, ctx, a.reps),
               end_to_end=end_to_end(ort, ctx, a.reps), focus=focus_curve(ort, ctx))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
