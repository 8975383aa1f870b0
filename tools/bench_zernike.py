"""Zernike fit of the wavefront on the device (ort_wavefront_zernike_dev, ort_trace3d_zernike) against fitting on the host.

1. Bench grid (double-Gauss, 5792 x 2896 rays x 5 fields, FAST, OPD), swept full grid with trace3d_grid_dev into caller
   buffers; ort_wavefront_zernike_dev at n_max 4, 8 and 12, kernel time from the library's profile events (one pair
   around its four launches), alternated with the OPD sweep that produced its inputs, median over --reps.
2. The Gram kernel (k_zern_gram) alone from torch.profiler at n_max 8 and 12: FP64 rate counted from the upper triangle
   of G and b per kept ray (the useful DFMA) and from the 4 x 4 blocks the kernel computes (the executed DFMA), over
   ort_fp64_peak measured in this run and over the nominal 148 SMs x 64 FP64 lanes x 2 flop x the card's max SM clock.
3. ort_trace3d_zernike end to end on the host clock.
4. Today's path for one field: wavefront() and full_trace() on the same grid (compacted maps copied back), then a
   numpy least-squares fit of the symmetric terms on the host.

    python tools/bench_zernike.py [--reps 7] [--out FILE]
Prints one JSON document (and writes it to FILE).  Needs a B200: there is no CPU path."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bench_focus import gpu_info  # noqa: E402  (tools/ is on sys.path when run as a script)

NY, NX = 5792, 2896
LAM = 587.5618e-6


def _setup(ort, ctx):
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, NY, None, False, ctx, "bench")
    return s, Hs, p, xs, ys, flds, ext


def device(ort, ctx, reps):
    import torch
    import zernike_ref as zr
    s, Hs, p, xs, ys, flds, ext = _setup(ort, ctx)
    nf, NN = len(Hs), NY * NX
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys).to(dev), torch.from_numpy(xs).to(dev)
    out = {k: torch.empty((nf, NN), dtype=torch.float64, device=dev) for k in ("opd", "r", "theta")}
    out["mask"] = torch.empty((nf, NN), dtype=torch.uint8, device=dev)
    out["stats"] = torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device=dev)
    ptrs = {k: v.data_ptr() for k, v in out.items()}
    coef = torch.zeros((nf, zr.n_terms(12)), dtype=torch.float64, device=dev)
    resid = torch.zeros((nf, 2), dtype=torch.float64, device=dev)
    status = torch.zeros(nf, dtype=torch.int32, device=dev)
    sets = dict(n_sets=nf, stride=NN, **{k: ptrs[k] for k in ("opd", "r", "theta", "mask", "stats")})
    ctx.profile_enable(True)

    def sweep():
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"], ptrs,
                             ys_per_field=True, ext=ext, opd_scale=-1.0 / LAM)
        ctx.sync()
        return float(np.sum(ctx.profile_read()))

    def fit(n_max):
        ctx.wavefront_zernike_dev(sets, n_max, p["a_stop"], coef.data_ptr(), resid.data_ptr(), status.data_ptr())
        ctx.sync()
        t = ctx.profile_read()
        assert len(t) == 1
        return float(t[0])

    orders = (4, 8, 12)
    sweep()
    for n in orders:
        fit(n)
    tsw, tfit = [], {n: [] for n in orders}
    for _ in range(reps):
        tsw.append(sweep())
        for n in orders:
            tfit[n].append(fit(n))
    ctx.profile_enable(False)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    kept = int(stats["n_kept"].sum())
    ms_sweep = float(np.median(tsw))
    res = dict(grid=[NY, NX], fields=nf, rays=NN * nf, kept_rays=kept, arith="FAST", norm="stop",
               timer="ort_profile events (one pair around the four fit launches), alternated with the OPD sweep",
               sweep_kernel_ms=ms_sweep, sweep_ms_all=tsw, fit={})
    for n in orders:
        ctx.wavefront_zernike_dev(sets, n, p["a_stop"], coef.data_ptr(), resid.data_ptr(), status.data_ptr())
        ctx.sync()
        st = status.cpu().numpy()
        m = float(np.median(tfit[n]))
        res["fit"][str(n)] = dict(fit_ms=m, fit_vs_sweep=m / ms_sweep, fit_ms_all=tfit[n], status=st.tolist(),
                                  rms_resid_waves=resid.cpu().numpy()[:, 0].tolist(),
                                  bytes_two_passes=2 * 25 * NN * nf)
    # the Gram kernel alone, from a profiler run of its own
    from torch.profiler import ProfilerActivity, profile
    gram = {}
    for n in (8, 12):
        ctx.wavefront_zernike_dev(sets, n, p["a_stop"], coef.data_ptr(), resid.data_ptr(), status.data_ptr())
        ctx.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ctx.wavefront_zernike_dev(sets, n, p["a_stop"], coef.data_ptr(), resid.data_ptr(), status.data_ptr())
            ctx.sync()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and "k_zern" in e.name:
                k = e.name.split("k_zern_")[1].split("(")[0].split("E")[0]
                per.setdefault(k, []).append(e.device_time_total / 1e3 if hasattr(e, "device_time_total") else e.cuda_time_total / 1e3)
        js = int(zr.symmetric(n).sum())
        jp = (js + 1 + 3) // 4 * 4
        nblk = (jp // 4) * (jp // 4 + 1) // 2
        ms = float(np.median(per["gram"]))
        useful = 2.0 * (js * (js + 1) // 2 + js) * kept
        executed = 2.0 * 16 * nblk * kept
        gram[str(n)] = dict(fitted_terms=js, gram_kernel_ms=ms, kernel_ms={k: float(np.median(v)) for k, v in per.items()},
                            useful_flop=useful, executed_flop=executed, useful_tflops=useful / ms / 1e9,
                            executed_tflops=executed / ms / 1e9)
    peak, _ = ctx.fp64_peak()
    g = gpu_info()
    try:
        nominal = 148 * 64 * 2 * float(g.split(",")[2].split()[0]) * 1e6 / 1e12     # "name, power.limit, 1965 MHz"
    except (ValueError, IndexError):
        nominal = float("nan")
    for v in gram.values():
        v["share_of_measured_fp64_peak"] = v["useful_tflops"] / peak
        v["share_of_nominal_fp64"] = v["useful_tflops"] / nominal
    res["gram"] = gram
    res["fp64_peak_measured_tflops"] = peak
    res["fp64_nominal_tflops"] = nominal
    return res


def end_to_end(ort, ctx, reps):
    s, Hs, p, xs, ys, flds, ext = _setup(ort, ctx)

    def call():
        t = time.perf_counter()
        ctx.trace3d_zernike(flds, ys, xs, p["stop"], p["a_stop"], 8, p["a_stop"], ext=ext, opd_scale=-1.0 / LAM)
        return (time.perf_counter() - t) * 1e3

    call()
    t = [call() for _ in range(reps)]
    ctx.set_apertures(None)
    return dict(grid=[NY, NX], fields=len(Hs), n_max=8, timer="host clock, end to end", trace3d_zernike_ms=float(np.median(t)),
                trace3d_zernike_ms_all=t)


def todays_path(ort, ctx):
    """wavefront() + full_trace() + a numpy lstsq of the symmetric terms, for the full-field point"""
    import zernike_ref as zr
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    H = 1.0
    t0 = time.perf_counter()
    w = ort.wavefront(s.layout, s, [H], NY, backend=ctx)[0]
    t1 = time.perf_counter()
    e = ort.full_trace(s.layout, s, H, NY, backend=ctx)
    t2 = time.perf_counter()
    n = len(w.opd) // 2
    sym = zr.symmetric(8)
    A = zr.basis(8, e.r[:n], e.t[:n], cols=sym)
    t3 = time.perf_counter()
    c = np.linalg.lstsq(A, w.opd[:n], rcond=None)[0]
    t4 = time.perf_counter()
    z = ort.zernike(s.layout, s, [H], n_max=8, k_rays=NY, norm="rmax", backend=ctx)[0]
    return dict(field=H, kept_rays=n, n_max=8, design_matrix=[n, int(sym.sum())], wavefront_ms=(t1 - t0) * 1e3,
                full_trace_ms=(t2 - t1) * 1e3, basis_ms=(t3 - t2) * 1e3, lstsq_ms=(t4 - t3) * 1e3,
                total_ms=(t4 - t0) * 1e3, host_cpus=os.cpu_count(),
                max_abs_diff_vs_device_waves=float(np.max(np.abs(z.coef[sym] - c))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ort_b200 as ort
    ctx = ort.Context(0)
    res = dict(gpu=gpu_info(), device=ctx.device_info()["name"], device_fit=device(ort, ctx, a.reps),
               end_to_end=end_to_end(ort, ctx, a.reps), todays_path=todays_path(ort, ctx))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
