"""Diffraction PSF of the wavefront on the device (ort_wavefront_psf_dev, ort_trace3d_psf) against computing it on the host.

1. Bench grid (double-Gauss, 5792 x 2896 rays x 5 fields, FAST, OPD), swept full grid with trace3d_grid_dev into caller
   buffers; ort_wavefront_psf_dev at n_pix 127, 255 and 511 (default pitch lam F# / 2), time from the library's profile
   events (one pair around its five launches), alternated with the OPD sweep that produced its inputs, median over --reps.
2. Each PSF kernel alone from torch.profiler in a run of its own; the algorithmic FP64 rate of stage A (k_psf_x), counted
   as 4 ny nx ceil(n_u / 2) flop per set, over ort_fp64_peak measured in this run.
3. ort_trace3d_psf end to end on the host clock, n_pix 255.
4. Today's path for one field at n_pix 255: copy the OPD map, the mask and the grid coordinates back, then a numpy matrix
   Fourier transform (the cos form, complex128 matrix products) on the host.

    python tools/bench_psf.py [--reps 7] [--out FILE]
Prints one JSON document (and writes it to FILE).  Needs a B200: there is no CPU path."""
import argparse
import json
import os
import re
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench_focus import gpu_info  # noqa: E402  (tools/ is on sys.path when run as a script)

NY, NX = 5792, 2896
LAM = 587.5618e-6
SIDES = (127, 255, 511)


def _setup(ort, ctx):
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, NY, None, False, ctx, "bench")
    sc = 1.0 / (LAM * s.f)
    return s, Hs, p, xs, ys, flds, ext, sc, 1.0 / (4.0 * sc * p["y_EP"])


def device(ort, ctx, reps):
    import torch
    s, Hs, p, xs, ys, flds, ext, sc, pitch = _setup(ort, ctx)
    nf, NN = len(Hs), NY * NX
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys).to(dev), torch.from_numpy(xs).to(dev)
    out = {"opd": torch.empty((nf, NN), dtype=torch.float64, device=dev),
           "mask": torch.empty((nf, NN), dtype=torch.uint8, device=dev),
           "stats": torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device=dev)}
    ptrs = {k: v.data_ptr() for k, v in out.items()}
    side_max = max(SIDES)
    psf = torch.zeros((nf, side_max * side_max), dtype=torch.float64, device=dev)
    strehl = torch.zeros((nf, 2), dtype=torch.float64, device=dev)
    peak = torch.zeros(nf, dtype=torch.int32, device=dev)
    status = torch.zeros(nf, dtype=torch.int32, device=dev)
    sets = dict(n_sets=nf, stride=NN, **{k: ptrs[k] for k in ("opd", "mask", "stats")})
    ctx.profile_enable(True)

    def sweep():
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"], ptrs,
                             ys_per_field=True, ext=ext, opd_scale=-1.0 / LAM)
        ctx.sync()
        return float(np.sum(ctx.profile_read()))

    def run(n):
        ctx.wavefront_psf_dev(sets, d_ys.data_ptr(), 1, NY, d_xs.data_ptr(), NX, n, n, pitch, pitch, sc, psf.data_ptr(),
                              strehl.data_ptr(), peak.data_ptr(), status.data_ptr())

    def timed(n):
        run(n)
        ctx.sync()
        t = ctx.profile_read()
        assert len(t) == 1
        return float(t[0])

    sweep()
    for n in SIDES:
        timed(n)
    tsw, tpsf = [], {n: [] for n in SIDES}
    for _ in range(reps):
        tsw.append(sweep())
        for n in SIDES:
            tpsf[n].append(timed(n))
    ctx.profile_enable(False)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    ms_sweep = float(np.median(tsw))
    res = dict(grid=[NY, NX], fields=nf, rays=NN * nf, kept_rays=int(stats["n_kept"].sum()), arith="FAST",
               pitch_mm=pitch, scale=sc,
               timer="psf_ms and sweep_kernel_ms: ort_profile CUDA events (one pair around the five PSF launches, one "
                     "per sweep launch), alternated; kernel_ms: torch.profiler (CUPTI kernel records) in runs of their "
                     "own, not CUDA events",
               sweep_kernel_ms=ms_sweep, sweep_ms_all=tsw, psf={})
    from torch.profiler import ProfilerActivity, profile
    peak_tf, _ = ctx.fp64_peak()
    for n in SIDES:
        run(n)
        ctx.sync()
        m = float(np.median(tpsf[n]))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                run(n)
            ctx.sync()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and "k_psf_" in e.name:
                k = re.match(r"[a-z]+", e.name.split("k_psf_")[1]).group(0)
                t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                per.setdefault(k, []).append(t / 1e3)
        ms_x = float(np.median(per["x"]))
        flop_x = 4.0 * NY * NX * ((n + 1) // 2) * nf
        res["psf"][str(n)] = dict(psf_ms=m, psf_vs_sweep=m / ms_sweep, psf_ms_all=tpsf[n],
                                  kernel_ms={k: float(np.median(v)) for k, v in per.items()},
                                  stage_a_flop=flop_x, stage_a_tflops=flop_x / ms_x / 1e9,
                                  stage_a_share_of_measured_fp64_peak=flop_x / ms_x / 1e9 / peak_tf,
                                  status=status.cpu().numpy().tolist(), strehl=strehl.cpu().numpy()[:, 0].tolist())
    res["fp64_peak_measured_tflops"] = peak_tf
    return res


def end_to_end(ort, ctx, reps, n=255):
    s, Hs, p, xs, ys, flds, ext, sc, pitch = _setup(ort, ctx)

    def call():
        t = time.perf_counter()
        ctx.trace3d_psf(flds, ys, xs, p["stop"], p["a_stop"], n, n, pitch, pitch, sc, ext=ext, opd_scale=-1.0 / LAM)
        return (time.perf_counter() - t) * 1e3

    call()
    t = [call() for _ in range(reps)]
    ctx.set_apertures(None)
    return dict(grid=[NY, NX], fields=len(Hs), n_pix=n, timer="host clock, end to end", trace3d_psf_ms=float(np.median(t)),
                trace3d_psf_ms_all=t)


def todays_path(ort, ctx, n=255):
    """the OPD map, mask and coordinates of the full-field point copied back, then a numpy MFT on the host"""
    import torch
    s, Hs, p, xs, ys, flds, ext, sc, pitch = _setup(ort, ctx)
    f = len(Hs) - 1
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys[f:f + 1].copy()).to(dev), torch.from_numpy(xs).to(dev)
    opd = torch.empty(NY * NX, dtype=torch.float64, device=dev)
    mask = torch.empty(NY * NX, dtype=torch.uint8, device=dev)
    ctx.trace3d_grid_dev(flds[f:f + 1], d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"],
                         dict(opd=opd.data_ptr(), mask=mask.data_ptr()), ys_per_field=True, ext=ext,
                         opd_scale=-1.0 / LAM)
    ctx.sync()
    t0 = time.perf_counter()
    W, m, y, x = opd.cpu().numpy(), mask.cpu().numpy(), d_ys.cpu().numpy()[0], d_xs.cpu().numpy()
    t1 = time.perf_counter()
    u = (np.arange(n) - (n - 1) / 2) * pitch
    keep = (m == 1).reshape(NY, NX)
    P = np.where(keep, np.exp(2j * np.pi * np.where(keep, W.reshape(NY, NX), 0.0)), 0)
    Cx = 2.0 * np.cos(2 * np.pi * sc * x[:, None] * u[None, :])
    Yv = np.exp(2j * np.pi * sc * u[:, None] * y[None, :])
    E = Yv @ (P @ Cx)
    host = np.abs(E) ** 2 / (2.0 * keep.sum()) ** 2
    t2 = time.perf_counter()
    d = ctx.trace3d_psf(flds[f:f + 1], ys[f:f + 1], xs, p["stop"], p["a_stop"], n, n, pitch, pitch, sc, ext=ext,
                        opd_scale=-1.0 / LAM)
    ctx.set_apertures(None)
    return dict(field=float(Hs[f]), n_pix=n, copy_back_ms=(t1 - t0) * 1e3, numpy_mft_ms=(t2 - t1) * 1e3,
                total_ms=(t2 - t0) * 1e3, host_cpus=os.cpu_count(),
                max_abs_diff_vs_device=float(np.max(np.abs(host - d["psf"][0]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ort_b200 as ort
    ctx = ort.Context(0)
    res = dict(gpu=gpu_info(), device=ctx.device_info()["name"], device_psf=device(ort, ctx, a.reps),
               end_to_end=end_to_end(ort, ctx, a.reps), todays_path=todays_path(ort, ctx))
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
