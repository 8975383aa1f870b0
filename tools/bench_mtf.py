"""Diffraction MTF of the wavefront on the device (ort_wavefront_mtf_dev, ort_trace3d_mtf) against computing it on the host.

1. Bench grid (double-Gauss, 5792 x 2896 rays x 5 fields, FAST, OPD), swept full grid with trace3d_grid_dev into caller
   buffers; ort_wavefront_mtf_dev at n_freq 8, 32 and 128 (evenly spaced from 0 to the cutoff 1 / (lam F#)), time from
   the library's profile events (one pair around its four launches), alternated with the OPD sweep that produced its
   inputs, median over --reps.
2. Each MTF kernel alone from torch.profiler in a run of its own; the algorithmic FP64 rate of the two lag kernels over
   ort_fp64_peak measured in this run.  The products the definition needs after the mirror symmetry are counted from the
   shapes: per distinct lag k, sagittal ny (nx - k + floor((k - 1) / 2) + [k even]) products of 4 flop (2 DFMA, the
   real part only), tangential nx (ny - k) products of 8 flop (4 DFMA).
3. ort_trace3d_mtf end to end on the host clock, n_freq 32.
4. Today's path for one field at n_freq 32: copy the OPD map and the mask back, then numpy lag sums of the mirrored
   pupil on the host.

    python tools/bench_mtf.py [--reps 7] [--out FILE]
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
N_FREQS = (8, 32, 128)


def _setup(ort, ctx):
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(ort.Layout(P["surfaces"]), P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p, xs, ys, flds, ext = ort.host._wavefront_setup(s.layout, s, Hs, NY, None, False, ctx, "bench")
    sc = 1.0 / (LAM * s.f)
    return s, Hs, p, xs, ys, flds, ext, sc, 2.0 * sc * p["y_EP"]


def lags(freqs, s, d, kmax):
    """the distinct lags the definition needs: lag 0 and k0, k0 + 1 of every frequency, within 0 .. kmax"""
    out = {0}
    for nu in freqs:
        q = nu / (s * d)
        if q < kmax + 1:
            out |= {k for k in (int(np.floor(q)), int(np.floor(q)) + 1) if k <= kmax}
    return sorted(out)


def flops(freqs, s, xs, ys):
    """algorithmic flop of the sagittal and tangential lag sums over all sets (see the module docstring)"""
    nx = len(xs)
    dx = xs[-1] / (nx - 1)
    sag = tan = 0.0
    for y in ys:
        ny = len(y)
        dy = abs((y[-1] - y[0]) / (ny - 1))
        sag += 4.0 * ny * sum(nx - k + ((k - 1) >> 1) + (1 - k % 2) for k in lags(freqs, s, dx, 2 * (nx - 1)))
        tan += 8.0 * nx * sum(ny - k for k in lags(freqs, s, dy, ny - 1))
    return sag, tan


def device(ort, ctx, reps):
    import torch
    s, Hs, p, xs, ys, flds, ext, sc, nu_c = _setup(ort, ctx)
    nf, NN = len(Hs), NY * NX
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys).to(dev), torch.from_numpy(xs).to(dev)
    out = {"opd": torch.empty((nf, NN), dtype=torch.float64, device=dev),
           "mask": torch.empty((nf, NN), dtype=torch.uint8, device=dev),
           "stats": torch.zeros(nf * ort.STATS_BYTES, dtype=torch.uint8, device=dev)}
    ptrs = {k: v.data_ptr() for k, v in out.items()}
    otf = torch.zeros((nf, 2, max(N_FREQS), 2), dtype=torch.float64, device=dev)
    status = torch.zeros(nf, dtype=torch.int32, device=dev)
    sets = dict(n_sets=nf, stride=NN, **{k: ptrs[k] for k in ("opd", "mask", "stats")})
    freqs = {n: np.linspace(0.0, nu_c, n) for n in N_FREQS}
    ctx.profile_enable(True)

    def sweep():
        ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"], ptrs,
                             ys_per_field=True, ext=ext, opd_scale=-1.0 / LAM)
        ctx.sync()
        return float(np.sum(ctx.profile_read()))

    def run(n):
        ctx.wavefront_mtf_dev(sets, d_ys.data_ptr(), 1, NY, d_xs.data_ptr(), NX, freqs[n], sc, otf.data_ptr(),
                              status.data_ptr())

    def timed(n):
        run(n)
        ctx.sync()
        t = ctx.profile_read()
        assert len(t) == 1
        return float(t[0])

    sweep()
    for n in N_FREQS:
        timed(n)
    tsw, tmtf = [], {n: [] for n in N_FREQS}
    for _ in range(reps):
        tsw.append(sweep())
        for n in N_FREQS:
            tmtf[n].append(timed(n))
    ctx.profile_enable(False)
    stats = np.frombuffer(out["stats"].cpu().numpy().tobytes(), dtype=ort.STATS_DTYPE)
    ms_sweep = float(np.median(tsw))
    res = dict(grid=[NY, NX], fields=nf, rays=NN * nf, kept_rays=int(stats["n_kept"].sum()), arith="FAST", scale=sc,
               cutoff_cycles_per_mm=nu_c,
               timer="mtf_ms and sweep_kernel_ms: ort_profile CUDA events (one pair around the four MTF launches, one "
                     "per sweep launch), alternated; kernel_ms: torch.profiler (CUPTI kernel records) in runs of their "
                     "own, not CUDA events",
               sweep_kernel_ms=ms_sweep, sweep_ms_all=tsw, mtf={})
    from torch.profiler import ProfilerActivity, profile
    peak_tf, _ = ctx.fp64_peak()
    for n in N_FREQS:
        run(n)
        ctx.sync()
        m = float(np.median(tmtf[n]))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                run(n)
            ctx.sync()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and "k_mtf_" in e.name:
                k = re.match(r"[a-z]+", e.name.split("k_mtf_")[1]).group(0)
                t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                per.setdefault(k, []).append(t / 1e3)
        kms = {k: float(np.median(v)) for k, v in per.items()}
        f_sag, f_tan = flops(freqs[n], sc, xs, ys)
        o = otf.cpu().numpy()[:, :, :n]
        res["mtf"][str(n)] = dict(mtf_ms=m, mtf_vs_sweep=m / ms_sweep, mtf_ms_all=tmtf[n], kernel_ms=kms,
                                  sag_flop=f_sag, tan_flop=f_tan,
                                  sag_tflops=f_sag / kms["sag"] / 1e9, tan_tflops=f_tan / kms["tan"] / 1e9,
                                  sag_share_of_measured_fp64_peak=f_sag / kms["sag"] / 1e9 / peak_tf,
                                  tan_share_of_measured_fp64_peak=f_tan / kms["tan"] / 1e9 / peak_tf,
                                  lag_kernels_share_of_measured_fp64_peak=(f_sag + f_tan) / (kms["sag"] + kms["tan"])
                                  / 1e9 / peak_tf,
                                  status=status.cpu().numpy().tolist(),
                                  mtf_sag_at_half_cutoff=np.hypot(o[:, 0, n // 2, 0], o[:, 0, n // 2, 1]).tolist(),
                                  mtf_tan_at_half_cutoff=np.hypot(o[:, 1, n // 2, 0], o[:, 1, n // 2, 1]).tolist())
    res["fp64_peak_measured_tflops"] = peak_tf
    return res


def end_to_end(ort, ctx, reps, n=32):
    s, Hs, p, xs, ys, flds, ext, sc, nu_c = _setup(ort, ctx)
    freqs = np.linspace(0.0, nu_c, n)

    def call():
        t = time.perf_counter()
        ctx.trace3d_mtf(flds, ys, xs, p["stop"], p["a_stop"], freqs, sc, ext=ext, opd_scale=-1.0 / LAM)
        return (time.perf_counter() - t) * 1e3

    call()
    t = [call() for _ in range(reps)]
    ctx.set_apertures(None)
    return dict(grid=[NY, NX], fields=len(Hs), n_freq=n, timer="host clock, end to end", trace3d_mtf_ms=float(np.median(t)),
                trace3d_mtf_ms_all=t)


def todays_path(ort, ctx, n=32):
    """the OPD map and mask of the full-field point copied back, then numpy lag sums of the mirrored pupil"""
    import torch
    s, Hs, p, xs, ys, flds, ext, sc, nu_c = _setup(ort, ctx)
    f = len(Hs) - 1
    freqs = np.linspace(0.0, nu_c, n)
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys[f:f + 1].copy()).to(dev), torch.from_numpy(xs).to(dev)
    opd = torch.empty(NY * NX, dtype=torch.float64, device=dev)
    mask = torch.empty(NY * NX, dtype=torch.uint8, device=dev)
    ctx.trace3d_grid_dev(flds[f:f + 1], d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"],
                         dict(opd=opd.data_ptr(), mask=mask.data_ptr()), ys_per_field=True, ext=ext,
                         opd_scale=-1.0 / LAM)
    ctx.sync()
    t0 = time.perf_counter()
    W, m, y = opd.cpu().numpy(), mask.cpu().numpy(), d_ys.cpu().numpy()[0]
    t1 = time.perf_counter()
    keep = (m == 1).reshape(NY, NX)
    P = np.where(keep, np.exp(2j * np.pi * np.where(keep, W.reshape(NY, NX), 0.0)), 0)
    A = np.concatenate([P[:, :0:-1], 2 * P[:, :1], P[:, 1:]], axis=1)         # the mirrored pupil, column 0 doubled
    dx, dy = xs[-1] / (NX - 1), (y[-1] - y[0]) / (NY - 1)
    host = np.zeros((2, n), dtype=np.complex128)
    for az, (d, kmax) in enumerate(((dx, 2 * (NX - 1)), (abs(dy), NY - 1))):
        C = {k: (np.vdot(A[:, :A.shape[1] - k], A[:, k:]) if az == 0 else np.vdot(A[:NY - k], A[k:]))
             for k in lags(freqs, sc, d, kmax)}
        for i, nu in enumerate(freqs):
            q = nu / (sc * d)
            if not q < kmax + 1:
                continue
            k0, fr = int(np.floor(q)), q - np.floor(q)
            val = lambda k: C[k] / C[0].real if k <= kmax else 0j
            v = (1 - fr) * val(k0) + fr * val(k0 + 1)
            host[az, i] = v.conjugate() if az == 1 and dy < 0 else v
    t2 = time.perf_counter()
    d = ctx.trace3d_mtf(flds[f:f + 1], ys[f:f + 1], xs, p["stop"], p["a_stop"], freqs, sc, ext=ext,
                        opd_scale=-1.0 / LAM)
    ctx.set_apertures(None)
    return dict(field=float(Hs[f]), n_freq=n, copy_back_ms=(t1 - t0) * 1e3, numpy_lag_sums_ms=(t2 - t1) * 1e3,
                total_ms=(t2 - t0) * 1e3, host_cpus=os.cpu_count(),
                max_abs_diff_vs_device=float(np.max(np.abs(host - d["otf"][0]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ort_b200 as ort
    ctx = ort.Context(0)
    res = dict(gpu=gpu_info(), device=ctx.device_info()["name"], device_mtf=device(ort, ctx, a.reps),
               end_to_end=end_to_end(ort, ctx, a.reps), todays_path=todays_path(ort, ctx))
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
