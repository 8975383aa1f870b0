"""Through-focus sweep (ort_trace3d_focus) against one grid sweep per focus (ort_trace3d_grid), on the device.

Large grid: the bench workload (double-Gauss, 5792 x 2896 rays x 5 fields, FAST, statistics only) at M = 1, 4, 16, 64
foci.  Kernel time from the library's profile events (ort_profile_*: k_focus, resp. the M k_grid launches), the two
arms alternated in one process, median over --reps.  Reference size: Cooke triplet, 64 x 32 grid, 3 fields, 21 foci,
end to end on the host clock: one through_focus call, statistics only and with the spot diagrams, against 21
full_trace_fields calls (which always return the spots).

    python tools/bench_focus.py [--reps 7] [--out FILE]
Prints one JSON document (and writes it to FILE).  Needs a B200: there is no CPU path."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else ""
    except Exception as e:                          # the measurement still stands; say why the line is missing
        return f"nvidia-smi unavailable: {e}"


def large(ort, ctx, reps):
    import torch
    NY, NX = 5792, 2896
    P = ort.prescriptions.DOUBLE_GAUSS
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = ort.prescriptions.DOUBLE_GAUSS_FIELDS
    p = ort.host._full_trace_setup(s.layout, s, Hs, 64, None, ctx)
    ys = np.stack([ort.host.jl_range(p["y1"][j], p["y2"][j], NY) for j in range(len(Hs))])
    xs = ort.host.jl_range(0.0, p["y_EP"], NX)
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j])) for j in range(len(Hs))]
    dev = torch.device("cuda", ctx.device)
    d_ys, d_xs = torch.from_numpy(ys).to(dev), torch.from_numpy(xs).to(dev)
    nf = len(Hs)
    d_st = torch.zeros(nf * 64 * ort.STATS_BYTES, dtype=torch.uint8, device=dev)
    ext, K = p["ext"], p["K"]
    rays = NY * NX * nf
    out = []
    ctx.profile_enable(True)
    for M in (1, 4, 16, 64):
        foci = p["focus"] + (np.linspace(-0.4, 0.4, M) if M > 1 else np.zeros(1))

        def focus_arm():
            ctx.set_layout(ext, K)
            ctx.trace3d_focus_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"], foci,
                                  {"stats": d_st.data_ptr()}, ys_per_field=True)
            ctx.sync()
            return float(np.sum(ctx.profile_read()))

        def sweeps_arm():
            for f in foci:
                e2 = ext.copy()
                e2[-2, 1] = f
                ctx.set_layout(e2, K)
                ctx.trace3d_grid_dev(flds, d_ys.data_ptr(), NY, d_xs.data_ptr(), NX, p["stop"], p["a_stop"],
                                     {"stats": d_st.data_ptr()}, ys_per_field=True)
            ctx.sync()
            return float(np.sum(ctx.profile_read()))

        focus_arm(), sweeps_arm()                  # warm-up of both shapes
        tf, ts = [], []
        for _ in range(reps):
            tf.append(focus_arm())
            ts.append(sweeps_arm())
        mf, ms = float(np.median(tf)), float(np.median(ts))
        out.append(dict(n_foci=M, focus_kernel_ms=mf, sweeps_kernel_ms=ms, ratio=ms / mf, focus_vs_one_sweep=mf / (ms / M),
                        ray_foci_per_s=rays * M / (mf * 1e-3), focus_ms_all=tf, sweeps_ms_all=ts))
        print(json.dumps({k: v for k, v in out[-1].items() if not k.endswith("_all")}), file=sys.stderr)
    ctx.profile_enable(False)
    return dict(grid=[NY, NX], fields=nf, rays_per_call=rays, arith="FAST", outputs="stats only", timer="ort_profile events",
                results=out)


def reference(ort, ctx, reps):
    P = ort.prescriptions.COOKE
    s = ort.solve(P["surfaces"], P["a"], P["h"], backend=ctx)
    Hs = (0.0, 0.7, 1.0)
    bfd = float(s.marginal.z[-1] - s.marginal.z[-2])
    foci = bfd + np.linspace(-1.0, 1.0, 21)

    def one():
        ort.through_focus(s.layout, s, Hs, foci, 64, backend=ctx)

    def one_spots():        # the spot diagrams too (compacted, mirrored), as full_trace_fields returns them
        ort.through_focus(s.layout, s, Hs, foci, 64, spots=True, backend=ctx)

    def many():
        for f in foci:
            ort.full_trace_fields(s.layout, s, Hs, 64, focus=float(f), backend=ctx)

    one(), one_spots(), many()
    t1, t1s, t2 = [], [], []
    for _ in range(reps):
        t = time.perf_counter(); one(); t1.append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter(); one_spots(); t1s.append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter(); many(); t2.append((time.perf_counter() - t) * 1e3)
    m1, m1s, m2 = float(np.median(t1)), float(np.median(t1s)), float(np.median(t2))
    return dict(system="COOKE", grid=[64, 32], fields=len(Hs), n_foci=len(foci), timer="host clock, end to end",
                full_trace_fields="ex, ey, r, theta compacted, copied back and mirrored per call",
                through_focus_ms=m1, through_focus_outputs="statistics only (spots=False)",
                through_focus_spots_ms=m1s, through_focus_spots_outputs="statistics + mirrored spots per focus (spots=True)",
                full_trace_fields_ms=m2, speedup_stats_only=m2 / m1, speedup_with_spots=m2 / m1s,
                through_focus_ms_all=t1, through_focus_spots_ms_all=t1s, full_trace_fields_ms_all=t2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ort_b200 as ort
    ctx = ort.Context(0)
    res = dict(gpu=gpu_info(), device=ctx.device_info()["name"], large=large(ort, ctx, a.reps),
               reference=reference(ort, ctx, a.reps))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
