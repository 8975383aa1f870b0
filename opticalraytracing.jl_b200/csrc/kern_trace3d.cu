// kern_trace3d.cu -- the 3-D skew real-ray trace kernels (sm_100a, FP64 CUDA cores).
//
//   k_grid<ARITH,RPT>  K1: pupil-grid sweep, replaces the hot loop of full_trace
//                      (src/PupilSampling.jl:115-138): RPT rays per thread, whole surface loop in
//                      registers, prescription in the constant bank (__grid_constant__ kernel
//                      parameter), fused mask / eps / r / theta / wavegrad epilogue, per-thread
//                      shifted-moment accumulation + warp-shuffle reduction for the spot statistics.
//                      Tile-strided CTAs, gridDim.x * gridDim.y = SMs * resident CTAs/SM * waves (grid_dims, ort_api.cu).
//                      SIMPLE instantiation for prescriptions of refracting spheres and planes (three-body surface loop).
//   k_grid_finalize    K6: deterministic fold of the per-CTA partials into ort_stats per field.
//   k_tile_scan / k_compact   ordered compaction in the reference's push! order (:134-137).
//   k_focus / k_compact_focus through-focus sweep: each ray traced once, evaluated on up to ORT_MAX_FOCI image planes.
//   k_rays<ARITH>      arbitrary rays, every surface recorded (raytrace(...,Vector{RealRay}) :34-65).
//   k_candidates<ARITH> K5: one CTA per candidate prescription staged in shared memory.
#include "kern.cuh"

// ------------------------------------------------------------------------------------------
// per-ray trace drivers shared by the kernels
// ------------------------------------------------------------------------------------------
struct Hit {               // what the grid epilogue needs from one traced ray
    double xs, ys;         // position at the stop surface   (xv[stop], yv[stop])
    double xf, yf;         // position at the last surface   (xv[end],  yv[end])
    unsigned flags;
    double opl;            // EXTENSION: optical path length incl. start term and reference sphere
};

// start term of the OPL (EXTENSION): collimated field -> n0 (x k1 + y k2), the lead of the start point
// over the plane wavefront through the origin; object point at z0 -> n0 (-z0) / k3.  Same operations as
// orc_opl_start.
__device__ __forceinline__ double strict_opl_start(const RayS& r, int mode, double n0, double y, double x, double z0)
{
    if (mode == 1) return SD(SM(n0, -z0), r.k3);
    return SM(n0, SA(SM(x, r.k1), SM(y, r.k2)));
}

// close the OPL on the reference sphere (EXTENSION): tau = -b - sign(rr) sqrt(b^2 - (|q|^2 - rr^2))
__device__ __forceinline__ double strict_opl_close(const RayS& r, const ort_field& f, double nlast)
{
    if (f.opd_radius == 0.0) return r.opl;
    const double qx = SS(r.x, f.opd_xc), qy = SS(r.y, f.opd_yc);
    const double b = SA(SM(qx, r.k1), SM(qy, r.k2));
    const double cq = SS(SA(SM(qx, qx), SM(qy, qy)), SM(f.opd_radius, f.opd_radius));
    const double sg = (f.opd_radius < 0.0) ? -1.0 : 1.0;
    const double tau = SS(-b, SM(sg, SQ(SS(SM(b, b), cq))));
    return SA(r.opl, SM(nlast, tau));
}

template <bool EXT, class SurfArray, bool POLY, bool XF>
__device__ __forceinline__ Hit trace_strict_impl(const SurfArray& S, int nsurf, int stop, double y, double x, double u, double v,
                                                 const ort_field* fld, double n0, double nlast, bool vignette, const double* poly,
                                                 int npoly, int* bad)
{
    RayS r;
    strict_init<XF>(r, y, x, u, v);
    if (EXT) r.opl = strict_opl_start(r, fld->mode, n0, y, x, fld->z0);
    Hit h; h.xs = h.ys = CUDART_NAN; h.opl = 0.0;
    for (int i = 0; i < nsurf; i++) {
        strict_step<EXT, POLY, XF>(S[i], r, vignette, (POLY && poly) ? poly + (size_t)i * npoly : nullptr, npoly);
        if (i == stop - 1) { h.xs = r.x; h.ys = r.y; }
    }
    h.xf = r.x; h.yf = r.y; h.flags = r.flags;
    if (EXT) h.opl = strict_opl_close(r, *fld, nlast);
    if (XF) *bad = r.bad;
    return h;
}

template <bool EXT, class SurfArray, bool POLY = false>
__device__ __forceinline__ Hit trace_strict(const SurfArray& S, int nsurf, int stop,
                                            double y, double x, double u, double v,
                                            const ort_field* fld = nullptr, double n0 = 1.0, double nlast = 1.0,
                                            bool vignette = false, const double* poly = nullptr, int npoly = 0)
{
    return trace_strict_impl<EXT, SurfArray, POLY, false>(S, nsurf, stop, y, x, u, v, fld, n0, nlast, vignette, poly, npoly, nullptr);
}

// the strict re-trace of guard-band rays lives out of line so it does not bloat the hot loop
template <bool EXT, class SurfArray, bool POLY = false>
__device__ __noinline__ Hit trace_strict_cold(const SurfArray& S, int nsurf, int stop,
                                              double y, double x, double u, double v,
                                              const ort_field* fld = nullptr, double n0 = 1.0, double nlast = 1.0,
                                              bool vignette = false, const double* poly = nullptr, int npoly = 0)
{
    return trace_strict<EXT, SurfArray, POLY>(S, nsurf, stop, y, x, u, v, fld, n0, nlast, vignette, poly, npoly);
}

// STRICT with the deferred slow paths (xdiv / xsqrt, ort_internal.cuh): a flagged ray is traced again with the intrinsics
template <bool EXT, class SurfArray, bool POLY = false>
__device__ __forceinline__ Hit trace_strict_xf(const SurfArray& S, int nsurf, int stop,
                                               double y, double x, double u, double v,
                                               const ort_field* fld = nullptr, double n0 = 1.0, double nlast = 1.0,
                                               bool vignette = false, const double* poly = nullptr, int npoly = 0)
{
    int bad = 0;
    const Hit h = trace_strict_impl<EXT, SurfArray, POLY, true>(S, nsurf, stop, y, x, u, v, fld, n0, nlast, vignette, poly, npoly, &bad);
    if (bad) return trace_strict_cold<EXT, SurfArray, POLY>(S, nsurf, stop, y, x, u, v, fld, n0, nlast, vignette, poly, npoly);
    return h;
}

// sign bit set iff a is NaN or +-Inf (exponent field all ones)
__device__ __forceinline__ int nonfinite_bit(double a) { return 0x7FEFFFFF - (hi32(a) & 0x7FFFFFFF); }

__device__ __forceinline__ bool is_nan_bits(double a)
{
    return (hi32(a) & 0x7FFFFFFF) > 0x7FF00000 ||
           ((hi32(a) & 0x7FFFFFFF) == 0x7FF00000 && __double2loint(a) != 0);
}

// RPT rays through the whole prescription in FAST arithmetic.  Two loops split at the stop surface
// (no per-step select for the stop capture).  amb[j] < 0 on return: ray j needs the strict re-trace
// (guard band hit, or a miss / TIR / non-finite value turned its position into NaN).
// R2ONLY: the caller only needs r^2 of the stop position (lean output sets): h.xs carries it, h.ys is unused -- three
// doubles instead of six live across the second surface loop.  KZCHECK = false: the prescription ends with a plain plane, so
// a non-finite Kz has already reached x, y (s = (t - z) / Kz) and needs no test of its own.
template <int RPT, bool EXT, class SurfArray, bool MIRROR = true, int SIMPLE = 0, bool R2ONLY = false, int POLY = 0, class QT = NoPolyK>
__device__ __forceinline__ void trace_fast(const SurfArray& S, int nsurf, int stop, double n0,
                                           const double* y, const double* x, const double* u,
                                           const double* v, Hit* h, int* amb,
                                           const ort_field* fld = nullptr, double nlast = 1.0, bool vignette = false,
                                           const double* K0 = nullptr, bool kzcheck = true, const double* poly = nullptr,
                                           int npoly = 0, const QT* Q = nullptr)
{
    RaysF<RPT> r;
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        if (K0) {           // collimated field: the optical direction is the same for every ray of the field
            r.x[j] = x[j]; r.y[j] = y[j]; r.z[j] = 0.0;
            r.Kx[j] = K0[0]; r.Ky[j] = K0[1]; r.Kz[j] = K0[2];
            r.amb[j] = 0; r.opl[j] = 0.0; r.vig[j] = 0;
        } else fast_init(r, j, n0, y[j], x[j], u[j], v[j]);
        if (EXT) {          // start term: K = n0 k, so n0 (x k1 + y k2) = x Kx + y Ky;  n0 (-z0) / k3 = -n0^2 z0 / Kz
            r.opl[j] = (fld->mode == 1) ? fast_div(-(n0 * n0) * fld->z0, r.Kz[j]) : fma(x[j], r.Kx[j], y[j] * r.Ky[j]);
        }
    }
    int i = 0;
    for (; i < stop; i++)
        if constexpr (POLY == 2) fast_step<RPT, EXT, MIRROR, SIMPLE, 2>(S[i], r, vignette, nullptr, 0, 0, &Q->r[i]);
        else fast_step<RPT, EXT, MIRROR, SIMPLE, POLY>(S[i], r, vignette, (POLY && poly) ? poly + (size_t)i * npoly : nullptr, npoly, nsurf * npoly);
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        if (R2ONLY) { h[j].xs = fma(r.x[j], r.x[j], r.y[j] * r.y[j]); h[j].ys = 0.0; }
        else { h[j].xs = r.x[j]; h[j].ys = r.y[j]; }
    }
    for (; i < nsurf; i++)
        if constexpr (POLY == 2) fast_step<RPT, EXT, MIRROR, SIMPLE, 2>(S[i], r, vignette, nullptr, 0, 0, &Q->r[i]);
        else fast_step<RPT, EXT, MIRROR, SIMPLE, POLY>(S[i], r, vignette, (POLY && poly) ? poly + (size_t)i * npoly : nullptr, npoly, nsurf * npoly);
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        h[j].xf = r.x[j]; h[j].yf = r.y[j];
        h[j].flags = (EXT && r.vig[j]) ? ORT_FLAG_VIGN : 0u;
        amb[j] = r.amb[j] | nonfinite_bit(r.x[j]) | nonfinite_bit(r.y[j]);
        if (kzcheck) amb[j] |= nonfinite_bit(r.Kz[j]);
        h[j].opl = 0.0;
        if (EXT) {          // reference sphere in optical cosines: n tau = -q.K - sgn(rr) sgn(n) sqrt((q.K)^2 - n^2 (|q|^2 - rr^2))
            double opl = r.opl[j];
            if (fld->opd_radius != 0.0) {
                const double qx = r.x[j] - fld->opd_xc, qy = r.y[j] - fld->opd_yc;
                const double bK = fma(qx, r.Kx[j], qy * r.Ky[j]);
                const double cq = fma(qx, qx, fma(qy, qy, -fld->opd_radius * fld->opd_radius));
                const double d = fma(bK, bK, -(nlast * nlast) * cq);
                double sq = fast_sqrt(d);
                if ((fld->opd_radius < 0.0) != (nlast < 0.0)) sq = -sq;
                opl = opl - bK - sq;
                amb[j] |= nonfinite_bit(opl);
            }
            h[j].opl = opl;
        }
    }
}

// ------------------------------------------------------------------------------------------
// K1: pupil-grid sweep
// ------------------------------------------------------------------------------------------
// Spot statistics: every CTA first traces the field's centre ray (row ny/2, column 0) and uses its
// (ex, ey) as a common shift c, so the per-thread accumulation is 2 DADD + 2 DFMA per axis on
// d = e - c (no cancellation: |mean - c| is of the order of the spot size) and all partial sums of
// a field are plain sums -- folded in a fixed order, hence bit-reproducible run to run.
struct RawAcc {
    int n, nflag_lo, nflag_hi;                  // counts; nflag_* pack (miss, tir) and (domain, clip) as 16+16 bits
    double s1x, s2x, s1y, s2y, rmax;            // rmax holds r (strict) or r^2 (fast)
    double s1o, s2o; int nvig;                  // EXTENSION: OPD moments, vignetted count
    int nstrict;                                // rays that went through the strict re-trace
};

__device__ __forceinline__ void raw_add(RawPart& p, const RawPart& q)
{
    p.n += q.n; p.s1x += q.s1x; p.s2x += q.s2x; p.s1y += q.s1y; p.s2y += q.s2y;
    p.rmax = fmax(p.rmax, q.rmax);
    p.nmiss += q.nmiss; p.ntir += q.ntir; p.ndom += q.ndom; p.nclip += q.nclip;
    p.s1o += q.s1o; p.s2o += q.s2o; p.nvig += q.nvig; p.nstrict += q.nstrict;
}

__device__ __forceinline__ void raw_warp_reduce(RawPart& p)
{
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        p.n += __shfl_down_sync(0xffffffffu, p.n, d);
        p.s1x += __shfl_down_sync(0xffffffffu, p.s1x, d);
        p.s2x += __shfl_down_sync(0xffffffffu, p.s2x, d);
        p.s1y += __shfl_down_sync(0xffffffffu, p.s1y, d);
        p.s2y += __shfl_down_sync(0xffffffffu, p.s2y, d);
        p.rmax = fmax(p.rmax, __shfl_down_sync(0xffffffffu, p.rmax, d));
        p.nmiss += __shfl_down_sync(0xffffffffu, p.nmiss, d);
        p.ntir += __shfl_down_sync(0xffffffffu, p.ntir, d);
        p.ndom += __shfl_down_sync(0xffffffffu, p.ndom, d);
        p.nclip += __shfl_down_sync(0xffffffffu, p.nclip, d);
        p.s1o += __shfl_down_sync(0xffffffffu, p.s1o, d);
        p.s2o += __shfl_down_sync(0xffffffffu, p.s2o, d);
        p.nvig += __shfl_down_sync(0xffffffffu, p.nvig, d);
        p.nstrict += __shfl_down_sync(0xffffffffu, p.nstrict, d);
    }
}

// deterministic: shuffle tree inside each warp, then thread 0 folds the warp leaders in warp order
template <int NWARPS>
__device__ __forceinline__ void raw_block_reduce(RawPart& p, RawPart* smem /* [NWARPS] */)
{
    raw_warp_reduce(p);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) smem[warp] = p;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < NWARPS; w++) raw_add(p, smem[w]);
}

// everything after the trace for one ray: stop-radius mask (:131-132), strict re-trace of guard-band
// rays, outputs (:133-137, :165-167) and statistics
__device__ __forceinline__ void field_slopes(const ort_field& fld, double y0, double x0, double& u, double& v)
{
    u = fld.u; v = fld.v;
    if (fld.mode == 1) {                         // RayBasis: :124-127 then tan at :38-39
        u = tan(SD(SS(fld.ybar, y0), fld.z0));
        v = tan(SD(-x0, fld.z0));
    }
}

// LEAN = 1: the caller wants exactly the spot diagram and the mask (ex, ey, mask -- BASELINE config 2's 17 B per
// ray): no per-pointer null tests, 32-bit indexing off per-field base pointers.  LEAN = 2: statistics only (config 3's
// 0 B per ray): no stores at all.  LEAN = 0: any combination of outputs.
// LEAN == 1 stores go through lp (this ray's slots in ex, ey, mask[, opd]): the kernel derives the three pointers once per
// tile and the rays of a thread sit at compile-time offsets from them, instead of 64-bit address arithmetic per ray and array.
struct LeanPtrs { double *ex, *ey, *opd; uint8_t* mask; };
template <int ARITH, int EXTK, int LEAN, bool R2ONLY = false, int POLYK = 0>
__device__ __forceinline__ int grid_epilogue(const Presc& P, const GridArgs& A, const ort_field& fld,
                                             const double* ysf, Hit h, int amb, unsigned idx,
                                             bool valid, size_t fbase, double cx, double cy, double co, RawAcc& acc,
                                             const LeanPtrs& lp)
{
    constexpr bool EXT = EXTK != 0;
    const size_t o = fbase + idx;
    const bool vignette = EXTK == 1 && (A.ext & ORT_EXT_VIGNETTE);
    double ri = 0.0, r2 = 0.0;
    bool clip = false;
    if (ARITH == ORT_ARITH_FAST) {
        r2 = R2ONLY ? h.xs : fma(h.xs, h.xs, h.ys * h.ys);
        amb |= tiny_vs_bit(r2 - A.a_stop2, A.a_stop2);                  // within 2^-30 of the stop edge
        clip = r2 > A.a_stop2;
    }
    const bool sv = (ARITH == ORT_ARITH_STRICT) || amb < 0;
    if (sv) {
        if (ARITH != ORT_ARITH_STRICT) {            // rare in FAST mode: recompute the ray's inputs here and re-trace it
            const unsigned iy = idx / (unsigned)A.nx, ix = idx - iy * (unsigned)A.nx;
            const double y0 = __ldg(ysf + iy), x0 = __ldg(A.xs + ix);
            double u, v; field_slopes(fld, y0, x0, u, v);
            h = trace_strict_cold<EXT, decltype(P.s), POLYK != 0>(P.s, P.nsurf, A.stop, y0, x0, u, v, &fld, P.n0, P.nlast, vignette, P.poly, P.npoly);
        }                                           // STRICT: h is the reference-arithmetic trace already (k_grid)
        ri = jl_hypot(h.xs, h.ys);                                      // :131
        clip = ri > A.a_stop;
        r2 = ri * ri;
        if (valid) {        // miss / TIR / domain flags can only come out of a strict trace: counted here, off the fast path
            acc.nstrict++;
            acc.nflag_lo += (h.flags & ORT_FLAG_MISS ? 1 : 0) + (h.flags & ORT_FLAG_TIR ? 0x10000 : 0);
            acc.nflag_hi += (h.flags & ORT_FLAG_DOMAIN ? 1 : 0);
        }
    } else if (!LEAN && A.r) {
        ri = (r2 > 0.0) ? fast_sqrt(r2) : r2;
    }
    const bool vig = EXTK == 1 && (h.flags & ORT_FLAG_VIGN);
    // :132 (+ surface apertures).  A ray that stayed on the fast path is finite by construction (non-finite
    // values set amb), so the NaN tests are only needed after a strict trace.
    const bool drop = clip || vig || (sv && (is_nan_bits(h.xf) || is_nan_bits(h.yf)));
    const unsigned flags = h.flags | (clip ? ORT_FLAG_CLIP : 0u);
    const int kept = valid && !drop;
    const double ex = h.xf;                                             // :135
    const double ey = SS(h.yf, fld.h_prime);                            // :134  (one subtraction: nothing to contract)
    double opd = 0.0;
    if (EXT && (A.ext & ORT_EXT_OPD)) opd = SM(SS(h.opl, fld.opl_ref), A.opd_scale);
    if (LEAN) {
        if (valid) {
            if (LEAN == 1) { *lp.ex = ex; *lp.ey = ey; *lp.mask = (uint8_t)kept; }
            if (LEAN == 1 && EXT) *lp.opd = opd;                    // the OPD sweep's output set: ex, ey, opd, mask
            if (EXTK == 1) acc.nvig += vig ? 1 : 0;
            if (clip) acc.nflag_hi += 0x10000;
        }
    } else if (valid) {
        if (A.ex) A.ex[o] = ex;
        if (A.ey) A.ey[o] = ey;
        if (A.r) A.r[o] = ri;                                           // :136
        if (A.theta) A.theta[o] = atan2(h.ys, h.xs);                    // :133
        if (A.wx) A.wx[o] = SD(SM(ex, A.wg_nu), A.wg_lambda);           // :166
        if (A.wy) A.wy[o] = SD(SM(ey, A.wg_nu), A.wg_lambda);
        if (EXT && A.opd) A.opd[o] = opd;
        if (A.mask) A.mask[o] = (uint8_t)kept;
        if (A.flags) A.flags[o] = (uint8_t)flags;
        acc.nflag_hi += clip ? 0x10000 : 0;
        if (EXT) acc.nvig += vig ? 1 : 0;
    }
    if (kept) {
        const double dx = ex - cx, dy = ey - cy;
        acc.s1x += dx; acc.s2x = fma(dx, dx, acc.s2x);
        acc.s1y += dy; acc.s2y = fma(dy, dy, acc.s2y);
        { const double rv = (ARITH == ORT_ARITH_STRICT) ? ri : r2; if (rv > acc.rmax) acc.rmax = rv; }   // kept rays: never NaN
        if (EXT) { const double dd = opd - co; acc.s1o += dd; acc.s2o = fma(dd, dd, acc.s2o); }
        acc.n++;
    }
    return kept;
}

// SIMPLE (FAST only): the prescription holds refracting spheres and planes only (Presc::simple): ORT_SIMPLE_RPT rays per
// thread through the three-body fast_step<.., SIMPLE>, ORT_BPSP resident CTAs/SM.
// EXTK: 0 = the reference's outputs only; 1 = extensions (OPD and / or per-surface apertures, chosen at run time; polynomial
// terms in STRICT); 2 = OPD only (no aperture test compiled in: the instantiation of OPD sweeps over SIMPLE prescriptions).
template <int ARITH, int RPT, int EXTK, int LEAN = 0, bool MIRROR = true, int SIMPLE = 0, int POLYK = 0>
__global__ void __launch_bounds__(ORT_TILE, (ARITH == ORT_ARITH_FAST) ? POLYK ? ORT_BPS_POLY : (SIMPLE == 2 ? ORT_BPSC : SIMPLE ? (EXTK ? ORT_BPSE : ORT_BPSP) : (RPT == 1 ? ORT_BPS1 : (EXTK ? ORT_BPS2E : ORT_BPS2))) : ORT_BPSS)
k_grid(const __grid_constant__ Presc P, const __grid_constant__ GridArgs A, const __grid_constant__ typename PolyArg<POLYK>::type Q)
{
    constexpr bool EXT = EXTK != 0;
    __shared__ RawPart s_part[ORT_TILE / 32];
    __shared__ double s_shift[3];
    const int f = blockIdx.y;
    const ort_field& fld = A.fields[f];
    const unsigned NN = A.NN;
    const unsigned nsub = (NN + ORT_TILE - 1) / ORT_TILE;            // 256-ray sub-tiles (compaction unit)
    const unsigned ntiles = (nsub + RPT - 1) / RPT;
    const size_t fbase = (size_t)f * NN;
    const double* ysf = A.ys + (size_t)f * A.ys_stride;
    const unsigned ysoff = (unsigned)f * (unsigned)A.ys_stride;      // n_fields * ny < 2^31
    const bool vignette = EXTK == 1 && (A.ext & ORT_EXT_VIGNETTE);

    RawAcc acc;
    acc.n = acc.nflag_lo = acc.nflag_hi = acc.nvig = acc.nstrict = 0;
    acc.s1x = acc.s2x = acc.s1y = acc.s2y = acc.s1o = acc.s2o = 0.0; acc.rmax = -CUDART_INF;

    if (threadIdx.x == 0) {                      // common shift of this field: its centre ray
        const double y0 = __ldg(ysf + A.ny / 2), x0 = __ldg(A.xs);
        double u, v; field_slopes(fld, y0, x0, u, v);
        Hit h; int amb = 0;
        if (ARITH == ORT_ARITH_FAST)
            trace_fast<1, EXT, decltype(P.s), SIMPLE == 0, SIMPLE, false, POLYK, typename PolyArg<POLYK>::type>(P.s, P.nsurf, A.stop, P.n0, &y0, &x0, &u, &v, &h, &amb, &fld, P.nlast, vignette,
                                                                   nullptr, true, P.poly, P.npoly, &Q);
        if (ARITH == ORT_ARITH_STRICT || amb < 0)
            h = trace_strict_cold<EXT, decltype(P.s), (EXT && ARITH == ORT_ARITH_STRICT) || POLYK != 0>(P.s, P.nsurf, A.stop, y0, x0, u, v, &fld, P.n0,
                                                                                                  P.nlast, vignette, P.poly, P.npoly);
        const double ey = h.yf - fld.h_prime;
        const bool bad = nonfinite_bit(h.xf) < 0 || nonfinite_bit(ey) < 0;
        s_shift[0] = bad ? 0.0 : h.xf;
        s_shift[1] = bad ? 0.0 : ey;
        const double od = (h.opl - fld.opl_ref) * A.opd_scale;
        s_shift[2] = (!EXT || !(A.ext & ORT_EXT_OPD) || bad || nonfinite_bit(od) < 0) ? 0.0 : od;     // no OPD asked for: its statistics stay 0
    }
    __syncthreads();
    const double cx = s_shift[0], cy = s_shift[1], co = s_shift[2];
    // the lean output sets need only r^2 of the stop position; a prescription that ends with a plain plane (full_trace's image
    // plane) needs no finiteness test on Kz
    constexpr bool R2ONLY = ARITH == ORT_ARITH_FAST && LEAN != 0;
    const bool kzcheck = P.s[P.nsurf - 1].kcode != SURF_PLANE;

    // collimated field (mode 0): K = n0 normalize([v, u, 1]) once per thread, not once per ray
    const bool collimated = (fld.mode == 0);
    double K0[3] = {0.0, 0.0, 0.0};
    if (ARITH == ORT_ARITH_FAST && collimated) {
        const double inv = P.n0 * fast_rsqrt(fma(fld.v, fld.v, fma(fld.u, fld.u, 1.0)));
        K0[0] = fld.v * inv; K0[1] = fld.u * inv; K0[2] = inv;
    }
    // (iy, ix) of this thread's rays advance by a constant (dq, dr) per tile: no division in the loop
    const unsigned nxu = (unsigned)A.nx;
    const unsigned step = gridDim.x * (RPT * ORT_TILE);
    const unsigned dq = step / nxu, dr = step - dq * nxu;
    unsigned iyj[RPT], ixj[RPT];
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const unsigned i0 = (blockIdx.x * RPT + j) * ORT_TILE + threadIdx.x;
        iyj[j] = i0 / nxu; ixj[j] = i0 - iyj[j] * nxu;
    }

    for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        double y0[RPT], x0[RPT], u[RPT], v[RPT];
        unsigned idx[RPT];
        bool valid[RPT];
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            const unsigned i0 = (tile * RPT + j) * ORT_TILE + threadIdx.x;
            valid[j] = i0 < NN;
            idx[j] = min(i0, NN - 1);            // padded lanes trace a ray of the last row: the warp stays convergent
            const unsigned iy = min(iyj[j], (unsigned)A.ny - 1), ix = ixj[j];       // y outer, x inner (:123); ix < nx always
            y0[j] = __ldg(A.ys + (ysoff + iy)); x0[j] = __ldg(A.xs + ix);      // 32-bit offsets: one IMAD.WIDE each
            u[j] = 0.0; v[j] = 0.0;              // collimated FAST sweeps take the direction from K0 (the strict re-trace derives its own)
            ixj[j] += dr; iyj[j] += dq;
            if (ixj[j] >= nxu) { ixj[j] -= nxu; iyj[j]++; }
        }
        if (!collimated || ARITH != ORT_ARITH_FAST) {        // one uniform test per tile
#pragma unroll
            for (int j = 0; j < RPT; j++) field_slopes(fld, y0[j], x0[j], u[j], v[j]);
        }
        Hit h[RPT];
        int amb[RPT];
        if (ARITH == ORT_ARITH_FAST)
            trace_fast<RPT, EXT, decltype(P.s), MIRROR, SIMPLE, R2ONLY, POLYK, typename PolyArg<POLYK>::type>(P.s, P.nsurf, A.stop, P.n0, y0, x0, u, v, h, amb, &fld, P.nlast, vignette,
                                                                collimated ? K0 : nullptr, kzcheck, P.poly, P.npoly, &Q);
        else {      // STRICT: the thread's RPT rays advance surface by surface together (independent chains of the slow ops: / and sqrt)
            RayS r[RPT];
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                strict_init<ORT_STRICT_XF>(r[j], y0[j], x0[j], u[j], v[j]);
                if (EXT) r[j].opl = strict_opl_start(r[j], fld.mode, P.n0, y0[j], x0[j], fld.z0);
                h[j].xs = h[j].ys = CUDART_NAN; h[j].opl = 0.0;
            }
            const int nsurf = P.nsurf, stop = A.stop;
            for (int i = 0; i < nsurf; i++) {
#pragma unroll
                for (int j = 0; j < RPT; j++) {
                    strict_step<EXT, EXT, ORT_STRICT_XF>(P.s[i], r[j], vignette, (EXT && P.poly) ? P.poly + (size_t)i * P.npoly : nullptr, P.npoly);
                    if (i == stop - 1) { h[j].xs = r[j].x; h[j].ys = r[j].y; }
                }
            }
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                h[j].xf = r[j].x; h[j].yf = r[j].y; h[j].flags = r[j].flags;
                if (EXT) h[j].opl = strict_opl_close(r[j], fld, P.nlast);
                // an operand left the range of xdiv / xsqrt's fast path (ort_internal.cuh): this ray once more with the
                // library's division and square root
                if (ORT_STRICT_XF && r[j].bad)
                    h[j] = trace_strict_cold<EXT, decltype(P.s), EXT>(P.s, P.nsurf, A.stop, y0[j], x0[j], u[j], v[j], &fld, P.n0, P.nlast, vignette, P.poly, P.npoly);
            }
        }
        int keptj[RPT];
        LeanPtrs lp0 = {nullptr, nullptr, nullptr, nullptr};
        if (LEAN == 1) {                        // valid rays of this thread: element e0 + j * ORT_TILE of the field's arrays
            const size_t e0 = fbase + (size_t)tile * (RPT * ORT_TILE) + threadIdx.x;
            lp0.ex = A.ex + e0; lp0.ey = A.ey + e0; lp0.mask = A.mask + e0;
            if (EXT) lp0.opd = A.opd + e0;
        }
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            if (ARITH != ORT_ARITH_FAST) amb[j] = 0;
            const LeanPtrs lp = {lp0.ex + j * ORT_TILE, lp0.ey + j * ORT_TILE, EXT ? lp0.opd + j * ORT_TILE : nullptr, lp0.mask + j * ORT_TILE};
            keptj[j] = grid_epilogue<ARITH, EXTK, LEAN, R2ONLY, POLYK>(P, A, fld, ysf, h[j], amb[j], idx[j], valid[j],
                                                                fbase, cx, cy, co, acc, lp);
        }
        if (LEAN != 2 && A.tile_counts) {       // ordered compaction requested: kept rays per 256-ray sub-tile (one uniform test per tile)
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                const int c = __syncthreads_count(keptj[j]);
                const unsigned sub = tile * RPT + j;
                if (threadIdx.x == 0 && sub < nsub) A.tile_counts[(size_t)f * nsub + sub] = c;
            }
        }
    }
    RawPart p;
    p.n = acc.n; p.s1x = acc.s1x; p.s2x = acc.s2x; p.s1y = acc.s1y; p.s2y = acc.s2y; p.rmax = acc.rmax;
    p.cx = cx; p.cy = cy; p.co = co; p.s1o = acc.s1o; p.s2o = acc.s2o; p.nvig = acc.nvig; p.nstrict = acc.nstrict;
    p.nmiss = acc.nflag_lo & 0xFFFF; p.ntir = acc.nflag_lo >> 16; p.ndom = acc.nflag_hi & 0xFFFF; p.nclip = acc.nflag_hi >> 16;
    raw_block_reduce<ORT_TILE / 32>(p, s_part);
    if (threadIdx.x == 0) {
        if (ARITH != ORT_ARITH_STRICT) p.rmax = sqrt(p.rmax);
        A.partials[(size_t)f * gridDim.x + blockIdx.x] = p;
    }
}

// K6: fold the per-CTA partial sums of one field in a fixed order (bit-reproducible run to run) and
// convert the shifted raw moments to (n, mean, M2).
__global__ void __launch_bounds__(256) k_grid_finalize(const RawPart* partials, int nparts, ort_stats* stats)
{
    __shared__ RawPart s_part[8];
    const int f = blockIdx.x;
    RawPart p;
    p.n = 0; p.s1x = p.s2x = p.s1y = p.s2y = p.s1o = p.s2o = 0.0; p.rmax = -CUDART_INF; p.cx = p.cy = p.co = 0.0;
    p.nmiss = p.ntir = p.ndom = p.nclip = p.nvig = p.nstrict = 0;
    for (int j = threadIdx.x; j < nparts; j += 256) raw_add(p, partials[(size_t)f * nparts + j]);
    raw_block_reduce<8>(p, s_part);
    if (threadIdx.x == 0) {
        const RawPart& p0 = partials[(size_t)f * nparts];
        ort_stats s;
        s.n_kept = p.n;
        if (p.n > 0) {
            const double n = (double)p.n;
            s.mean_x = p0.cx + p.s1x / n; s.mean_y = p0.cy + p.s1y / n;
            s.m2_x = fmax(p.s2x - p.s1x * p.s1x / n, 0.0);
            s.m2_y = fmax(p.s2y - p.s1y * p.s1y / n, 0.0);
            s.r_max = p.rmax;
            s.mean_opd = p0.co + p.s1o / n;
            s.m2_opd = fmax(p.s2o - p.s1o * p.s1o / n, 0.0);
        } else { s.mean_x = s.mean_y = s.m2_x = s.m2_y = s.mean_opd = s.m2_opd = 0.0; s.r_max = -CUDART_INF; }
        s.n_miss = p.nmiss; s.n_tir = p.ntir; s.n_domain = p.ndom; s.n_clip = p.nclip; s.n_vig = p.nvig; s.n_strict = p.nstrict;
        stats[f] = s;
    }
}

// Exclusive scan of the per-tile kept counts, two levels: every CTA scans one chunk of SCAN_CHUNK tiles
// in place (coalesced, 8 tiles per thread, warp-shuffle scans) and publishes the chunk total; k_compact
// adds the totals of the preceding chunks (<= a few dozen values).
#define SCAN_CHUNK 2048
__global__ void __launch_bounds__(256) k_tile_scan(int* counts, int* chunk_tot, unsigned ntiles, unsigned nchunks)
{
    __shared__ int s_warp[8];
    const unsigned f = blockIdx.y, chunk = blockIdx.x;
    int* c = counts + (size_t)f * ntiles + (size_t)chunk * SCAN_CHUNK;
    const unsigned n = min((unsigned)SCAN_CHUNK, ntiles - chunk * SCAN_CHUNK);
    const unsigned base = threadIdx.x * 8;
    int v[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) { v[j] = (base + j < n) ? c[base + j] : 0; sum += v[j]; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int woff = 0, tot = 0;
    for (int w = 0; w < 8; w++) { if (w < warp) woff += s_warp[w]; tot += s_warp[w]; }
    int run = woff + incl - sum;
#pragma unroll
    for (int j = 0; j < 8; j++) { if (base + j < n) c[base + j] = run; run += v[j]; }
    if (threadIdx.x == 0) chunk_tot[(size_t)f * nchunks + chunk] = tot;
}

// second level: exclusive scan of the chunk totals of one field (one CTA per field; <= 4096 chunks for 2^31 rays)
__global__ void __launch_bounds__(256) k_chunk_scan(int* chunk_tot, unsigned nchunks)
{
    __shared__ int s_warp[8];
    int* c = chunk_tot + (size_t)blockIdx.x * nchunks;
    int carry = 0;
    for (unsigned base0 = 0; base0 < nchunks; base0 += 256) {
        const unsigned i = base0 + threadIdx.x;
        const int v = (i < nchunks) ? c[i] : 0;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int woff = 0, tot = 0;
        for (int w = 0; w < 8; w++) { if (w < warp) woff += s_warp[w]; tot += s_warp[w]; }
        if (i < nchunks) c[i] = carry + woff + incl - v;
        carry += tot;
        __syncthreads();
    }
}

// Index of thread tid's ray among the kept rays of field f (m: the ray is kept), in a compaction kernel of one CTA per
// (tile, field).  Every thread of the CTA calls it: it synchronises the CTA.  The kernel passes tid = threadIdx.x and
// ntiles: read or computed in here they compile to other code (threadIdx.x loses the bound of the kernel's launch
// bounds, and the loop over the preceding warps unrolls differently: 30 registers instead of 22).
__device__ __forceinline__ int compact_offset(const CompactArgs& C, unsigned tile, unsigned f, unsigned ntiles, unsigned tid,
                                              int m)
{
    __shared__ int s_warp[ORT_TILE / 32];
    const unsigned ball = __ballot_sync(0xffffffffu, m);
    const int lane = tid & 31, warp = tid >> 5;
    if (lane == 0) s_warp[warp] = __popc(ball);
    __syncthreads();
    int off = C.tile_offsets[(size_t)f * ntiles + tile];
    {   // + scanned total of the preceding chunks of this field
        const unsigned nchunks = (ntiles + SCAN_CHUNK - 1) / SCAN_CHUNK, mychunk = tile / SCAN_CHUNK;
        const int* ct = C.tile_offsets + (size_t)gridDim.y * ntiles + (size_t)f * nchunks;
        off += ct[mychunk];
    }
    for (int w = 0; w < warp; w++) off += s_warp[w];
    return off + __popc(ball & ((1u << lane) - 1u));
}

// order-preserving scatter of up to 7 arrays: one CTA per (tile, field)
__global__ void __launch_bounds__(ORT_TILE) k_compact(CompactArgs C)
{
    const unsigned tile = blockIdx.x, f = blockIdx.y;
    const unsigned ntiles = (C.NN + ORT_TILE - 1) / ORT_TILE;
    const unsigned i = tile * ORT_TILE + threadIdx.x;
    const size_t fbase = (size_t)f * C.NN;
    const int m = (i < C.NN) ? C.mask[fbase + i] : 0;
    const int off = compact_offset(C, tile, f, ntiles, threadIdx.x, m);
    if (m) {
#pragma unroll
        for (int a = 0; a < 7; a++)
            if (C.src[a]) C.dst[a][fbase + off] = C.src[a][fbase + i];
    }
}

// ------------------------------------------------------------------------------------------
// through-focus sweep: every ray traced once up to the image plane, then M image planes (foci)
// ------------------------------------------------------------------------------------------
// The image plane is the last row of the extended layout ([Inf 0 1], t[end-1] = focus, src/PupilSampling.jl:111-114).
// Nothing before it depends on the focus: the stop clip, the miss / TIR / domain flags, r and theta are fixed one
// surface earlier, and the position on a plane is one transfer from the state after the last glass surface.  k_focus
// keeps that state per ray in five or six doubles (FocusRay) and evaluates the transfer once per focus with the plane
// lines of the body k_grid would run -- strict_step's for STRICT, fast_step's plain-plane body for FAST, restated
// operation for operation -- so every per-ray output is bit-identical to a k_grid sweep of the layout with
// t[end-1] = foci[j].
//
// FAST: fast_div(n, d) = n * r with r a function of d alone, so the reciprocal of Kz is taken once per ray and a focus
// costs one DADD, one DMUL and two DFMA (x, y) plus the statistics.  The position is affine in the rounded (t - z), so
// it is non-finite at some focus iff it is at the smallest or the largest one: those two decide the strict re-trace.
//
// Drop rule: a ray is dropped for every focus of its field if the stop clips it, or if its position is NaN at ANY focus
// (only a ray with k3 = 0 after the last glass surface can be NaN at one focus and not at another).  mask, flags, r,
// theta and the kept count are therefore per field; for every ray that is finite at all foci this is full_trace's own
// per-focus rule.
struct FocusRay {
    // STRICT state: a0 = x, a1 = y, a2 = sprev, a3 = v, a4 = u.  FAST state: a0 = x, a1 = y, a2 = z, a3 = Kx, a4 = Ky,
    // a5 = 1 / Kz as fast_div forms it.
    double a0, a1, a2, a3, a4, a5;
};

// strict_step's first and last position lines at a plane (sag s = 0), with t = the focus: src/PupilSampling.jl:46-47, 52-53
__device__ __forceinline__ void focus_pos_strict(const FocusRay& q, double t, double& xf, double& yf)
{
    const double ti = SS(t, q.a2);
    double y = SA(q.a1, SM(q.a4, ti));
    double x = SA(q.a0, SM(q.a3, ti));
    y = SA(y, SM(0.0, q.a4));
    x = SA(x, SM(0.0, q.a3));
    xf = x; yf = y;
}

// fast_step's plain-plane body: s = fast_div(t - z, Kz); x = fma(s, Kx, x); y = fma(s, Ky, y)
__device__ __forceinline__ void focus_pos_fast(const FocusRay& q, double t, double& xf, double& yf)
{
    const double s = (t - q.a2) * q.a5;
    xf = fma(s, q.a3, q.a0);
    yf = fma(s, q.a4, q.a1);
}

// the reciprocal fast_div multiplies its numerator by
__device__ __forceinline__ double fast_div_rcp(double d)
{
    double r = mufu_rcp(d);
    const double e = fma(-d, r, 1.0);
    return fma(r, fma(e, e, e), r);
}

struct FocusS {                     // strict state after surface nsurf - 2
    FocusRay q;
    double xs, ys;                  // position at the stop surface
    unsigned flags;                 // ORT_FLAG_* of surfaces 0 .. nsurf-2, plus FOCUS_TIR_LAST (see below)
};

// Internal bit of FocusS::flags: the image plane refracts with total internal reflection IF strict_step's plane normal is
// m = (0, 0, -1).  strict_step uses that normal when the position on the plane has |x|, |y| < 1e150; otherwise it
// normalises (sgn x / sqrt(Inf - (x^2 + y^2)), ..., -1), which is the same m while x^2 + y^2 is finite and NaN (no flag)
// when it is not.  So the flag is raised iff this bit is set and x^2 + y^2 on the plane is finite -- decided by k_focus
// once the positions at the foci are known.
#define FOCUS_TIR_LAST 0x80u

// STRICT trace through surfaces 0 .. nsurf-2 (k_grid's per-surface body), the stop position at stop - 1, and the image
// plane's TIR decision (FOCUS_TIR_LAST)
template <bool XF>
__device__ __forceinline__ FocusS focus_strict_impl(const Presc& P, int stop, double y, double x, double u, double v, int* bad)
{
    RayS r;
    strict_init<XF>(r, y, x, u, v);
    FocusS o; o.xs = o.ys = CUDART_NAN;
    const int ns = P.nsurf - 1;
    for (int i = 0; i < ns; i++) {
        strict_step<false, false, XF>(P.s[i], r);
        if (i == stop - 1) { o.xs = r.x; o.ys = r.y; }
    }
    const SurfK& S = P.s[ns];
    double dot = SA(0.0, SM(r.k1, 0.0)); dot = SA(dot, SM(r.k2, 0.0)); dot = SA(dot, SM(r.k3, -1.0));
    const double gam = -dot;
    const double Dr = SS(1.0, SM(S.etasq, SS(1.0, SM(gam, gam))));
    if (Dr < 0.0) r.flags |= FOCUS_TIR_LAST;
    o.q.a0 = r.x; o.q.a1 = r.y; o.q.a2 = r.sprev; o.q.a3 = r.v; o.q.a4 = r.u; o.q.a5 = 0.0;
    o.flags = r.flags;
    if (XF) *bad = r.bad;
    return o;
}

__device__ __noinline__ FocusS focus_strict_cold(const Presc& P, int stop, double y, double x, double u, double v)
{
    return focus_strict_impl<false>(P, stop, y, x, u, v, nullptr);
}

// k_grid's grid shape (tile-strided CTAs, blockIdx.y = field) and surface bodies.  Statistics per (field, focus): the
// shifted moments of k_grid (the shift of focus j is the field's centre ray at focus j); per tile and focus the warp
// reduces by shuffle and lane 0 adds into its own row of s_acc, so every partial is a fixed-order sum.  Counts, r_max
// and flags are the same for every focus of a field and go into every record.
template <int ARITH, int RPT, bool MIRROR, int SIMPLE>
__global__ void __launch_bounds__(ORT_TILE, 2)
k_focus(const __grid_constant__ Presc P, const __grid_constant__ FocusArgs F)
{
    constexpr int NWARPS = ORT_TILE / 32;
    __shared__ double s_acc[NWARPS][ORT_MAX_FOCI][4];
    __shared__ double s_c[ORT_MAX_FOCI][2];
    __shared__ RawPart s_part[NWARPS];
    __shared__ RawPart s_p0;
    __shared__ double2 s_xy[RPT][ORT_TILE];     // FAST: position at the stop, kept out of registers (r^2 recomputed from it)
    // per-thread counters and r_max, each thread in its own slot: registers stay with the rays (no spills at RPT = 3)
    __shared__ int s_cnt[4][ORT_TILE];          // kept, (miss, tir) and (domain, clip) packed 16 + 16 as in RawAcc, strict
    __shared__ double s_rmax[ORT_TILE];
    const GridArgs& A = F.G;
    const int M = F.n_foci;
    const int f = blockIdx.y;
    const ort_field& fld = A.fields[f];
    const unsigned NN = A.NN;
    const unsigned nsub = (NN + ORT_TILE - 1) / ORT_TILE;
    const unsigned ntiles = (nsub + RPT - 1) / RPT;
    const size_t fbase = (size_t)f * NN;
    const double* ysf = A.ys + (size_t)f * A.ys_stride;
    const unsigned ysoff = (unsigned)f * (unsigned)A.ys_stride;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    for (int i = threadIdx.x; i < NWARPS * ORT_MAX_FOCI * 4; i += ORT_TILE) (&s_acc[0][0][0])[i] = 0.0;
    if (threadIdx.x == 0) {                      // common shift of every focus: the field's centre ray there
        const double y0 = __ldg(ysf + A.ny / 2), x0 = __ldg(A.xs);
        double u, v; field_slopes(fld, y0, x0, u, v);
        const FocusS c = focus_strict_cold(P, A.stop, y0, x0, u, v);
        for (int m = 0; m < M; m++) {
            double xf, yf; focus_pos_strict(c.q, F.foci[m], xf, yf);
            const double ey = yf - fld.h_prime;
            const bool bad = nonfinite_bit(xf) < 0 || nonfinite_bit(ey) < 0;
            s_c[m][0] = bad ? 0.0 : xf;
            s_c[m][1] = bad ? 0.0 : ey;
        }
    }
    __syncthreads();

    int* const cnt_n = &s_cnt[0][threadIdx.x];
    int* const cnt_lo = &s_cnt[1][threadIdx.x];
    int* const cnt_hi = &s_cnt[2][threadIdx.x];
    int* const cnt_strict = &s_cnt[3][threadIdx.x];
    *cnt_n = *cnt_lo = *cnt_hi = *cnt_strict = 0;
    s_rmax[threadIdx.x] = -CUDART_INF;
    const SurfK& SL = P.s[P.nsurf - 1];          // the image plane
    const bool refr_last = (SL.kcode & SURF_REFR) != 0;
    const bool collimated = (fld.mode == 0);
    double K0[3] = {0.0, 0.0, 0.0};
    if (ARITH == ORT_ARITH_FAST && collimated) {
        const double inv = P.n0 * fast_rsqrt(fma(fld.v, fld.v, fma(fld.u, fld.u, 1.0)));
        K0[0] = fld.v * inv; K0[1] = fld.u * inv; K0[2] = inv;
    }
    const unsigned nxu = (unsigned)A.nx;

    for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        double y0[RPT], x0[RPT], u[RPT], v[RPT];
        unsigned idx[RPT];
        bool valid[RPT];
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            const unsigned i0 = (tile * RPT + j) * ORT_TILE + threadIdx.x;
            valid[j] = i0 < NN;
            idx[j] = min(i0, NN - 1);            // padded lanes trace the last ray: the warp stays convergent
            const unsigned iy = idx[j] / nxu, ix = idx[j] - iy * nxu;      // a division per ray instead of 2 RPT registers
            y0[j] = __ldg(A.ys + (ysoff + iy)); x0[j] = __ldg(A.xs + ix);
            u[j] = 0.0; v[j] = 0.0;
        }
        if (!collimated || ARITH != ORT_ARITH_FAST) {
#pragma unroll
            for (int j = 0; j < RPT; j++) field_slopes(fld, y0[j], x0[j], u[j], v[j]);
        }
        FocusRay q[RPT];
        double xs[RPT], ys[RPT];                // stop position of STRICT and re-traced rays (FAST: s_xy)
        unsigned flg[RPT];
        bool sv[RPT];
        if (ARITH == ORT_ARITH_FAST) {
            RaysF<RPT> r;
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                if (collimated) {
                    r.x[j] = x0[j]; r.y[j] = y0[j]; r.z[j] = 0.0;
                    r.Kx[j] = K0[0]; r.Ky[j] = K0[1]; r.Kz[j] = K0[2];
                    r.amb[j] = 0; r.opl[j] = 0.0; r.vig[j] = 0;
                } else fast_init(r, j, P.n0, y0[j], x0[j], u[j], v[j]);
            }
            const int ns = P.nsurf - 1;
            int i = 0;
            for (; i < A.stop; i++) fast_step<RPT, false, MIRROR, SIMPLE, 0>(P.s[i], r);
#pragma unroll
            for (int j = 0; j < RPT; j++) s_xy[j][threadIdx.x] = make_double2(r.x[j], r.y[j]);
            for (; i < ns; i++) fast_step<RPT, false, MIRROR, SIMPLE, 0>(P.s[i], r);
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                int amb = r.amb[j];
                if (refr_last) {                 // fast_step's refracting-plane decision and k_grid's test of the final Kz
                    const double Dp = fma(r.Kz[j], r.Kz[j], SL.dn2);
                    amb |= hi32(Dp) - SL.tir_thr;
                    amb |= nonfinite_bit(MIRROR ? sign_of_n2(fast_sqrt(Dp), SL.n2mask) : fast_sqrt(Dp));
                }
                q[j].a0 = r.x[j]; q[j].a1 = r.y[j]; q[j].a2 = r.z[j]; q[j].a3 = r.Kx[j]; q[j].a4 = r.Ky[j];
                q[j].a5 = fast_div_rcp(r.Kz[j]);
                double xa, ya, xb, yb;
                focus_pos_fast(q[j], F.t_lo, xa, ya);
                focus_pos_fast(q[j], F.t_hi, xb, yb);
                amb |= nonfinite_bit(xa) | nonfinite_bit(ya) | nonfinite_bit(xb) | nonfinite_bit(yb);
                const double2 st = s_xy[j][threadIdx.x];
                const double r2 = fma(st.x, st.x, st.y * st.y);                  // grid_epilogue's r^2 and stop guard band
                amb |= tiny_vs_bit(r2 - A.a_stop2, A.a_stop2);
                sv[j] = amb < 0;
                flg[j] = 0u;
            }
        } else {
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                int bad = 0;
                FocusS o = focus_strict_impl<ORT_STRICT_XF>(P, A.stop, y0[j], x0[j], u[j], v[j], &bad);
                if (ORT_STRICT_XF && bad) o = focus_strict_cold(P, A.stop, y0[j], x0[j], u[j], v[j]);
                q[j] = o.q; xs[j] = o.xs; ys[j] = o.ys; flg[j] = o.flags; sv[j] = true;
            }
        }
        int kept[RPT];
        int nk = 0, nclip = 0;
        double rm = -CUDART_INF;
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            double ri = 0.0, r2 = 0.0;
            bool clip;
            if (ARITH == ORT_ARITH_FAST && !sv[j]) {
                const double2 st = s_xy[j][threadIdx.x];
                xs[j] = st.x; ys[j] = st.y;
                r2 = fma(st.x, st.x, st.y * st.y);
                clip = r2 > A.a_stop2;
                if (A.r) ri = (r2 > 0.0) ? fast_sqrt(r2) : r2;
            } else {
                if (ARITH == ORT_ARITH_FAST) {       // rare in FAST mode: the ray's inputs once more, strict trace
                    const unsigned iy = idx[j] / nxu, ix = idx[j] - iy * nxu;
                    const double yy = __ldg(ysf + iy), xx = __ldg(A.xs + ix);
                    double uu, vv; field_slopes(fld, yy, xx, uu, vv);
                    const FocusS o = focus_strict_cold(P, A.stop, yy, xx, uu, vv);
                    q[j] = o.q; xs[j] = o.xs; ys[j] = o.ys; flg[j] = o.flags;
                }
                ri = jl_hypot(xs[j], ys[j]);
                clip = ri > A.a_stop;
                r2 = ri * ri;
            }
            bool nan_any = false;
            if (sv[j]) {                             // NaN at any focus drops the ray for all of them
                bool fin_all = true;                 // x^2 + y^2 on the plane finite at every focus (FOCUS_TIR_LAST)
                for (int m = 0; m < M; m++) {
                    double xf, yf; focus_pos_strict(q[j], F.foci[m], xf, yf);
                    nan_any = nan_any || is_nan_bits(xf) || is_nan_bits(yf);
                    fin_all = fin_all && isfinite(SA(SM(xf, xf), SM(yf, yf)));
                }
                if (flg[j] & FOCUS_TIR_LAST) flg[j] = (flg[j] & ~FOCUS_TIR_LAST) | (fin_all ? ORT_FLAG_TIR : 0u);
                if (valid[j]) {
                    *cnt_strict += 1;
                    *cnt_lo += (flg[j] & ORT_FLAG_MISS ? 1 : 0) + (flg[j] & ORT_FLAG_TIR ? 0x10000 : 0);
                    *cnt_hi += (flg[j] & ORT_FLAG_DOMAIN ? 1 : 0);
                }
            }
            const bool drop = clip || nan_any;
            kept[j] = valid[j] && !drop;
            const double rv = (ARITH == ORT_ARITH_STRICT) ? ri : r2;
            if (valid[j]) {
                const size_t o = fbase + idx[j];
                if (A.r) A.r[o] = ri;
                if (A.theta) A.theta[o] = atan2(ys[j], xs[j]);
                if (A.mask) A.mask[o] = (uint8_t)kept[j];
                if (A.flags) A.flags[o] = (uint8_t)(flg[j] | (clip ? ORT_FLAG_CLIP : 0u));
                nclip += clip ? 1 : 0;
            }
            if (kept[j]) { if (rv > rm) rm = rv; nk++; }      // kept rays: never NaN
        }
        *cnt_n += nk;
        *cnt_hi += nclip << 16;
        if (rm > s_rmax[threadIdx.x]) s_rmax[threadIdx.x] = rm;
        int any_kept = 0;
#pragma unroll
        for (int j = 0; j < RPT; j++) any_kept |= kept[j];
        const bool warp_kept = __any_sync(0xffffffffu, any_kept);       // uniform per warp: no reduction for an empty warp
        const bool want_e = A.ex != nullptr;
        if (warp_kept || want_e) {
            for (int m = 0; m < M; m++) {
                const double t = F.foci[m];
                const double cxm = s_c[m][0], cym = s_c[m][1];
                double sx = 0.0, sxx = 0.0, sy = 0.0, syy = 0.0;
#pragma unroll
                for (int j = 0; j < RPT; j++) {
                    double xf, yf;
                    if (ARITH == ORT_ARITH_FAST && !sv[j]) focus_pos_fast(q[j], t, xf, yf);
                    else focus_pos_strict(q[j], t, xf, yf);
                    const double ex = xf;
                    const double ey = SS(yf, fld.h_prime);
                    if (want_e && valid[j]) {
                        const size_t o = ((size_t)f * M + m) * NN + idx[j];
                        A.ex[o] = ex; A.ey[o] = ey;
                    }
                    if (kept[j]) {
                        const double dx = ex - cxm, dy = ey - cym;
                        sx += dx; sxx = fma(dx, dx, sxx);
                        sy += dy; syy = fma(dy, dy, syy);
                    }
                }
                if (warp_kept) {
#pragma unroll
                    for (int d = 16; d >= 1; d >>= 1) {
                        sx += __shfl_down_sync(0xffffffffu, sx, d);
                        sxx += __shfl_down_sync(0xffffffffu, sxx, d);
                        sy += __shfl_down_sync(0xffffffffu, sy, d);
                        syy += __shfl_down_sync(0xffffffffu, syy, d);
                    }
                    if (lane == 0) {
                        s_acc[warp][m][0] += sx; s_acc[warp][m][1] += sxx;
                        s_acc[warp][m][2] += sy; s_acc[warp][m][3] += syy;
                    }
                }
            }
        }
        if (A.tile_counts) {                    // ordered compaction: kept rays per 256-ray sub-tile
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                const int c = __syncthreads_count(kept[j]);
                const unsigned sub = tile * RPT + j;
                if (threadIdx.x == 0 && sub < nsub) A.tile_counts[(size_t)f * nsub + sub] = c;
            }
        }
    }
    RawPart p;
    const int nflag_lo = *cnt_lo, nflag_hi = *cnt_hi;
    p.n = *cnt_n; p.s1x = p.s2x = p.s1y = p.s2y = 0.0; p.rmax = s_rmax[threadIdx.x];
    p.cx = p.cy = p.co = 0.0; p.s1o = p.s2o = 0.0; p.nvig = 0; p.nstrict = *cnt_strict;
    p.nmiss = nflag_lo & 0xFFFF; p.ntir = nflag_lo >> 16; p.ndom = nflag_hi & 0xFFFF; p.nclip = nflag_hi >> 16;
    raw_block_reduce<NWARPS>(p, s_part);         // its __syncthreads also orders the last s_acc updates
    if (threadIdx.x == 0) {
        if (ARITH != ORT_ARITH_STRICT) p.rmax = sqrt(p.rmax);
        s_p0 = p;
    }
    __syncthreads();
    for (int m = threadIdx.x; m < M; m += ORT_TILE) {
        RawPart q = s_p0;
        for (int w = 0; w < NWARPS; w++) {
            q.s1x += s_acc[w][m][0]; q.s2x += s_acc[w][m][1];
            q.s1y += s_acc[w][m][2]; q.s2y += s_acc[w][m][3];
        }
        q.cx = s_c[m][0]; q.cy = s_c[m][1];
        A.partials[((size_t)f * M + m) * gridDim.x + blockIdx.x] = q;
    }
}

// compaction of a focus sweep: one CTA per (tile, field); the foci of a field share its mask and tile offsets.
// C.src / C.dst [0], [1] are ex, ey ([n_fields][n_foci][NN]); [2], [3] are r, theta ([n_fields][NN]).
__global__ void __launch_bounds__(ORT_TILE) k_compact_focus(CompactArgs C, int n_foci)
{
    const unsigned tile = blockIdx.x, f = blockIdx.y;
    const unsigned ntiles = (C.NN + ORT_TILE - 1) / ORT_TILE;
    const unsigned i = tile * ORT_TILE + threadIdx.x;
    const size_t fbase = (size_t)f * C.NN;
    const int m = (i < C.NN) ? C.mask[fbase + i] : 0;
    const int off = compact_offset(C, tile, f, ntiles, threadIdx.x, m);
    if (m) {
        for (int a = 2; a < 4; a++)
            if (C.src[a]) C.dst[a][fbase + off] = C.src[a][fbase + i];
        for (int j = 0; j < n_foci; j++) {
            const size_t b = ((size_t)f * n_foci + j) * C.NN;
            for (int a = 0; a < 2; a++)
                if (C.src[a]) C.dst[a][b + off] = C.src[a][b + i];
        }
    }
}

// ------------------------------------------------------------------------------------------
// arbitrary rays, all surfaces recorded
// ------------------------------------------------------------------------------------------
template <int ARITH, bool EXT>
__global__ void __launch_bounds__(256)
k_rays(const __grid_constant__ Presc P, RaysArgs A)
{
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= A.N) return;
    const double y0 = A.y0[i], x0 = A.x0[i], u0 = A.u0[i], v0 = A.v0[i];
    const int nsurf = P.nsurf;
    const bool vignette = EXT && P.has_apertures;
    bool strict = (ARITH == ORT_ARITH_STRICT);
    if (!strict) {
        RaysF<1> r;
        fast_init(r, 0, P.n0, y0, x0, u0, v0);
        for (int s = 0; s < nsurf; s++) {
            fast_step<1, EXT, true, 0, EXT ? 1 : 0>(P.s[s], r, vignette, (EXT && P.poly) ? P.poly + (size_t)s * P.npoly : nullptr, P.npoly, nsurf * P.npoly);
            if (A.xv) A.xv[(size_t)s * A.N + i] = r.x[0];
            if (A.yv) A.yv[(size_t)s * A.N + i] = r.y[0];
        }
        const int amb = r.amb[0] | nonfinite_bit(r.x[0]) | nonfinite_bit(r.y[0]) | nonfinite_bit(r.Kz[0]);
        if (amb >= 0) {
            if (A.kout) {   // K = n k -> direction cosines; the reference's k is a LINE direction with k3 > 0
                const double inv = 1.0 / sqrt(fma(r.Kx[0], r.Kx[0], fma(r.Ky[0], r.Ky[0], r.Kz[0] * r.Kz[0])));
                const double sg = (r.Kz[0] < 0.0) ? -inv : inv;
                A.kout[i] = r.Kx[0] * sg; A.kout[A.N + i] = r.Ky[0] * sg; A.kout[2 * A.N + i] = r.Kz[0] * sg;
            }
            if (A.flags) A.flags[i] = (EXT && r.vig[0]) ? (uint8_t)ORT_FLAG_VIGN : (uint8_t)0;
            if (EXT && A.opl) A.opl[i] = r.opl[0];
        } else strict = true;
    }
    if (strict) {
        RayS r;
        strict_init(r, y0, x0, u0, v0);
        for (int s = 0; s < nsurf; s++) {
            strict_step<EXT, EXT>(P.s[s], r, vignette, (EXT && P.poly) ? P.poly + (size_t)s * P.npoly : nullptr, P.npoly);
            if (A.xv) A.xv[(size_t)s * A.N + i] = r.x;
            if (A.yv) A.yv[(size_t)s * A.N + i] = r.y;
        }
        if (A.kout) { A.kout[i] = r.k1; A.kout[A.N + i] = r.k2; A.kout[2 * A.N + i] = r.k3; }
        if (A.flags) A.flags[i] = (uint8_t)r.flags;
        if (EXT && A.opl) A.opl[i] = r.opl;
    }
}

// per-thread running moments about the first kept sample + Chan merge (candidate kernel: every
// CTA owns one prescription, so there is no common shift to share across CTAs)
struct Acc {
    int n;
    double cx, cy, s1x, s2x, s1y, s2y, rmax;
};
__device__ __forceinline__ void acc_zero(Acc& a)
{
    a.n = 0; a.cx = a.cy = a.s1x = a.s2x = a.s1y = a.s2y = 0.0; a.rmax = -CUDART_INF;
}
__device__ __forceinline__ void acc_add(Acc& a, double ex, double ey, double rr)
{
    if (a.n == 0) { a.cx = ex; a.cy = ey; }
    double dx = ex - a.cx, dy = ey - a.cy;
    a.s1x += dx; a.s2x = fma(dx, dx, a.s2x);
    a.s1y += dy; a.s2y = fma(dy, dy, a.s2y);
    a.rmax = fmax(a.rmax, rr);
    a.n++;
}
__device__ __forceinline__ Part acc_to_part(const Acc& a, bool rmax_is_squared)
{
    Part p; part_zero(p);
    if (a.n > 0) {
        double n = (double)a.n;
        p.n = a.n;
        p.mx = a.cx + a.s1x / n;
        p.my = a.cy + a.s1y / n;
        p.m2x = fmax(a.s2x - a.s1x * a.s1x / n, 0.0);
        p.m2y = fmax(a.s2y - a.s1y * a.s1y / n, 0.0);
        p.rmax = rmax_is_squared ? sqrt(a.rmax) : a.rmax;
    }
    return p;
}

// ------------------------------------------------------------------------------------------
// K5: candidate prescriptions, one CTA each, prescription staged in shared memory
// ------------------------------------------------------------------------------------------

// AIMED: every candidate carries its own prelude record (k_aim_candidates): stop, stop radius, field slope,
// image height, focus (the image plane [Inf 0 1] is appended here, t[end-1] = focus, src/PupilSampling.jl:111-114)
// and its own aimed pupil grid ys = range(y1, y2, ny), xs = range(0, y_EP, nx) (:121-122).
template <int ARITH, bool AIMED>
__global__ void __launch_bounds__(ORT_TILE, 3)
k_candidates(CandArgs A)
{
    __shared__ SurfK s_surf[ORT_MAX_ROWS];
    __shared__ Part s_part[ORT_TILE / 32];
    // FAST sweeps come with the classified lists of k_cand_classify: this kernel then takes the GENERAL candidates
    // (mirrors, conics, weak or dummy spheres), one per CTA, grid-strided
    const int nlist = A.lists ? A.lists[2] : 0;
    for (long long li = blockIdx.x; li < (A.lists ? (long long)nlist : A.C); li += gridDim.x) {
    if (li != (long long)blockIdx.x) __syncthreads();           // the previous candidate's shared state is still being read
    const long long c = A.lists ? (long long)A.lists[3 + 2 * A.C + li] : li;
    const int rows = A.rows, nsurf = AIMED ? rows : rows - 1;
    const double* Rc = A.RtnK + (size_t)c * 4 * rows;
    const double* rec = AIMED ? A.aim + (size_t)c * ORT_AIM_NOUT : nullptr;
    __shared__ int s_mirror, s_general;
    if (threadIdx.x == ORT_TILE - 2) { s_mirror = 0; s_general = 0; }
    __syncthreads();
    if (threadIdx.x < rows - 1) {
        const int i = threadIdx.x;
        derive_surface(s_surf[i], Rc[i + 1], Rc[3 * rows + i + 1], Rc[rows + i], Rc[2 * rows + i],
                       Rc[2 * rows + i + 1]);
        if (!(Rc[2 * rows + i] > 0.0) || !(Rc[2 * rows + i + 1] > 0.0)) atomicOr(&s_mirror, 1);   // a reflecting candidate
        if (ARITH == ORT_ARITH_FAST && !simple_surface(s_surf[i], gap_scale(Rc + rows, rows))) atomicOr(&s_general, 1);
    } else if (AIMED && threadIdx.x == rows - 1) {
        derive_surface(s_surf[rows - 1], CUDART_INF, 0.0, rec[5], Rc[3 * rows - 1], 1.0);
        if (!simple_surface(s_surf[rows - 1], 0.0)) atomicOr(&s_general, 1);
    }
    __syncthreads();
    // per-candidate scalars live in shared memory (the shared-grid variant reads them from the constant bank):
    // re-read by LDS broadcast where used, so they cost no registers across the surface loop
    __shared__ double s_par[10];
    __shared__ int s_stop;
    if (threadIdx.x == ORT_TILE - 1) {
        if (AIMED) {
            const int st = (int)rec[6];
            const bool good = rec[11] == 0.0 && st >= 1 && st <= rows - 1;     // NaN record / failed prelude -> NaN result
            s_stop = good ? st : 0;
            s_par[0] = rec[0]; s_par[1] = rec[1]; s_par[2] = SD(SS(rec[1], rec[0]), (double)(A.ny - 1));
            s_par[3] = rec[2]; s_par[4] = SD(rec[2], (double)(A.nx - 1));
            s_par[5] = rec[7]; s_par[6] = rec[7] * rec[7]; s_par[7] = rec[3]; s_par[8] = rec[4];
        } else {
            s_stop = A.stop;
            s_par[5] = A.a_stop; s_par[6] = A.a_stop2; s_par[7] = A.u; s_par[8] = A.h_prime;
        }
    }
    __syncthreads();
    const volatile double* par = s_par;
    const bool mirror = s_mirror != 0;
    const int stop = s_stop;
    const bool ok = stop > 0;
#define CAND_PAR(i, shared_grid_value) (AIMED ? par[i] : (shared_grid_value))
    Acc acc; acc_zero(acc);
    const unsigned NN = (unsigned)A.ny * (unsigned)A.nx;
    constexpr int RPT = (ARITH == ORT_ARITH_FAST) ? 2 : 1;      // 2 rays per thread share the LDS of the prescription
    const double n0 = Rc[2 * rows];
    double K0[3] = {0.0, 0.0, 0.0};                             // collimated field: K = n0 normalize([v, u, 1]) once
    if (ARITH == ORT_ARITH_FAST) {
        const double fu = CAND_PAR(7, A.u);
        const double inv = n0 * fast_rsqrt(fma(A.v, A.v, fma(fu, fu, 1.0)));
        K0[0] = A.v * inv; K0[1] = fu * inv; K0[2] = inv;
    }
    // The two aimed edge rays (first / last grid row at x = 0) cross the stop exactly at its rim by construction
    // (src/PupilSampling.jl:67-83): they always land in the guard band of the clip test.  Lanes 0 and 1 of warp 0 take
    // them through the strict trace side by side up front; the fast loop skips them.
    const unsigned edge_b = (unsigned)(A.ny - 1) * (unsigned)A.nx;
    constexpr bool EDGE_FIRST = AIMED && ARITH == ORT_ARITH_FAST;
    if (EDGE_FIRST && ok && threadIdx.x < 2) {
        if (rec[14] == 1.0) {           // traced by k_aim_edges, one thread per edge ray across the whole population
            const double* e = rec + 16 + 4 * threadIdx.x;
            if (e[0] == 1.0) acc_add(acc, e[1], e[2], e[3]);
        } else {                        // hand-made record without edge data
            const double ye = threadIdx.x ? par[1] : par[0];
            const Hit he = trace_strict_cold<false>(s_surf, nsurf, stop, ye, 0.0, par[7], A.v);
            const double ri = jl_hypot(he.xs, he.ys);
            if (!(ri > par[5] || is_nan_bits(he.xf) || is_nan_bits(he.yf))) acc_add(acc, he.xf, he.yf - par[8], ri * ri);
        }
    }
    for (unsigned i0 = threadIdx.x; ok && i0 < NN; i0 += ORT_TILE * RPT) {
        double y0[RPT], x0[RPT], uu[RPT], vv[RPT];
        bool valid[RPT];
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            const unsigned i = i0 + j * ORT_TILE;
            valid[j] = i < NN && !(EDGE_FIRST && (i == 0 || i == edge_b));
            const unsigned ic = i < NN ? i : NN - 1;
            const unsigned iy = ic / (unsigned)A.nx, ix = ic - iy * (unsigned)A.nx;
            if (AIMED) {        // range(a, b, n)[i] = a + i * step, last point exactly b
                y0[j] = (iy == (unsigned)A.ny - 1) ? par[1] : SA(par[0], SM((double)iy, par[2]));
                x0[j] = (ix == (unsigned)A.nx - 1) ? par[3] : SM((double)ix, par[4]);
            } else { y0[j] = __ldg(A.ys + iy); x0[j] = __ldg(A.xs + ix); }
            uu[j] = 0.0; vv[j] = A.v;                           // the fast path takes the direction from K0
        }
        Hit h[RPT]; int amb[RPT];
        if (ARITH == ORT_ARITH_FAST) {      // CTA-uniform choice between the general and the no-mirror fast path
            if (mirror) trace_fast<RPT, false, SurfK*, true>(s_surf, nsurf, stop, n0, y0, x0, uu, vv, h, amb, nullptr, 1.0, false, K0);
            else trace_fast<RPT, false, SurfK*, false>(s_surf, nsurf, stop, n0, y0, x0, uu, vv, h, amb, nullptr, 1.0, false, K0);
        }
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            double ri = 0.0, r2 = 0.0; bool clip = false;
            if (ARITH == ORT_ARITH_FAST) {
                const double a_stop2 = CAND_PAR(6, A.a_stop2);
                r2 = fma(h[j].xs, h[j].xs, h[j].ys * h[j].ys);
                amb[j] |= tiny_vs_bit(r2 - a_stop2, a_stop2);
                clip = r2 > a_stop2;
            }
            if (ARITH == ORT_ARITH_STRICT || (amb[j] < 0 && valid[j])) {
                const double fu = CAND_PAR(7, A.u);
                h[j] = (ARITH == ORT_ARITH_STRICT) ? trace_strict_xf<false>(s_surf, nsurf, stop, y0[j], x0[j], fu, A.v)
                                                   : trace_strict_cold<false>(s_surf, nsurf, stop, y0[j], x0[j], fu, A.v);
                ri = jl_hypot(h[j].xs, h[j].ys);
                clip = ri > CAND_PAR(5, A.a_stop);
                r2 = ri * ri;
            }
            const bool drop = clip || is_nan_bits(h[j].xf) || is_nan_bits(h[j].yf);
            if (valid[j] && !drop) acc_add(acc, h[j].xf, h[j].yf - CAND_PAR(8, A.h_prime), r2);
        }
    }
#undef CAND_PAR
    Part p = acc_to_part(acc, true);
    part_block_reduce<ORT_TILE / 32>(p, s_part);
    if (threadIdx.x == 0) {
        double* o = A.out + 4 * c;
        o[0] = ok ? (double)p.n : CUDART_NAN;
        if (ok && p.n > 0) { o[1] = p.mx; o[2] = p.my; o[3] = sqrt((p.m2x + p.m2y) / (double)p.n); }
        else { o[1] = o[2] = o[3] = CUDART_NAN; }
    }
    }
}

// FAST sweeps first sort the population (one thread per candidate): lists[0] / lists[1] / lists[2] = number of SIMPLE /
// SIMPLE-CONIC / GENERAL candidates, lists[3 ..) / lists[3 + C ..) / lists[3 + 2 C ..) their indices.  SIMPLE-CONIC =
// refracting conics / spheres and planes only, every index positive (the class of Presc::simple == 2): the same kernel
// with the conic body.  SIMPLE = refracting spheres (|R| <= 64 L) and planes only,
// every index positive (simple_surface): those go to k_candidates_simple.  The order inside a list is whatever the
// atomics produce; every candidate's result is computed alone and written to its own slot, so results do not depend on it.
__global__ void __launch_bounds__(128) k_cand_classify(int rows, long long C, const double* RtnK, int aimed, int* lists)
{
    const long long c = (long long)blockIdx.x * 128 + threadIdx.x;
    if (c >= C) return;
    const double* Rc = RtnK + (size_t)c * 4 * rows;
    const double L = gap_scale(Rc + rows, rows);
    bool simple = true, conic = true;
    for (int i = 0; i + 1 < rows; i++) {
        SurfK S;
        const double Ri = Rc[i + 1], Ki = Rc[3 * rows + i + 1], ti = Rc[rows + i], n1 = Rc[2 * rows + i], n2 = Rc[2 * rows + i + 1];
        derive_surface(S, Ri, Ki, ti, n1, n2);
        const bool pos = n1 > 0.0 && n2 > 0.0;
        if (!pos || !simple_surface(S, L)) simple = false;
        // the conic body needs finite operands and a refracting surface wherever the surface is curved (ort_set_layout)
        const bool plane = (S.kcode & SURF_KIND_MASK) == SURF_PLANE;
        const bool finite_ops = !(Ri == 0.0) && Ri == Ri && isfinite(Ki) && isfinite(ti) && isfinite(n1) && isfinite(n2);
        if (!pos || !finite_ops || (!plane && !(S.kcode & SURF_REFR))) conic = false;
    }
    if (aimed && !(Rc[3 * rows - 1] > 0.0)) simple = conic = false;     // the appended image plane refracts into n = 1
    const int cls = simple ? 0 : (conic ? 1 : 2);
    const int slot = atomicAdd(&lists[cls], 1);
    lists[3 + cls * C + slot] = (int)c;
}

// K5 for SIMPLE candidates: the three-body surface loop (fast_step<.., SIMPLE>), CS_RPT rays per thread, its own launch
// bounds (no spills), plain shifted sums instead of per-thread Chan records.  One candidate per CTA pass, grid-strided
// over the list of k_cand_classify.  Measured on 65 536 triplets x 4096 rays (tools/bench_cand.py): 64 threads x 2 rays x
// 12 CTAs/SM 5.38 ms, 128 x 2 x 6 5.42, 128 x 2 x 5 (no spills) 5.53, 64 x 3 x 8 5.54, 128 x 3 x 4 5.60 (4096 rays are
// 10.67 passes of 384: 3 % padding), 256 x 2 x 3 5.57, 128 x 4 x 3 5.66; the mixed kernel of round 1: 5.95.
#ifndef CS_THREADS
#define CS_THREADS 64
#endif
#ifndef CS_RPT
#define CS_RPT 2
#endif
#ifndef CS_MINB
#define CS_MINB 12
#endif
template <bool AIMED, int SIMPLE = 1>
__global__ void __launch_bounds__(CS_THREADS, CS_MINB)
k_candidates_simple(CandArgs A)
{
    __shared__ SurfK s_surf[ORT_MAX_ROWS];
    __shared__ double s_par[12];
    __shared__ int s_stop;
    __shared__ double s_red[CS_THREADS / 32][6];
    __shared__ int s_redn[CS_THREADS / 32];
    const int rows = A.rows, nsurf = AIMED ? rows : rows - 1;
    const int nlist = A.lists[SIMPLE - 1];
    const unsigned NN = (unsigned)A.ny * (unsigned)A.nx, nxu = (unsigned)A.nx;
    const unsigned step = CS_THREADS * CS_RPT, dq = step / nxu, dr = step - dq * nxu;
    for (int li = blockIdx.x; li < nlist; li += gridDim.x) {
        if (li != (int)blockIdx.x) __syncthreads();
        const long long c = A.lists[3 + (SIMPLE - 1) * A.C + li];
        const double* Rc = A.RtnK + (size_t)c * 4 * rows;
        const double* rec = AIMED ? A.aim + (size_t)c * ORT_AIM_NOUT : nullptr;
        if (threadIdx.x < rows - 1) {
            const int i = threadIdx.x;
            derive_surface(s_surf[i], Rc[i + 1], Rc[3 * rows + i + 1], Rc[rows + i], Rc[2 * rows + i], Rc[2 * rows + i + 1]);
            simple_surface(s_surf[i], gap_scale(Rc + rows, rows));
        } else if (AIMED && threadIdx.x == rows - 1) {
            derive_surface(s_surf[rows - 1], CUDART_INF, 0.0, rec[5], Rc[3 * rows - 1], 1.0);
            simple_surface(s_surf[rows - 1], 0.0);
        } else if (threadIdx.x == CS_THREADS - 1) {
            if (AIMED) {
                const int st = (int)rec[6];
                const bool good = rec[11] == 0.0 && st >= 1 && st <= rows - 1;     // NaN record / failed prelude -> NaN result
                s_stop = good ? st : 0;
                s_par[0] = rec[0]; s_par[1] = rec[1]; s_par[2] = SD(SS(rec[1], rec[0]), (double)(A.ny - 1));
                s_par[3] = rec[2]; s_par[4] = SD(rec[2], (double)(A.nx - 1));
                s_par[5] = rec[7]; s_par[6] = rec[7] * rec[7]; s_par[7] = rec[3]; s_par[8] = rec[4];
                // common shift of the moments: the two rim rays straddle the spot
                const bool have = rec[14] == 1.0 && rec[16] == 1.0 && rec[20] == 1.0;
                s_par[9] = have ? 0.5 * (rec[18] + rec[22]) : 0.0;
            } else {
                s_stop = A.stop;
                s_par[5] = A.a_stop; s_par[6] = A.a_stop2; s_par[7] = A.u; s_par[8] = A.h_prime; s_par[9] = 0.0;
            }
        }
        __syncthreads();
        const volatile double* par = s_par;
        const int stop = s_stop;
        const bool ok = stop > 0;
        const double n0 = Rc[2 * rows];
        const double cy = par[9];
        double K0[3];
        {
            const double fu = par[7];
            const double inv = n0 * fast_rsqrt(fma(A.v, A.v, fma(fu, fu, 1.0)));
            K0[0] = A.v * inv; K0[1] = fu * inv; K0[2] = inv;
        }
        int n = 0;
        double s1x = 0.0, s2x = 0.0, s1y = 0.0, s2y = 0.0, rmax = -CUDART_INF;
        const unsigned edge_b = (unsigned)(A.ny - 1) * nxu;
        if (AIMED && ok && threadIdx.x < 2) {           // the two rim rays (first / last row at x = 0), see k_candidates
            double ex, ey, rr; bool keep;
            if (rec[14] == 1.0) { const double* e = rec + 16 + 4 * threadIdx.x; keep = e[0] == 1.0; ex = e[1]; ey = e[2]; rr = e[3]; }
            else {
                const Hit he = trace_strict_cold<false>(s_surf, nsurf, stop, threadIdx.x ? par[1] : par[0], 0.0, par[7], A.v);
                const double ri = jl_hypot(he.xs, he.ys);
                keep = !(ri > par[5] || is_nan_bits(he.xf) || is_nan_bits(he.yf)); ex = he.xf; ey = he.yf - par[8]; rr = ri * ri;
            }
            if (keep) { const double dy = ey - cy; s1x += ex; s2x = fma(ex, ex, s2x); s1y += dy; s2y = fma(dy, dy, s2y); rmax = fmax(rmax, rr); n++; }
        }
        unsigned iyj[CS_RPT], ixj[CS_RPT];
#pragma unroll
        for (int j = 0; j < CS_RPT; j++) { const unsigned i = threadIdx.x + j * CS_THREADS; iyj[j] = i / nxu; ixj[j] = i - iyj[j] * nxu; }
        // the candidate's grid parameters in registers for the whole sweep (an LDS in front of every trace otherwise)
        const double g_y1 = par[0], g_y2 = par[1], g_dy = par[2], g_xe = par[3], g_dx = par[4], a_stop2 = par[6], hpc = par[8] + cy;
        for (unsigned i0 = threadIdx.x; ok && i0 < NN; i0 += step) {
            double y0[CS_RPT], x0[CS_RPT], uu[CS_RPT], vv[CS_RPT];
            bool valid[CS_RPT];
#pragma unroll
            for (int j = 0; j < CS_RPT; j++) {
                const unsigned i = i0 + j * CS_THREADS;
                valid[j] = i < NN && !(AIMED && (i == 0 || i == edge_b));
                const unsigned iy = min(iyj[j], (unsigned)A.ny - 1), ix = ixj[j];       // idle lanes shadow a ray of the last row
                if (AIMED) {        // range(a, b, n)[i] = a + i * step, last point exactly b
                    y0[j] = (iy == (unsigned)A.ny - 1) ? g_y2 : SA(g_y1, SM((double)iy, g_dy));
                    x0[j] = (ix == nxu - 1) ? g_xe : SM((double)ix, g_dx);
                } else { y0[j] = __ldg(A.ys + iy); x0[j] = __ldg(A.xs + ix); }
                uu[j] = 0.0; vv[j] = A.v;                           // the fast path takes the direction from K0
                ixj[j] += dr; iyj[j] += dq;
                if (ixj[j] >= nxu) { ixj[j] -= nxu; iyj[j]++; }
            }
            Hit h[CS_RPT]; int amb[CS_RPT];
            trace_fast<CS_RPT, false, SurfK*, false, SIMPLE>(s_surf, nsurf, stop, n0, y0, x0, uu, vv, h, amb, nullptr, 1.0, false, K0);
#pragma unroll
            for (int j = 0; j < CS_RPT; j++) {
                double r2 = fma(h[j].xs, h[j].xs, h[j].ys * h[j].ys);
                amb[j] |= tiny_vs_bit(r2 - a_stop2, a_stop2);
                bool drop = r2 > a_stop2;
                if (amb[j] < 0 && valid[j]) {                       // guard band / miss / TIR: the reference arithmetic decides
                    h[j] = trace_strict_cold<false>(s_surf, nsurf, stop, y0[j], x0[j], par[7], A.v);
                    const double ri = jl_hypot(h[j].xs, h[j].ys);
                    drop = ri > par[5] || is_nan_bits(h[j].xf) || is_nan_bits(h[j].yf);
                    r2 = ri * ri;
                }
                if (valid[j] && !drop) {
                    const double ex = h[j].xf, dy = h[j].yf - hpc;      // (yf - h') - cy up to one rounding of the shift
                    s1x += ex; s2x = fma(ex, ex, s2x); s1y += dy; s2y = fma(dy, dy, s2y);
                    if (r2 > rmax) rmax = r2;
                    n++;
                }
            }
        }
        // deterministic CTA reduction: shuffle tree, then thread 0 folds the warp leaders in warp order
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            n += __shfl_down_sync(0xffffffffu, n, d);
            s1x += __shfl_down_sync(0xffffffffu, s1x, d); s2x += __shfl_down_sync(0xffffffffu, s2x, d);
            s1y += __shfl_down_sync(0xffffffffu, s1y, d); s2y += __shfl_down_sync(0xffffffffu, s2y, d);
            rmax = fmax(rmax, __shfl_down_sync(0xffffffffu, rmax, d));
        }
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) { s_redn[warp] = n; s_red[warp][0] = s1x; s_red[warp][1] = s2x; s_red[warp][2] = s1y; s_red[warp][3] = s2y; s_red[warp][4] = rmax; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < CS_THREADS / 32; w++) {
                n += s_redn[w]; s1x += s_red[w][0]; s2x += s_red[w][1]; s1y += s_red[w][2]; s2y += s_red[w][3];
            }
            double* o = A.out + 4 * c;
            o[0] = ok ? (double)n : CUDART_NAN;
            if (ok && n > 0) {
                const double dn = (double)n;
                const double m2 = fmax(s2x - s1x * s1x / dn, 0.0) + fmax(s2y - s1y * s1y / dn, 0.0);
                o[1] = s1x / dn; o[2] = cy + s1y / dn; o[3] = sqrt(m2 / dn);
            } else { o[1] = o[2] = o[3] = CUDART_NAN; }
        }
    }
}

// The two aimed edge rays of every candidate in the strict trace, 2 threads per candidate: results land in slots
// 14..23 of the prelude record so the FAST population sweep does not serialise a strict re-trace in every CTA.
struct CandSurfGen {
    const double* Rc; int rows; double focus;
    __device__ __forceinline__ SurfK operator[](int i) const
    {
        SurfK S;
        if (i < rows - 1) derive_surface(S, Rc[i + 1], Rc[3 * rows + i + 1], Rc[rows + i], Rc[2 * rows + i], Rc[2 * rows + i + 1]);
        else derive_surface(S, CUDART_INF, 0.0, focus, Rc[3 * rows - 1], 1.0);
        return S;
    }
};

__global__ void __launch_bounds__(128) k_aim_edges(int rows, long long C, const double* RtnK, double* aim, int shared)
{
    const long long t = (long long)blockIdx.x * 128 + threadIdx.x;
    const long long c = t >> 1;
    const int e = (int)(t & 1);
    if (c >= C) return;
    double* rec = aim + (size_t)c * ORT_AIM_NOUT;
    const int stop = (int)rec[6];
    const bool good = rec[11] == 0.0 && stop >= 1 && stop <= rows - 1;
    double* o = rec + 16 + 4 * e;
    if (!good) { if (e == 0) { rec[14] = 0.0; rec[15] = 0.0; } o[0] = o[1] = o[2] = o[3] = CUDART_NAN; return; }
    CandSurfGen gen; gen.Rc = RtnK + (shared ? 0 : (size_t)c * 4 * rows); gen.rows = rows; gen.focus = rec[5];
    const Hit h = trace_strict_xf<false>(gen, rows, stop, rec[e], 0.0, rec[3], 0.0);
    const double ri = jl_hypot(h.xs, h.ys);
    const bool drop = ri > rec[7] || is_nan_bits(h.xf) || is_nan_bits(h.yf);
    o[0] = drop ? 0.0 : 1.0; o[1] = h.xf; o[2] = h.yf - rec[4]; o[3] = ri * ri;
    if (e == 0) { rec[14] = 1.0; rec[15] = 0.0; }
}

cudaError_t launch_aim_edges(int rows, long long C, const double* RtnK, double* aim, int shared_prescription, cudaStream_t st)
{
    if (C == 0) return cudaSuccess;
    k_aim_edges<<<(unsigned)((2 * C + 127) / 128), 128, 0, st>>>(rows, C, RtnK, aim, shared_prescription);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// launch wrappers (called from ort_api.cu)
// ------------------------------------------------------------------------------------------
// kernel variant of a FAST sweep: 0 general, 1 EXT (OPD / apertures / polynomial terms), 2 SIMPLE, 3 SIMPLE x EXT,
// 4 SIMPLE-conic (Presc::simple == 2); STRICT has 0 and 1
int grid_variant(const Presc& P, int arith, int ext)
{
    const bool simple = arith == ORT_ARITH_FAST && P.simple == 1 && !P.has_mirror;
    if (ext || P.poly) return (simple && !P.poly) ? 3 : 1;
    if (arith == ORT_ARITH_FAST && P.simple == 2 && !P.has_mirror) return 4;
    return simple ? 2 : 0;
}

int grid_rays_per_thread(int arith, int variant)
{
    return arith == ORT_ARITH_FAST ? (variant == 2 ? ORT_SIMPLE_RPT : (variant == 3 ? ORT_SE_RPT : (variant == 4 ? ORT_SC_RPT : ORT_FAST_RPT))) : ORT_STRICT_RPT;
}

int grid_blocks_per_sm(int arith, int variant)
{
    int nb = 0;
    cudaError_t e;
    if (arith == ORT_ARITH_FAST && variant == 2)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_FAST, ORT_SIMPLE_RPT, 0, 1, false, true>, ORT_TILE, 0);
    else if (arith == ORT_ARITH_FAST && variant == 3)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_FAST, ORT_SE_RPT, 2, 0, false, true>, ORT_TILE, 0);
    else if (arith == ORT_ARITH_FAST && variant == 4)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_FAST, ORT_SC_RPT, 0, 1, false, 2>, ORT_TILE, 0);
    else if (arith == ORT_ARITH_FAST)
        e = variant ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 1>, ORT_TILE, 0)
                    : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0>, ORT_TILE, 0);
    else
        e = (variant & 1) ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_STRICT, ORT_STRICT_RPT, 1>, ORT_TILE, 0)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_grid<ORT_ARITH_STRICT, ORT_STRICT_RPT, 0>, ORT_TILE, 0);
    if (e != cudaSuccess || nb < 1) nb = 1;
    return nb;
}

cudaError_t launch_grid(const Presc& P, const GridArgs& A, int arith, dim3 grid, cudaStream_t st, const PolyK* Q)
{
    const bool ext = A.ext != 0 || P.poly != nullptr;          // polynomial terms live in the EXT instantiations
    if (arith == ORT_ARITH_FAST) {
        const bool others = A.r || A.theta || A.wx || A.wy || A.flags || A.opd;
        const bool lean = !ext && !others && A.ex && A.ey && A.mask;
        const bool stats_only = !ext && !others && !A.ex && !A.ey && !A.mask;
        const int variant = grid_variant(P, arith, ext);
        const bool simple = variant == 2;
        // the output set of an OPD sweep (ex, ey, opd, mask + statistics) has its own lean epilogue
        const bool lean_opd = (A.ext & ORT_EXT_OPD) && A.ex && A.ey && A.mask && A.opd && !(A.r || A.theta || A.wx || A.wy || A.flags);
        if (variant == 3 && !(A.ext & ORT_EXT_VIGNETTE) && lean_opd) k_grid<ORT_ARITH_FAST, ORT_SE_RPT, 2, 1, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (variant == 3 && !(A.ext & ORT_EXT_VIGNETTE)) k_grid<ORT_ARITH_FAST, ORT_SE_RPT, 2, 0, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (variant == 3 && lean_opd) k_grid<ORT_ARITH_FAST, ORT_SE_RPT, 1, 1, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (variant == 3) k_grid<ORT_ARITH_FAST, ORT_SE_RPT, 1, 0, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (variant == 4 && lean) k_grid<ORT_ARITH_FAST, ORT_SC_RPT, 0, 1, false, 2><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (variant == 4 && stats_only) k_grid<ORT_ARITH_FAST, ORT_SC_RPT, 0, 2, false, 2><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (variant == 4) k_grid<ORT_ARITH_FAST, ORT_SC_RPT, 0, 0, false, 2><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (simple && lean) k_grid<ORT_ARITH_FAST, ORT_SIMPLE_RPT, 0, 1, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (simple && stats_only) k_grid<ORT_ARITH_FAST, ORT_SIMPLE_RPT, 0, 2, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (simple) k_grid<ORT_ARITH_FAST, ORT_SIMPLE_RPT, 0, 0, false, true><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        // polynomial terms (no mirrors: ort_set_polynomials): spot + mask sweeps without the extension outputs have their own instantiation
        else if (P.poly && Q && !A.ext && !others && A.ex && A.ey && A.mask) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 1, false, 0, 2><<<grid, ORT_TILE, 0, st>>>(P, A, *Q);
        else if (P.poly && Q) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 1, 0, false, 0, 2><<<grid, ORT_TILE, 0, st>>>(P, A, *Q);
        else if (P.poly && !A.ext && !others && A.ex && A.ey && A.mask) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 1, false, 0, 1><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (P.poly) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 1, 0, false, 0, 1><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (ext && !P.has_mirror) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 1, 0, false><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (ext) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 1><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (lean && !P.has_mirror) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 1, false><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (stats_only && !P.has_mirror) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 2, false><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (!P.has_mirror) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 0, false><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (lean) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 1><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else if (stats_only) k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0, 2><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else k_grid<ORT_ARITH_FAST, ORT_FAST_RPT, 0><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
    } else {
        if (ext) k_grid<ORT_ARITH_STRICT, ORT_STRICT_RPT, 1><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
        else k_grid<ORT_ARITH_STRICT, ORT_STRICT_RPT, 0><<<grid, ORT_TILE, 0, st>>>(P, A, NoPolyK());
    }
    return cudaGetLastError();
}

cudaError_t launch_grid_finalize(const RawPart* partials, int nparts, int n_fields, ort_stats* stats,
                                 cudaStream_t st)
{
    k_grid_finalize<<<n_fields, 256, 0, st>>>(partials, nparts, stats);
    return cudaGetLastError();
}

size_t compact_tile_ints(unsigned NN)
{
    const size_t ntiles = (NN + ORT_TILE - 1) / ORT_TILE;
    return ntiles + ntiles / SCAN_CHUNK + 2;
}

// the two scan levels over the [n_fields][ntiles] tile counts; the chunk totals live right behind them
static cudaError_t launch_tile_scan(int* tile_counts, unsigned ntiles, int n_fields, cudaStream_t st)
{
    const unsigned nchunks = (ntiles + SCAN_CHUNK - 1) / SCAN_CHUNK;
    k_tile_scan<<<dim3(nchunks, n_fields), 256, 0, st>>>(tile_counts, tile_counts + (size_t)n_fields * ntiles, ntiles, nchunks);
    k_chunk_scan<<<n_fields, 256, 0, st>>>(tile_counts + (size_t)n_fields * ntiles, nchunks);
    return cudaGetLastError();
}

cudaError_t launch_compact(int* tile_counts, const CompactArgs& C, int n_fields, cudaStream_t st)
{
    const unsigned ntiles = (C.NN + ORT_TILE - 1) / ORT_TILE;
    cudaError_t e = launch_tile_scan(tile_counts, ntiles, n_fields, st);
    if (e != cudaSuccess) return e;
    k_compact<<<dim3(ntiles, n_fields), ORT_TILE, 0, st>>>(C);
    return cudaGetLastError();
}

// resident CTAs/SM of the k_focus instantiation of a k_grid variant (0 general, 2 SIMPLE, 4 SIMPLE-conic; FAST general
// with and without MIRROR share their bounds); sizes the grid in ort_api.cu like grid_blocks_per_sm does k_grid's
int focus_blocks_per_sm(int arith, int variant)
{
    int nb = 0;
    cudaError_t e;
    if (arith != ORT_ARITH_FAST) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_focus<ORT_ARITH_STRICT, ORT_STRICT_RPT, true, 0>, ORT_TILE, 0);
    else if (variant == 2) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_focus<ORT_ARITH_FAST, ORT_SIMPLE_RPT, false, 1>, ORT_TILE, 0);
    else if (variant == 4) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_focus<ORT_ARITH_FAST, ORT_SC_RPT, false, 2>, ORT_TILE, 0);
    else e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_focus<ORT_ARITH_FAST, ORT_FAST_RPT, true, 0>, ORT_TILE, 0);
    if (e != cudaSuccess || nb < 1) nb = 1;
    return nb;
}

// the k_focus instantiation of the k_grid variant this prescription runs (grid_variant without extensions)
cudaError_t launch_focus(const Presc& P, const FocusArgs& F, int arith, dim3 grid, cudaStream_t st)
{
    if (arith == ORT_ARITH_FAST) {
        const int variant = grid_variant(P, arith, 0);
        if (variant == 2) k_focus<ORT_ARITH_FAST, ORT_SIMPLE_RPT, false, 1><<<grid, ORT_TILE, 0, st>>>(P, F);
        else if (variant == 4) k_focus<ORT_ARITH_FAST, ORT_SC_RPT, false, 2><<<grid, ORT_TILE, 0, st>>>(P, F);
        else if (!P.has_mirror) k_focus<ORT_ARITH_FAST, ORT_FAST_RPT, false, 0><<<grid, ORT_TILE, 0, st>>>(P, F);
        else k_focus<ORT_ARITH_FAST, ORT_FAST_RPT, true, 0><<<grid, ORT_TILE, 0, st>>>(P, F);
    } else {
        k_focus<ORT_ARITH_STRICT, ORT_STRICT_RPT, true, 0><<<grid, ORT_TILE, 0, st>>>(P, F);
    }
    return cudaGetLastError();
}

cudaError_t launch_compact_focus(int* tile_counts, const CompactArgs& C, int n_fields, int n_foci, cudaStream_t st)
{
    const unsigned ntiles = (C.NN + ORT_TILE - 1) / ORT_TILE;
    cudaError_t e = launch_tile_scan(tile_counts, ntiles, n_fields, st);
    if (e != cudaSuccess) return e;
    k_compact_focus<<<dim3(ntiles, n_fields), ORT_TILE, 0, st>>>(C, n_foci);
    return cudaGetLastError();
}

cudaError_t launch_rays(const Presc& P, const RaysArgs& A, int arith, cudaStream_t st)
{
    const unsigned nb = (unsigned)((A.N + 255) / 256);
    if (nb == 0) return cudaSuccess;
    const bool ext = A.opl != nullptr || P.has_apertures || P.poly != nullptr;
    if (arith == ORT_ARITH_FAST) {
        if (ext) k_rays<ORT_ARITH_FAST, true><<<nb, 256, 0, st>>>(P, A);
        else k_rays<ORT_ARITH_FAST, false><<<nb, 256, 0, st>>>(P, A);
    } else {
        if (ext) k_rays<ORT_ARITH_STRICT, true><<<nb, 256, 0, st>>>(P, A);
        else k_rays<ORT_ARITH_STRICT, false><<<nb, 256, 0, st>>>(P, A);
    }
    return cudaGetLastError();
}

int candidates_blocks_per_sm(int simple)
{
    int nb = 0;
    cudaError_t e = simple ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_candidates_simple<true, 1>, CS_THREADS, 0)
                           : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_candidates<ORT_ARITH_FAST, true>, ORT_TILE, 0);
    if (e != cudaSuccess || nb < 1) nb = 1;
    return nb;
}

// FAST: classify, then the SIMPLE candidates through k_candidates_simple and the rest through k_candidates, both
// grid-strided over their list (an empty list costs one wave of CTAs that exit at once).  STRICT: one CTA per candidate.
cudaError_t launch_candidates(const CandArgs& A, int arith, cudaStream_t st, int sm_count)
{
    if (A.C == 0) return cudaSuccess;
    if (arith != ORT_ARITH_FAST || !A.lists) {
        CandArgs B = A; B.lists = nullptr;
        const unsigned nb = (unsigned)A.C;
        if (A.aim) {
            if (arith == ORT_ARITH_FAST) k_candidates<ORT_ARITH_FAST, true><<<nb, ORT_TILE, 0, st>>>(B);
            else k_candidates<ORT_ARITH_STRICT, true><<<nb, ORT_TILE, 0, st>>>(B);
        } else {
            if (arith == ORT_ARITH_FAST) k_candidates<ORT_ARITH_FAST, false><<<nb, ORT_TILE, 0, st>>>(B);
            else k_candidates<ORT_ARITH_STRICT, false><<<nb, ORT_TILE, 0, st>>>(B);
        }
        return cudaGetLastError();
    }
    cudaError_t e = cudaMemsetAsync(A.lists, 0, 3 * sizeof(int), st);
    if (e != cudaSuccess) return e;
    k_cand_classify<<<(unsigned)((A.C + 127) / 128), 128, 0, st>>>(A.rows, A.C, A.RtnK, A.aim != nullptr, A.lists);
    static const int bps_s = candidates_blocks_per_sm(1), bps_g = candidates_blocks_per_sm(0);
    const long long gs = (long long)sm_count * bps_s * 8, gg = (long long)sm_count * bps_g;
    const unsigned nbs = (unsigned)(A.C < gs ? A.C : gs), nbg = (unsigned)(A.C < gg ? A.C : gg);
    if (A.aim) {
        k_candidates_simple<true, 1><<<nbs, CS_THREADS, 0, st>>>(A);
        k_candidates_simple<true, 2><<<nbs, CS_THREADS, 0, st>>>(A);
        k_candidates<ORT_ARITH_FAST, true><<<nbg, ORT_TILE, 0, st>>>(A);
    } else {
        k_candidates_simple<false, 1><<<nbs, CS_THREADS, 0, st>>>(A);
        k_candidates_simple<false, 2><<<nbs, CS_THREADS, 0, st>>>(A);
        k_candidates<ORT_ARITH_FAST, false><<<nbg, ORT_TILE, 0, st>>>(A);
    }
    return cudaGetLastError();
}
