/*
 * ort_b200.h -- C ABI of libort_b200.so: the B200 (sm_100a) implementation of the data-parallel
 * hot path of Sagnac/OpticalRayTracing.jl.
 *
 * The reference is pure Julia and has NO FFI/plugin interface; its "boundary" is multiple
 * dispatch on exported generics.  Each entry point below replaces the body of one reference
 * method and is what a Julia `ccall` shim binds (julia/OpticalRayTracingB200.jl, INTEGRATION.md).
 * All citations are file:line relative to the reference repository root.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, Float64 everywhere (Julia Vector{Float64} memory).
 *   - Return 0 (ORT_OK) or a negative ORT_E* code; message via ort_last_error().  Nothing
 *     throws or longjmps across the ABI.  Per-ray geometric failures are DATA: NaN positions
 *     exactly where the reference yields NaN, plus ORT_FLAG_* bits.
 *   - Host-pointer entry points are synchronous (outputs valid on return).  *_dev entry points
 *     take DEVICE pointers and a cudaStream_t (as void*), enqueue only, and never synchronise.
 *   - The caller owns every array it passes; the library owns the context, its stream, scratch.
 *   - One ort_ctx per (process, GPU); a context is not re-entrant (one host thread at a time); distinct contexts are
 *     independent.  All entry points of one context share its grow-only device scratch: the library orders that use
 *     across streams itself (a call enqueued on a stream other than the previous call's first waits, on the device,
 *     for the previous call's work), so *_dev calls of one context on different streams are SAFE but do not overlap;
 *     use one context per stream for concurrent sweeps.  The first call at a larger problem size grows the scratch and
 *     synchronises the device once (cudaDeviceSynchronize + cudaMalloc); steady-state *_dev calls only enqueue.
 *   - Multi-GPU: one process per GPU (ort_comm_init_rank, e.g. under torchrun / MPI) or one process driving several
 *     contexts (ort_comm_init_all).  The communicator is NCCL, resolved with dlopen("libnccl.so.2") on first use
 *     (override: ORT_NCCL_LIB); without it every ort_comm_* call returns ORT_ENCCL and everything else still works.
 *   - There is no CPU fallback: ort_init fails with ORT_ECUDA when no sm_100 device is usable.
 */
#ifndef ORT_B200_H
#define ORT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define ORT_VERSION 200 /* 0.2.0: communicator inside the library, ort_opts.gather_stats, ort_grid_out.stats_local;
                           ort_trace3d_focus / ort_trace3d_focus_dev (through-focus sweep) and ort_spot_energy_dev /
                           ort_trace3d_energy (encircled energy), ort_wavefront_zernike_dev / ort_trace3d_zernike
                           (Zernike fit of the wavefront), ort_wavefront_psf_dev / ort_trace3d_psf (diffraction PSF)
                           and ort_wavefront_mtf_dev / ort_trace3d_mtf (diffraction MTF) added without a version
                           change */

/* status codes */
#define ORT_OK            0
#define ORT_EINVAL       (-1)
#define ORT_ECUDA        (-2)
#define ORT_ENCCL        (-3)
#define ORT_EUNSUPPORTED (-4)
#define ORT_ENOMEM       (-5)

/* limits */
#define ORT_MAX_ROWS   64   /* prescription rows incl. object space and the appended image plane */
#define ORT_MAX_FIELDS 32   /* fields per ort_trace3d_grid call */
#ifndef ORT_MAX_LENS
#define ORT_MAX_LENS  128   /* rows of a paraxial Lens matrix */
#endif
#define ORT_MAX_GPUS   16   /* contexts of one process in ort_comm_init_all / ort_trace3d_grid_multi */
#define ORT_MAX_FOCI   64   /* image planes per ort_trace3d_focus call */

/* per-ray flag bits */
#define ORT_FLAG_MISS   1u  /* conic discriminant < 0: position NaN from here on (PupilSampling.jl:9, RayTracing.jl:83) */
#define ORT_FLAG_TIR    2u  /* total internal reflection: 3-D tracer continues UNDEVIATED (PupilSampling.jl:27-30,58); 2-D tracer sets U = NaN (RayTracing.jl:164) */
#define ORT_FLAG_DOMAIN 4u  /* Julia would have thrown DomainError (sqrt/asin of an out-of-range real) */
#define ORT_FLAG_CLIP   8u  /* r_stop > a_stop (PupilSampling.jl:131-132) */
#define ORT_FLAG_VIGN  16u  /* EXTENSION (opts.vignette): hypot(x, y) > a[i] at some surface (cf. the paraxial clip, RayTracing.jl:135) */

/* arithmetic modes */
#define ORT_ARITH_STRICT 0  /* reference operation order, no FMA, IEEE div/sqrt: bit-identical to the CPU restatement */
#define ORT_ARITH_FAST   1  /* direction-cosine reformulation with FMA and Newton div/sqrt (<= 1e-12 rel.);
                               every discrete decision (miss / TIR / stop clip) that falls inside a guard band is
                               re-traced in strict arithmetic, so mask and flags stay bit-identical */

typedef struct ort_ctx ort_ctx;

/* One field point of a pupil-grid sweep (src/PupilSampling.jl:94-109,124-127). */
typedef struct ort_field {
    int32_t mode;     /* 0: System, collimated -- slopes (u, v) below are used as given (u = tan(U), the
                            caller applies tan once, :97).  1: RayBasis, finite object -- per ray
                            U = (ybar - y)/z0, V = -x/z0 then u = tan(U), v = tan(V) (:124-127, :38-39) */
    int32_t reserved;
    double  u, v;     /* mode 0 */
    double  ybar, z0; /* mode 1 */
    double  h_prime;  /* subtracted from the final y (:134) */
    /* EXTENSION (opts.opd): reference sphere centred at (opd_xc, opd_yc) on the last plane with radius
       opd_radius (0 = none: OPL to the last plane), and the reference (chief-ray) OPL subtracted */
    double  opd_xc, opd_yc, opd_radius, opl_ref;
} ort_field;

typedef struct ort_opts {
    int32_t arith;    /* ORT_ARITH_* */
    int32_t compact;  /* 0: full-grid arrays (ny*nx per field, y outer / x inner) + mask.
                         1: ex, ey, r, theta (and wx, wy) are compacted per field in the reference's push!
                            order (PupilSampling.jl:134-137); field f's segment still starts at f*ny*nx and
                            holds stats[f].n_kept entries. */
    int32_t ys_per_field; /* 0: ys[ny] shared by all fields.  1: ys[n_fields][ny], each field has its own
                             aimed y-range (the reference aims y1, y2 per field, PupilSampling.jl:99-100,121) */
    int32_t ext;          /* EXTENSION bit field (no reference counterpart; SURVEY.md 8 f3/f4): ORT_EXT_OPD accumulates the
                             optical path length per ray (out->opd = (OPL - field.opl_ref) * opd_scale, stats.mean_opd /
                             m2_opd); ORT_EXT_VIGNETTE clips at every surface's clear aperture (ort_set_apertures) */
    double  wg_nu;    /* wavegrad (PupilSampling.jl:165-167): wx = ex*wg_nu/wg_lambda.  Used iff wx/wy given. */
    double  wg_lambda;
    double  opd_scale;    /* e.g. 1/lambda for waves; used iff ORT_EXT_OPD */
    int32_t gather_stats; /* MULTI-GPU (needs ort_comm_init_*): the sweep is this rank's block of y-rows of a sharded pupil
                             grid.  Right behind the statistics kernel, on the same stream, one ncclAllGather moves the
                             n_fields x 112 B records of every rank and a merge kernel folds them in rank order (Chan), so
                             out->stats holds the statistics of the WHOLE grid, bit-identical on every rank; this rank's
                             own records go to out->stats_local.  (src/PupilSampling.jl:139-146,169-173 over all shards) */
    int32_t reserved;
} ort_opts;
#define ORT_EXT_OPD      1
#define ORT_EXT_VIGNETTE 2

/* Per-field spot statistics over KEPT rays of the traced half pupil (unmirrored); the host applies
 * the mirror algebra of PupilSampling.jl:139-146,169-173.  Merge-able across GPUs (Chan). */
typedef struct ort_stats {
    int64_t n_kept;
    double  mean_x, mean_y;   /* centroid of (ex, ey) */
    double  m2_x, m2_y;       /* sum of squared deviations about the centroid */
    double  r_max;            /* maximum(r) (:142) */
    int64_t n_miss, n_tir, n_domain, n_clip;   /* rays carrying each flag */
    int64_t n_vig;            /* EXTENSION: rays clipped by a surface aperture */
    double  mean_opd, m2_opd; /* EXTENSION: mean and sum of squared deviations of out->opd over kept rays (0 without ORT_EXT_OPD) */
    int64_t n_strict;         /* rays whose outputs come from the strict re-trace (all of them in ORT_ARITH_STRICT; in
                                 ORT_ARITH_FAST the guard-band / miss / TIR rays) */
} ort_stats;

/* Output arrays of a grid sweep; any pointer may be NULL (= not wanted). */
typedef struct ort_grid_out {
    double    *ex, *ey;       /* transverse ray errors: xf, yf - h'                       (:134-135) */
    double    *r, *theta;     /* hypot / atan at the stop surface                         (:131,133,136-137) */
    double    *wx, *wy;       /* wavegrad of ex, ey                                       (:165-167) */
    double    *opd;           /* EXTENSION: optical path difference per ray (ORT_EXT_OPD) */
    uint8_t   *mask;          /* 1 = kept (always full grid, never compacted)             (:132) */
    uint8_t   *flags;         /* ORT_FLAG_* (always full grid) */
    ort_stats *stats;         /* [n_fields]; with opts.gather_stats the records merged over all ranks */
    ort_stats *stats_local;   /* [n_fields], optional, only read with opts.gather_stats: this rank's own shard (its
                                 n_kept is the length of this rank's compacted segments) */
} ort_grid_out;

/* ---- context ------------------------------------------------------------------------------- */
int         ort_version(void);
int         ort_init(ort_ctx **out, int device);           /* device = CUDA ordinal (LOCAL_RANK) */
void        ort_free(ort_ctx *ctx);
const char *ort_last_error(ort_ctx *ctx);                  /* ctx may be NULL (error of a failed ort_init) */
int         ort_sync(ort_ctx *ctx);
int         ort_device_info(ort_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor,
                            char *name, int name_len);
/* Host placement for the PCIe copies of the host-pointer entry points (Linux).  ort_device_numa reports the NUMA node the
 * context's GPU hangs off (-1 = unknown) and that node's CPU list ("0-31,64-95").  ort_bind_host_thread pins the CALLING
 * thread to those CPUs and makes that node the preferred one for its future allocations, so pinned buffers allocated
 * afterwards (ort_host_alloc, cudaHostAlloc) land next to the GPU; with one process per GPU on a two-socket host this is
 * what keeps eight concurrent device-to-host streams off the socket interconnect.  Returns ORT_OK, or ORT_EUNSUPPORTED when
 * the node is unknown or the process may not use those CPUs (cpuset); *bound (optional) = 1 affinity set, 2 memory policy
 * set, 3 both. */
int         ort_device_numa(ort_ctx *ctx, int *node, char *cpulist, int cpulist_len);
int         ort_bind_host_thread(ort_ctx *ctx, int *bound);
void       *ort_host_alloc(size_t bytes);                  /* pinned host memory for fast D2H/H2D */
void        ort_host_free(void *p);
int64_t     ort_launch_count(ort_ctx *ctx);                /* kernels launched by this context so far */
/* Measurement: when enabled, the dominant kernel of every trace3d_grid / paraxial / transfer /
 * candidates call is bracketed by a CUDA event pair on the launching stream (ring of 64).
 * ort_profile_read synchronises those events and returns the most recent n <= max_n durations (ms,
 * oldest first), then clears the ring. */
int         ort_profile_enable(ort_ctx *ctx, int on);
int         ort_profile_read(ort_ctx *ctx, double *ms_out, int max_n);

/* Prescription = the data contract of Layout (src/Types.jl:82-95): rows x [R t n K], row 1 = object
 * space.  K may be NULL (zeros, Layout{Spherical}).  Aspheric polynomial terms `p` are Julia closures
 * and cannot cross a C ABI: the shim must reject p != zero.  For full_trace pass the EXTENDED
 * surfaces (image plane appended, t[end-1] = focus; src/PupilSampling.jl:111-114). */
int ort_set_layout(ort_ctx *ctx, int rows, const double *R, const double *t, const double *n,
                   const double *K);

/* ---- EXTENSION: aspheric polynomial terms in COEFFICIENT form.  The reference's Layout carries p::Vector{Polynomial} of Julia
 *      closures (src/Types.jl:21-27, 88-92), which cannot cross a C ABI; here p_i(y) = sum_k coef[i][k] y^k for Layout row
 *      i (row 0 = object space, ignored), k < ncoef <= ORT_MAX_POLY.  Used exactly where the reference uses p: sag + p(y)
 *      (src/PupilSampling.jl:7, src/RayTracing.jl:82 -- of the vertex-plane y only, and ignored on a plane) and tilt +
 *      dp_dy(p, .) with the reference's complex-step derivative (src/RayTracing.jl:103), in the 3-D tracers and -- with
 *      aspheric = 1 -- the 2-D tracer / ray aiming.  Call after ort_set_layout (which clears them); coef = NULL clears.
 *      ORT_ARITH_FAST: the 3-D tracers run a K-form body for surfaces with terms (analytic dp/dy; within 1e-12 of the
 *      reference arithmetic, guard-band rays re-traced strictly, clip mask and flags bit-exact); prescriptions that also
 *      hold a mirror, or terms on a PLANE (whose sag ignores p while its tilt keeps dp_dy), resolve to STRICT.
 *      Parity unpinned: the evaluation order of a user's closure is unknowable (Horner here), and the reference has no
 *      test with p != zero. */
#define ORT_MAX_POLY 18
int ort_set_polynomials(ort_ctx *ctx, int rows, int ncoef, const double *coef);

/* EXTENSION: clear semi-apertures a[rows-1] of the surfaces of the current layout (row i+1 <-> a[i]); NULL or
 * +Inf entries = unlimited.  Used iff opts.ext & ORT_EXT_VIGNETTE.  Must follow ort_set_layout. */
int ort_set_apertures(ort_ctx *ctx, int n, const double *a);

/* ---- 3-D skew real-ray trace over a pupil grid: replaces the hot loop of full_trace,
 *      src/PupilSampling.jl:115-138 (per-ray body = raytrace(...,Vector{RealRay}) :34-65) plus the
 *      statistics inputs of :139-146,169-173.  ys[ny] = collect(range(y1,y2,k)), xs[nx] =
 *      collect(range(0,y_EP,k/2)) (:121-122).  stop = system.stop (1-based), a_stop = |a[stop]|. */
int ort_trace3d_grid(ort_ctx *ctx, const ort_field *fields, int n_fields,
                     const double *ys, int ny, const double *xs, int nx,
                     int stop, double a_stop, const ort_opts *opts, ort_grid_out *out);
int ort_trace3d_grid_dev(ort_ctx *ctx, const ort_field *fields /* host */, int n_fields,
                         const double *d_ys, int ny, const double *d_xs, int nx,
                         int stop, double a_stop, const ort_opts *opts,
                         const ort_grid_out *d_out /* device pointers inside */, void *stream);

/* ---- EXTENSION (no reference method): through-focus sweep.  The same pupil-grid sweep as ort_trace3d_grid, evaluated on
 *      n_foci image planes in one pass: every ray is traced once up to the image plane and then transferred to each
 *      plane, so the results at foci[j] are those of full_trace(..., focus = foci[j]) (src/PupilSampling.jl:85,111-114).
 *      foci[j] (host, finite) replaces t[rows-2] of the current layout as the image distance; the last row must be a
 *      plane (R = +-Inf, K = 0); stop <= rows - 2.  The layout's own t[rows-2] still takes part in how ort_set_layout
 *      classifies the prescription: a non-finite value resolves ORT_ARITH_FAST to STRICT, and it is one term of the length
 *      scale L that admits spheres with |R| <= 64 L to the SIMPLE kernel.  Set it to a focus of the sweep (full_trace's
 *      paraxial one): then FAST results are bit-identical to an ort_trace3d_grid sweep at every focus whose layout
 *      classifies the same -- which only a sphere within a few percent of the 64 L bound can fail to do.
 *      Outputs (any pointer may be NULL):
 *        ex, ey                    [n_fields][n_foci][ny*nx]; with opts.compact segment (f, j) holds stats[f*n_foci + j].n_kept
 *                                  entries in push! order
 *        r, theta, mask, flags     [n_fields][ny*nx], one per field (the same at every focus); with opts.compact r and
 *                                  theta are compacted per field like ex, ey
 *        stats                     [n_fields][n_foci]: n_kept, r_max and the flag counts are the same for every focus
 *        wx, wy, opd, stats_local  must be NULL
 *      Drop rule: a ray is dropped at every focus of its field if the stop clips it, if it misses a surface, or if its
 *      position is NaN at ANY focus.  For every ray that is finite at all foci this is full_trace's own rule at each
 *      focus; the two differ only for a ray with k3 = 0 after the last glass surface.  Likewise the image plane's TIR flag
 *      (a refracting image plane) is raised iff the reference raises it at every focus: x^2 + y^2 on the plane finite at
 *      all of them (the same k3 = 0 / overflow exception).
 *      Honours opts.arith, opts.compact and opts.ys_per_field, field modes 0 and 1.  ORT_EUNSUPPORTED for opts.ext != 0,
 *      opts.gather_stats and polynomial terms on the context.  A stats-only call launches two kernels whatever n_foci;
 *      compaction adds three. */
int ort_trace3d_focus(ort_ctx *ctx, const ort_field *fields, int n_fields, const double *ys, int ny,
                      const double *xs, int nx, int stop, double a_stop,
                      const double *foci /* host, n_foci */, int n_foci, const ort_opts *opts, ort_grid_out *out);
int ort_trace3d_focus_dev(ort_ctx *ctx, const ort_field *fields /* host */, int n_fields, const double *d_ys, int ny,
                          const double *d_xs, int nx, int stop, double a_stop, const double *foci /* host */, int n_foci,
                          const ort_opts *opts, const ort_grid_out *d_out /* device pointers inside */, void *stream);

/* ---- EXTENSION (no reference method): geometric encircled / ensquared energy of the spot, computed on the device from
 *      the outputs of a grid or through-focus sweep.  These are the figures a spot_diagram summarises; unlike the RMS they
 *      are order statistics of every kept ray, so they cannot be built from the mergeable moments of ort_stats.
 *      A SET is one field of a grid sweep or one (field, focus) of a through-focus sweep: set s = f * n_foci + j, the
 *      layout of stats[f][j] and ex[f][j][.].  Its kept rays are those with mask == 1, or the first stats[s].n_kept
 *      entries of a compacted segment; n = stats[s].n_kept.
 *        centre (cx, cy)   ORT_CENTER_CENTROID: (0, stats[s].mean_y), the centroid of the MIRRORED spot that
 *                          RealRayError and its RMS describe (mirrored x has mean exactly 0).
 *                          ORT_CENTER_PARAXIAL: (0, 0), i.e. the point (0, h') -- ey is already yf - h'.
 *        distance d        dy = __dadd_rn(ey, -cy);
 *                          ORT_ENERGY_CIRCLE: d = __dsqrt_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(dy, dy))), never
 *                          contracted, so numpy.sqrt(ex*ex + dy*dy) gives the same bits;
 *                          ORT_ENERGY_SQUARE: d = max(|ex|, |dy|), the half-width of the smallest centred square.
 *                          A ray and its mirror image (-ex, ey) have the same d, so every fraction over the n traced rays
 *                          is exactly that of the 2n-point mirrored spot.
 *        counts[s][k]      #{kept i : d_i <= radii[k]} (int64) for radii[0..n_radii), finite, >= 0, strictly ascending,
 *                          n_radii <= ORT_MAX_RADII.  The encircled-energy curve is counts / n (the caller divides).
 *        radius[s][i]      for fracs[0..n_fracs), 0 < q <= 1, n_fracs <= ORT_MAX_FRACS: with
 *                          k = clamp(ceil(__dmul_rn(q, (double)n)), 1, n), the k-th smallest d of the set (1-based), a bit
 *                          pattern that occurs among its d values; NaN when n = 0.
 *      A NaN d (a kept ray never has one) sorts after +Inf and lies within no radius.  Every result is exact -- integer
 *      counts and an element of the input -- so it is bit-identical run to run and equal to a numpy sort / searchsorted
 *      on the same arrays.  n_radii = 0 or n_fracs = 0 is allowed, not both. */
#define ORT_MAX_RADII 1024
#define ORT_MAX_FRACS 8
#define ORT_ENERGY_CIRCLE   0
#define ORT_ENERGY_SQUARE   1
#define ORT_CENTER_CENTROID 0
#define ORT_CENTER_PARAXIAL 1
typedef struct ort_energy_req {
    int32_t metric, center;   /* ORT_ENERGY_*, ORT_CENTER_* */
    int32_t n_radii, n_fracs;
    const double *radii, *fracs;  /* host */
} ort_energy_req;
typedef struct ort_spot_sets {
    int32_t n_sets, sets_per_mask;  /* sets_per_mask: 1 for a grid sweep, n_foci for a focus sweep (its mask is per field) */
    int64_t stride;                 /* ny*nx: set s starts at s*stride, its mask row at (s / sets_per_mask)*stride */
    const double *ex, *ey;
    const uint8_t *mask;            /* NULL = compacted segments */
    const ort_stats *stats;         /* [n_sets]; all device pointers */
} ort_spot_sets;
/* Device form (enqueue only on `stream`): the sets already in HBM, e.g. the outputs of ort_trace3d_grid_dev /
 * ort_trace3d_focus_dev.  d_counts [n_sets][n_radii] (may be NULL when n_radii = 0), d_radius [n_sets][n_fracs] (may be
 * NULL when n_fracs = 0).  ORT_EINVAL before anything is enqueued for: a NULL array, radii not finite / negative / not
 * strictly ascending, q outside (0, 1], counts above the maxima, both zero, n_sets outside [1, ORT_MAX_FIELDS *
 * ORT_MAX_FOCI], sets_per_mask < 1, stride <= 0 or >= 2^31, an unknown metric or centre.  Launches the same number of
 * kernels whatever n, n_radii, n_fracs and n_sets; integer atomics only. */
int ort_spot_energy_dev(ort_ctx *ctx, const ort_spot_sets *sets /* host struct */, const ort_energy_req *req,
                        int64_t *d_counts, double *d_radius, void *stream);
/* Host form: the grid sweep of the layout (n_foci = 0; polynomial terms and opts.ext accepted as by ort_trace3d_grid) or
 * the through-focus sweep at foci[0..n_foci) (as ort_trace3d_focus), full grid into the context's scratch, then the
 * energy on it; only stats [n_sets] (may be NULL), counts [n_sets][n_radii] and radius [n_sets][n_fracs] cross PCIe.
 * opts.compact must be 0 (ORT_EINVAL); opts.gather_stats is ORT_EUNSUPPORTED. */
int ort_trace3d_energy(ort_ctx *ctx, const ort_field *fields, int n_fields, const double *ys, int ny, const double *xs,
                       int nx, int stop, double a_stop, const double *foci, int n_foci /* 0 = grid sweep of the layout */,
                       const ort_opts *opts, const ort_energy_req *req, ort_stats *stats, int64_t *counts, double *radius);

/* ---- EXTENSION (no reference method): Zernike decomposition of the ray-traced wavefront, fitted on the device from the
 *      outputs of a grid sweep with ORT_EXT_OPD (the OPD map that Wavefront.opd of the Python host holds).
 *      Basis: ANSI Z80.28 / OSA, single index j = (n(n+2) + m)/2 for n = 0 .. n_max, m = -n, -n+2, .., n;
 *        Z_j(rho, theta) = N_n^m R_n^|m|(rho) x {cos m theta (m > 0); sin |m| theta (m < 0); 1 (m = 0)},
 *        N_n^m = sqrt(2(n+1) / (1 + delta_m0)): every term has unit RMS over the unit disk.  This ordering is the library's;
 *        J = (n_max+1)(n_max+2)/2 terms.
 *      Pupil coordinates: the sweep's own r and theta (hypot and atan2(y, x) at the stop surface, theta from the sagittal
 *        +x axis); rho = r / r_norm with r_norm = req.r_norm if > 0, else stats[s].r_max (the reference's rho = r / max(r),
 *        src/PupilSampling.jl:142).
 *      A SET is one field of a grid sweep; its kept rays are those with mask == 1, or the first stats[s].n_kept entries of
 *        a compacted segment.  The fit is the least-squares fit of opd over the MIRRORED wavefront, 2n points (r, theta)
 *        and (r, pi - theta) with the same opd.  Under that mirror cos m theta (m even) and sin m theta (m odd) are
 *        symmetric and every other term antisymmetric; over mirrored pairs the cross terms of the two classes cancel
 *        exactly, so the device fits only the J_s symmetric terms from the n traced rays (25 at n_max = 8, 49 at 12) and
 *        returns the antisymmetric coefficients as exactly 0.0.  In exact arithmetic this is the full-basis fit of the
 *        2n-point set.  The fit solves the normal equations G c = b, G = sum z z^T, b = sum z opd, by Cholesky.
 *      Outputs per set s:
 *        coef[s][J]     ANSI order, in the units of opd;
 *        resid[s][2]    RMS and PV (max - min) of opd - sum_j c_j Z_j over the kept rays, from a second pass over them;
 *        status[s]      0 ok; 1 n_kept < J_s (including 0); 2 G not numerically positive definite: a Cholesky pivot
 *                       <= 1e-10 x its diagonal entry of G; 3 a kept ray has a non-finite opd.  For status != 0 coef and
 *                       resid are NaN.
 *      Determinism: no floating-point atomics, per-CTA partial sums folded in a fixed order, so the results are
 *      bit-identical run to run on one device.  They are not bit-equal to a numpy fit, and the full-grid (masked) and
 *      compacted forms of the same sweep may differ in the last bits (their rays fall into different partial sums). */
#define ORT_ZERN_MAX_ORDER 12
typedef struct ort_zernike_req {
    int32_t n_max, reserved;        /* 0 .. ORT_ZERN_MAX_ORDER */
    double  r_norm;                 /* > 0: pupil radius of rho = 1; 0: stats[s].r_max of each set */
} ort_zernike_req;
typedef struct ort_wave_sets {
    int32_t n_sets, reserved;
    int64_t stride;                 /* ny*nx: set s starts at s*stride */
    const double *opd, *r, *theta;
    const uint8_t *mask;            /* NULL = compacted segments */
    const ort_stats *stats;         /* [n_sets]; all device pointers */
} ort_wave_sets;
/* Device form (enqueue only on `stream`): the sets already in HBM, e.g. the outputs of ort_trace3d_grid_dev with
 * ORT_EXT_OPD.  d_coef [n_sets][J], d_resid [n_sets][2], d_status [n_sets].  ORT_EINVAL before anything is enqueued
 * for: a NULL array, n_max outside [0, ORT_ZERN_MAX_ORDER], r_norm negative or not finite, n_sets outside
 * [1, ORT_MAX_FIELDS], stride <= 0 or >= 2^31.  Launches four kernels whatever n, n_max and n_sets. */
int ort_wavefront_zernike_dev(ort_ctx *ctx, const ort_wave_sets *sets /* host struct */, const ort_zernike_req *req,
                              double *d_coef, double *d_resid, int32_t *d_status, void *stream);
/* Host form: the grid sweep of the layout (polynomial terms and vignetting accepted as by ort_trace3d_grid) full grid
 * into the context's scratch with opd, r, theta, mask and stats, then the fit on it; only stats [n_fields] (may be NULL),
 * coef [n_fields][J], resid [n_fields][2] and status [n_fields] cross PCIe.  opts.ext must hold ORT_EXT_OPD and
 * opts.compact must be 0 (ORT_EINVAL); opts.gather_stats is ORT_EUNSUPPORTED. */
int ort_trace3d_zernike(ort_ctx *ctx, const ort_field *fields, int n_fields, const double *ys, int ny, const double *xs,
                        int nx, int stop, double a_stop, const ort_opts *opts, const ort_zernike_req *req,
                        ort_stats *stats, double *coef, double *resid, int32_t *status);

/* ---- EXTENSION (no reference method): diffraction point-spread function and Strehl ratio of the ray-traced wavefront,
 *      computed on the device from the outputs of a grid sweep with ORT_EXT_OPD in full-grid form (opts.compact = 0).
 *      A SET is one field of such a sweep; its kept rays are those with mask == 1, n = stats[s].n_kept.  W_i = opd of ray
 *        i (the Python host sweeps with opd_scale = -1/lambda: W in waves, the map Wavefront.opd holds);
 *        (x_i, y_i) = (xs[ix], ys[s][iy]) its launch coordinates on the pupil grid, i = iy*nx + ix.
 *      The PSF is that of the MIRRORED 2n-point set that RealRayError, Wavefront, the encircled energy and the Zernike fit
 *        describe: every traced ray stands for (+-x_i, y_i) with the same W_i (the x = 0 column counts twice):
 *          E(xi, eta)   = sum_{kept i} sum_{sigma = +-1} exp(2 pi i (W_i + s (sigma x_i xi + y_i eta)))
 *                       = sum_i 2 cos(2 pi s x_i xi) exp(2 pi i (W_i + s y_i eta))
 *          psf(xi, eta) = |E|^2 / (2n)^2        (1 = the diffraction-limited peak of the same, possibly vignetted, pupil)
 *          strehl_ref   = |sum_i exp(2 pi i W_i)|^2 / n^2     (psf at xi = eta = 0)
 *      Pixel (iu, iv) sits at xi = (iu - (n_u-1)/2) du, eta = (iv - (n_v-1)/2) dv, relative to the centre of the
 *        reference sphere (opd_xc, opd_yc), the chief ray's image point; xi runs along x (sagittal), eta along y.
 *      s = req.scale > 0, in cycles per (pupil unit x image unit).  The Python host passes s = 1/(lambda f), f = system.f:
 *        the sine-condition mapping of an entrance-pupil height h to the image-space direction sine h/f, i.e. the scalar
 *        Fraunhofer ("FFT PSF") model.  Obliquity, amplitude apodisation and pupil distortion are neglected.
 *      The grid wraps (aliases) with period 1/(s dx) in xi and 1/(s dy) in eta for uniform pupil steps dx, dy.
 *      Outputs per set s:
 *        psf[s][n_v][n_u];
 *        strehl[s][2]   (strehl_ref, the maximum of psf over the pixel grid);
 *        peak[s]        iv*n_u + iu of that maximum, the lowest index on a tie;
 *        status[s]      0 ok; 1 n = 0; 3 a kept ray has a non-finite opd (the codes of the Zernike fit; 2 is unused).
 *                       For status != 0 psf and strehl are NaN and peak is -1.
 *      The device may use y - ybar_s for phase accuracy (|E|^2 does not change).  Determinism: no floating-point atomics,
 *      partial sums folded in a fixed order: bit-identical run to run on one device, not bit-equal to numpy. */
#define ORT_PSF_MAX_SIDE 1024
typedef struct ort_psf_req {
    int32_t n_u, n_v;               /* pixels along xi and eta, 1 .. ORT_PSF_MAX_SIDE */
    double  du, dv;                 /* pixel pitch in image units, finite and > 0 */
    double  scale;                  /* s, finite and > 0 */
} ort_psf_req;
/* Device form (enqueue only on `stream`): the sets already in HBM in full-grid form (sets->mask required; r and theta are
 * not read), d_ys [ys_per_set ? n_sets : 1][ny] and d_xs [nx] the grid coordinates on the device.  d_psf
 * [n_sets][n_v][n_u], d_strehl [n_sets][2], d_peak and d_status [n_sets].  ORT_EINVAL before anything is enqueued for:
 * a NULL array, stride != ny*nx, ny or nx < 1, n_sets outside [1, ORT_MAX_FIELDS], n_u or n_v outside
 * [1, ORT_PSF_MAX_SIDE], du, dv or scale not finite or <= 0.  Launches five kernels whatever the sizes.  Scratch: the
 * stage-A products take 16 n_sets kx ny nup bytes (nup = ceil(n_u / 2) rounded up to 64 or 128, kx <= 4 chunks of nx),
 * about 2 kx nup / nx times the OPD input: small on wide grids, large on tall narrow ones (nx = 1 at n_u 1024 is 8 KB
 * per pupil row per set); the stage-B partials take 16 n_sets ky n_v ceil(n_u / 2) bytes (ky > 1 only while the pixel
 * tiles alone leave SMs idle).  A scratch that cannot grow is ORT_ENOMEM. */
int ort_wavefront_psf_dev(ort_ctx *ctx, const ort_wave_sets *sets /* host struct */, const double *d_ys, int ys_per_set,
                          int ny, const double *d_xs, int nx, const ort_psf_req *req, double *d_psf, double *d_strehl,
                          int32_t *d_peak, int32_t *d_status, void *stream);
/* Host form: the grid sweep of the layout (polynomial terms and vignetting accepted as by ort_trace3d_grid) full grid
 * into the context's scratch with opd, mask and stats, then the PSF on it; only stats [n_fields] (may be NULL),
 * psf [n_fields][n_v][n_u], strehl [n_fields][2], peak and status [n_fields] cross PCIe.  opts.ext must hold ORT_EXT_OPD
 * and opts.compact must be 0 (ORT_EINVAL); opts.gather_stats is ORT_EUNSUPPORTED. */
int ort_trace3d_psf(ort_ctx *ctx, const ort_field *fields, int n_fields, const double *ys, int ny, const double *xs, int nx,
                    int stop, double a_stop, const ort_opts *opts, const ort_psf_req *req, ort_stats *stats, double *psf,
                    double *strehl, int32_t *peak, int32_t *status);

/* ---- EXTENSION (no reference method): diffraction modulation transfer function of the ray-traced wavefront, computed on
 *      the device from the outputs of a grid sweep with ORT_EXT_OPD in full-grid form (opts.compact = 0): the optical
 *      transfer function of the PSF that ort_wavefront_psf_dev defines (same sets, same scale s, same mirrored pupil),
 *      along two azimuths.
 *      A SET is as for the PSF: W_i = opd (waves when the Python host sweeps with opd_scale = -1/lambda), P[iy][ix] =
 *        exp(2 pi i W) for kept rays (mask == 1) and 0 otherwise, n = stats[s].n_kept.
 *      The pupil must be a MIRRORED LATTICE, defined by index, not by value: xs[0] == 0, dx = xs[nx-1]/(nx-1) finite and
 *        > 0, dy_s = (ys_s[ny-1] - ys_s[0])/(ny-1) finite and != 0 (the host's ys run downwards from y1 > y2: dy_s < 0).
 *        The host's grids (xs = range(0, y_EP, k/2), ys = range(y1, y2, k)) have this form to within an ulp per element.
 *      Mirrored amplitude, jx in [-(nx-1), nx-1]: A[iy][jx] = P[iy][|jx|] for jx != 0, A[iy][0] = 2 P[iy][0].
 *          C_sag(k) = sum_iy sum_jx A[iy][jx+k] conj A[iy][jx]        k = 0 .. 2(nx-1)   (real: the mirror)
 *          C_tan(k) = sum_jx sum_iy A[iy+k][jx] conj A[iy][jx]        k = 0 .. ny-1
 *                   = sum_ix w_ix sum_iy P[iy+k][ix] conj P[iy][ix],  w_0 = 4, w_ix = 2 otherwise
 *          OTF(k)   = C(k) / C(0)     (C(0) = 2n + 2n0 for both, n0 = kept rays in the x = 0 column; OTF(0) = 1 exactly)
 *        i.e. OTF(nu) = int psf exp(-2 pi i nu . (xi, eta)) / int psf of that PSF: sagittal = nu along xi (x) at
 *        nu = k s dx, tangential = nu along eta (y) at nu = k s |dy_s|.  For dy_s < 0 a frequency nu > 0 pairs rows iy + k
 *        with iy the other way round, and the tangential OTF is conj C_tan(k) / C(0).
 *      Requested frequencies req.freqs[0 .. n_freq), cycles per image unit, finite and >= 0, in any order.  Per azimuth,
 *        q = nu / (s d) with d = dx or |dy_s|, k0 = floor(q), f = q - k0:
 *          OTF(nu) = (1 - f) OTF(k0) + f OTF(k0 + 1),   OTF(k) = 0 past the last lag.
 *        The diffraction cutoffs of the sampled pupil are 2 (nx-1) dx s (= 2 y_EP s = 1/(lambda F#) on the host's grids)
 *        and (ny-1) |dy_s| s.
 *      Outputs per set s:
 *        otf[s][2][n_freq][2]  [0] sagittal, [1] tangential; (re, im).  The sagittal imaginary part is exactly 0.
 *        status[s]             0 ok; 1 n = 0; 3 a kept ray has a non-finite opd (the PSF's codes); 4 the grid is not a
 *                              mirrored lattice (read from d_xs and d_ys).  The lowest code that applies.  For
 *                              status != 0 otf is NaN.
 *      Determinism: no floating-point atomics, partial sums folded in a fixed order: bit-identical run to run on one
 *      device, not bit-equal to numpy. */
#define ORT_MTF_MAX_FREQS 1024
typedef struct ort_mtf_req {
    int32_t n_freq, reserved;       /* 1 .. ORT_MTF_MAX_FREQS */
    const double *freqs;            /* host array [n_freq] */
    double  scale;                  /* s, as ort_psf_req.scale: finite and > 0 */
} ort_mtf_req;                      /* 24 bytes */
/* Device form (enqueue only on `stream`): the sets already in HBM in full-grid form (sets->mask required; r and theta are
 * not read), d_ys [ys_per_set ? n_sets : 1][ny] and d_xs [nx] the grid coordinates on the device.  d_otf
 * [n_sets][2][n_freq][2], d_status [n_sets].  ORT_EINVAL before anything is enqueued for: a NULL array, stride != ny*nx,
 * stride >= 2^31, nx < 2 or ny < 2, n_sets outside [1, ORT_MAX_FIELDS], n_freq outside [1, ORT_MTF_MAX_FREQS], a frequency negative or
 * not finite, scale not finite or <= 0.  Launches four kernels whatever the sizes.  Scratch: the pupil amplitude, once
 * row-major and once transposed, takes 32 n_sets ny nx bytes (2.7 GB for 5 fields of 5792 x 2896 rays, four times the
 * OPD input); the lag partials take 24 n_sets (2 n_freq + 1) g bytes with g <= a few thousand row groups.  A scratch
 * that cannot grow is ORT_ENOMEM. */
int ort_wavefront_mtf_dev(ort_ctx *ctx, const ort_wave_sets *sets /* host struct */, const double *d_ys, int ys_per_set,
                          int ny, const double *d_xs, int nx, const ort_mtf_req *req, double *d_otf, int32_t *d_status,
                          void *stream);
/* Host form: the grid sweep of the layout (polynomial terms and vignetting accepted as by ort_trace3d_grid) full grid
 * into the context's scratch with opd, mask and stats, then the MTF on it; only stats [n_fields] (may be NULL),
 * otf [n_fields][2][n_freq][2] and status [n_fields] cross PCIe.  opts.ext must hold ORT_EXT_OPD and opts.compact must
 * be 0 (ORT_EINVAL); opts.gather_stats is ORT_EUNSUPPORTED. */
int ort_trace3d_mtf(ort_ctx *ctx, const ort_field *fields, int n_fields, const double *ys, int ny, const double *xs, int nx,
                    int stop, double a_stop, const ort_opts *opts, const ort_mtf_req *req, ort_stats *stats, double *otf,
                    int32_t *status);

/* ---- 3-D skew trace of N arbitrary rays, all surfaces recorded: replaces
 *      raytrace(surfaces, y, x, U, V, Vector{RealRay}) src/PupilSampling.jl:34-65 for a batch.
 *      u0, v0 are SLOPES tan(U), tan(V).  xv, yv: [(rows-1)][N] (ray index fastest);
 *      kout: [3][N] final direction cosines (k[1], k[2], k[3] of :40); any output may be NULL. */
int ort_trace3d_rays(ort_ctx *ctx, int64_t N, const double *y0, const double *x0,
                     const double *u0, const double *v0, int arith,
                     double *xv, double *yv, double *kout, uint8_t *flags);
/* EXTENSION: same, plus the optical path length to the last surface (opl[N], start term 0) and
 * per-surface aperture flags when apertures are set. */
int ort_trace3d_rays_opl(ort_ctx *ctx, int64_t N, const double *y0, const double *x0,
                         const double *u0, const double *v0, int arith,
                         double *xv, double *yv, double *kout, uint8_t *flags, double *opl);
/* device-pointer form (enqueue only on `stream`): rays and outputs already in HBM, layouts as above; any output
 * pointer may be NULL */
int ort_trace3d_rays_dev(ort_ctx *ctx, int64_t N, const double *d_y0, const double *d_x0, const double *d_u0,
                         const double *d_v0, int arith, double *d_xv, double *d_yv, double *d_kout,
                         uint8_t *d_flags, double *d_opl, void *stream);

/* ---- 2-D meridional real-ray trace of N rays: replaces raytrace(surfaces, y, U, RealRay)
 *      src/RayTracing.jl:145-173.  aspheric = 1 is the Layout{Aspheric} method (:171-173: K from the
 *      layout, atan(tilt) branch); 0 the AbstractMatrix method (K = 0, asin(y/R) branch, :162).
 *      y_out, U_out, ts_out: [rows][N]; any may be NULL. */
int ort_trace2d_batch(ort_ctx *ctx, int64_t N, const double *y0, const double *U0, int aspheric,
                      double *y_out, double *U_out, double *ts_out, uint8_t *flags);

/* ---- ray aiming on the device (SURVEY.md section 8 f1): N independent secant solves, one thread each, over the
 *      2-D meridional tracer of the current layout.  Finds x (the entrance height y if vary_u = 0, the entrance
 *      angle U if vary_u = 1) such that the ray's height at surface `stop` equals target[j].
 *      mode 0 = the reference's iteration (src/RayTracing.jl:229-233, 282-286): fixed step eps = sqrt(eps()),
 *               x -= f eps / (f(x + eps) - f) while |f| > atol;
 *      mode 1 = root polish used for the edge rays (src/PupilSampling.jl:67-83 minimises |f| with Optim.BFGS; the
 *               same root is found by a secant iteration with relative step until |f| <= 4e-16 scale or stagnation).
 *      other[j] is the fixed coordinate (U if vary_u = 0, y if vary_u = 1).  iters (optional) returns the iteration
 *      count, negative if the solve left the domain or did not converge. */
int ort_aim2d(ort_ctx *ctx, int64_t N, const double *x_start, const double *other, const double *target,
              int stop, int vary_u, int mode, double atol_or_scale, int aspheric, double *x_out, int32_t *iters);

/* ---- paraxial y-nu trace of N rays through a k-row Lens [tau phi]: replaces
 *      raytrace(lens, y, w, a; clip) src/RayTracing.jl:127-143 (+ :55-69).  a may be NULL (no clip).
 *      y, w: final (y, nu) per ray (NaN if clipped); clip_idx: 1-based row where clipped, 0 if not;
 *      y_all, w_all: optional full tables [(k+1)][N] (the reference's rt). */
int ort_paraxial_batch(ort_ctx *ctx, int k, const double *tau, const double *phi, const double *a,
                       int clip, int arith, int64_t N, const double *y0, const double *w0,
                       double *y, double *w, int32_t *clip_idx, double *y_all, double *w_all);
int ort_paraxial_batch_dev(ort_ctx *ctx, int k, const double *tau, const double *phi,
                           const double *a, int clip, int arith, int64_t N,
                           const double *d_y0, const double *d_w0, double *d_y, double *d_w,
                           int32_t *d_clip_idx, double *d_y_all, double *d_w_all, void *stream);

/* ---- transfer-matrix apply to N rays: replaces transfer(M, v, tau, taup) and
 *      reverse_transfer(M, v, taup, tau), src/TransferMatrix.jl:8-17.  M: 2x2 column-major
 *      (Julia memory order).  v_in / v_out: 2 x N column-major = interleaved [y nu] pairs. */
int ort_transfer_batch(ort_ctx *ctx, const double M[4], double tau, double taup, int reverse,
                       int64_t N, const double *v_in, double *v_out);
int ort_transfer_batch_dev(ort_ctx *ctx, const double M[4], double tau, double taup, int reverse,
                           int64_t N, const double *d_v_in, double *d_v_out, void *stream);

/* ---- candidate-batched 3-D trace (BASELINE config 5; a synthetic batch of PupilSampling.jl:34-65,
 *      115-138 with no reference counterpart): C prescriptions RtnK[C][4][rows], one shared entrance
 *      grid ys x xs and one collimated field.  out[C][4] = n_kept, mean_x, mean_y, RMS about centroid. */
int ort_trace3d_candidates(ort_ctx *ctx, int rows, int64_t C, const double *RtnK,
                           const ort_field *field, const double *ys, int ny, const double *xs,
                           int nx, int stop, double a_stop, int arith, double *out);
int ort_trace3d_candidates_dev(ort_ctx *ctx, int rows, int64_t C, const double *d_RtnK,
                               const ort_field *field, const double *d_ys, int ny,
                               const double *d_xs, int nx, int stop, double a_stop, int arith,
                               double *d_out, void *stream);

/* ---- per-candidate prelude of full_trace (SURVEY.md section 8 f1): what src/PupilSampling.jl:85-108 does before the grid
 *      loop, for C candidate prescriptions at once, one thread per candidate: first-order solve (src/RayTracing.jl
 *      :208-221, :246-263, stop = argmin a ./ y), real chief ray traced backwards through the reversed prescription
 *      (:265-296, the Layout branch :272-274), real marginal ray (:223-240), field angle U = |H| * Ubar and the two
 *      edge rays (src/PupilSampling.jl:67-83; the roots the reference's BFGS-on-abs converges to, found by secant).
 *      RtnK[C][4][rows] WITHOUT the image-plane row, shared apertures a[rows-1] (host), image height h_prime of
 *      solve(surfaces, a, h_prime), relative field H, aspheric = the Layout{Aspheric} dispatch of the forward 2-D traces.
 *      out[C][24] = y1, y2, y_EP, u = tan U, h' = u f, focus (BFD), stop, a_stop, EP_t, Ubar, f, status (0 = ok;
 *      bit 0 chief / bit 1 marginal / bit 2 edge-ray aiming failed, 8 = unusable last row), marginal nu[end], U,
 *      [14] = 1 when [16..23] hold the two edge rays (y1, y2 at x = 0) taken through the strict 3-D trace: keep, eps_x,
 *      eps_y, r^2 each -- they sit exactly on the stop rim, i.e. always inside the guard band of the FAST clip test, so
 *      the sweep reads them from here instead of serialising a strict re-trace in every CTA.
 *      ort_trace3d_candidates_aimed consumes these records: every candidate is traced over ITS OWN aimed pupil grid
 *      ys = range(y1, y2, ny), xs = range(0, y_EP, nx), with its own stop / a_stop / u / h' and the image plane appended
 *      at its own focus (:111-114); out[C][4] as ort_trace3d_candidates (NaN for a candidate whose prelude failed). */
#define ORT_AIM_NOUT 24
int ort_aim_candidates(ort_ctx *ctx, int rows, int64_t C, const double *RtnK, const double *a, double h_prime,
                       double H, int aspheric, double *out);
int ort_aim_candidates_dev(ort_ctx *ctx, int rows, int64_t C, const double *d_RtnK, const double *a /* host */,
                           double h_prime, double H, int aspheric, double *d_out, void *stream);
/* The same prelude for ONE system at n_fields relative fields Hs[] (<= ORT_MAX_FIELDS), i.e. src/PupilSampling.jl:85-108 of
 * a field sweep in one call (two launches): R, t, n, K are the rows of the Layout (K may be NULL), out[n_fields][24]. */
int ort_aim_fields(ort_ctx *ctx, int rows, const double *R, const double *t, const double *n, const double *K,
                   const double *a, double h_prime, const double *Hs, int n_fields, int aspheric, double *out);
int ort_trace3d_candidates_aimed(ort_ctx *ctx, int rows, int64_t C, const double *RtnK, const double *aim, int ny,
                                 int nx, int arith, double *out);
int ort_trace3d_candidates_aimed_dev(ort_ctx *ctx, int rows, int64_t C, const double *d_RtnK, const double *d_aim,
                                     int ny, int nx, int arith, double *d_out, void *stream);

/* ---- candidate-batched first-order solve + Seidel sums (SURVEY.md section 8 f2): what the reference's optimize()
 *      evaluates per candidate (src/Optimization.jl:32-45): Lens(surfaces) src/RayTracing.jl:38-53, paraxial marginal
 *      and chief rays :208-221, :246-263, aberrations() src/SeidelAberrations.jl:6-53.  RtnK[C][4][rows] (K unused),
 *      shared apertures a[rows-1], image height h_prime, wavelength lambda, dispersion dn[rows] (NULL = zeros).
 *      out[C][16] = f, EBFD, stop, H, W040, W131, W222, W220P, W311, W020, W111, W220, W220M, W220T, marginal nu[end],
 *      chief nu[1]; per_surface (optional, [C][7][rows-1]) = spherical, coma, astigmatism, petzval, distortion, axial,
 *      lateral.  One thread per candidate, reference operation order (bit-identical to the CPU restatement). */
#define ORT_SEIDEL_NOUT 16
int ort_seidel_candidates(ort_ctx *ctx, int rows, int64_t C, const double *RtnK, const double *a, double h_prime,
                          double lambda, const double *dn, double *out, double *per_surface);
int ort_seidel_candidates_dev(ort_ctx *ctx, int rows, int64_t C, const double *d_RtnK, const double *a /* host */,
                              double h_prime, double lambda, const double *dn /* host */, double *d_out,
                              double *d_per_surface, void *stream);

/* ---- candidate-batched vignetting(system, a) (SURVEY.md section 8 f3; src/Vignetting.jl:1-30, type src/Types.jl:169-176).
 *      RtnK[C][4][rows]; a_solve[rows-1] = the apertures solve() picks the stop with; a_vig[rows-1] (NULL = a_solve)
 *      = the semi-diameters under test.  k = rows - 1.  out[C][6 k + 12]:
 *        [0 .. 5k)   M, column-major k x 5: a, limited |y|, unvignetted |y| + |ybar|, half |ybar|, full |ybar| - |y|
 *                    (half / full NaN where < |y|, :12-13)
 *        [5k .. 6k)  per-surface code: 1 = limit (:27), 2 = partial (:29), 4 = full (:28)
 *        [6k .. 6k+9) FOV 3 x 3 row-major: rows unvignetted / half / fully vignetted, columns 2 atand(u), u, h' (:20-26)
 *        6k+9 un (:15), 6k+10 stop, 6k+11 f.
 *      One thread per candidate, reference operation order; atand is CUDA libm atan * 180/pi (last-ulp, not bit, parity). */
#define ORT_VIG_TAIL 12
int ort_vignetting_candidates(ort_ctx *ctx, int rows, int64_t C, const double *RtnK, const double *a_solve,
                              const double *a_vig, double h_prime, double *out);
int ort_vignetting_candidates_dev(ort_ctx *ctx, int rows, int64_t C, const double *d_RtnK, const double *a_solve /* host */,
                                  const double *a_vig /* host */, double h_prime, double *d_out, void *stream);

/* ---- communicator inside the library (SURVEY.md section 8 b "Threading", 8 e): rays shard by contiguous blocks of y-rows
 *      (the outer loop index of src/PupilSampling.jl:123), candidate prescriptions by contiguous ranges; the only exchange
 *      is the all-gather of per-field statistics records (or of the 32 B-per-candidate merit table).
 *      One process per GPU:   rank 0 calls ort_comm_unique_id, ships the 128 bytes to the other ranks by any means (file,
 *                             environment, MPI, a torch.distributed store), every rank calls ort_comm_init_rank.
 *      One process, n GPUs:   ort_comm_init_all over n contexts on n distinct devices (ncclCommInitAll); then
 *                             ort_trace3d_grid_multi drives all of them from one host thread. */
#define ORT_COMM_ID_BYTES 128
int ort_comm_unique_id(void *id /* ORT_COMM_ID_BYTES */);
int ort_comm_init_rank(ort_ctx *ctx, const void *id, int rank, int world);
int ort_comm_init_all(ort_ctx **ctxs, int n);
int ort_comm_info(ort_ctx *ctx, int *rank, int *world, int *nccl_version);   /* world = 0: no communicator */
int ort_comm_free(ort_ctx *ctx);                                               /* also done by ort_free */
/* [lo, hi) of `total` items owned by `rank` of `world`: contiguous, sizes differ by at most one */
int ort_comm_range(int64_t total, int rank, int world, int64_t *lo, int64_t *hi);

/* Whole pupil grid over n contexts of ONE process (host pointers, synchronous): replaces the hot loop + reductions of
 * full_trace (src/PupilSampling.jl:115-146,169-173) exactly like ort_trace3d_grid, with the ny y-rows block-sharded over
 * the contexts.  Arguments and outputs as ort_trace3d_grid -- ys / xs / out describe the WHOLE grid; rank-order
 * concatenation of the shards reproduces the reference's loop (and push!) order; out->stats is merged over the shards
 * by the library's all-gather + merge kernel (identical on every device); out->stats_local, if given, is
 * [n][n_fields].  The layout (and apertures / polynomial terms) of ctxs[0] is used on every context. */
int ort_trace3d_grid_multi(ort_ctx **ctxs, int n, const ort_field *fields, int n_fields, const double *ys, int ny,
                           const double *xs, int nx, int stop, double a_stop, const ort_opts *opts, ort_grid_out *out);

/* BASELINE config 5 across ranks: this rank runs the per-candidate prelude (ort_aim_candidates) and the aimed sweep
 * (ort_trace3d_candidates_aimed) on ITS contiguous range ort_comm_range(C) of the population, then the ranks' segments of
 * the merit table are exchanged (one grouped NCCL broadcast per rank = an all-gather with uneven counts) so out[C][4]
 * is complete on every rank.  RtnK is the WHOLE population [C][4][rows] (replicated; only this rank's range is read).
 * Without a communicator (world 1) it is the plain prelude + sweep.  aim (optional, [C][ORT_AIM_NOUT]) receives this
 * rank's prelude records in place (rows of other ranks untouched). */
int ort_candidates_sharded(ort_ctx *ctx, int rows, int64_t C, const double *RtnK, const double *a, double h_prime,
                           double H, int aspheric, int ny, int nx, int arith, double *aim, double *out);
int ort_candidates_sharded_dev(ort_ctx *ctx, int rows, int64_t C, const double *d_RtnK, const double *a /* host */,
                               double h_prime, double H, int aspheric, int ny, int nx, int arith, double *d_aim,
                               double *d_out, void *stream);

/* ---- multi-GPU combine (host arithmetic): Chan merge of per-shard records recs[n_shards][n_fields], folded in
 *      shard (rank) order so every rank gets bit-identical results, and the reference's sigma of the mirrored spot
 *      (src/PupilSampling.jl:140-146,169-173) from one record. */
int    ort_merge_stats(const ort_stats *recs, int n_shards, int n_fields, ort_stats *out);
/* the same fold on the device (the merge kernel behind opts.gather_stats), for records already gathered in HBM:
 * bit-identical to ort_merge_stats.  Enqueue only. */
int    ort_merge_stats_dev(ort_ctx *ctx, const ort_stats *d_recs, int n_shards, int n_fields, ort_stats *d_out, void *stream);
double ort_rms_from_stats(const ort_stats *s);

/* ---- measurement helper: register-resident DFMA-chain microbenchmark; the FP64 roofline
 *      denominator (MEASURED_PEAKS.json holds no FP64 figure).  Returns TFLOP/s (2 flop per DFMA). */
int ort_fp64_peak(ort_ctx *ctx, double *tflops, double *ms);

/* Self-test of the STRICT kernels' division and square root (correctly rounded fast paths with the slow path deferred to a
 * per-ray re-trace, csrc/ort_internal.cuh xdiv / xsqrt) against the CUDA library's __ddiv_rn / __dsqrt_rn on >= n operand
 * pairs: random bit patterns, moderate magnitudes, every exponent, special values.  out8: [0] divisions tested, [1] flagged
 * for the slow path, [2] kept and different from the intrinsic (must be 0); [3..5] the same for square roots; [6], [7] flags
 * raised among operands of moderate magnitude (division: only zero numerators; square root: 0).  No reference counterpart. */
int ort_selftest_exact_ops(ort_ctx *ctx, long long n, unsigned long long seed, long long *out8);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* ORT_B200_H */
