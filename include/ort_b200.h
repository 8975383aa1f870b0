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
                           ort_trace3d_focus / ort_trace3d_focus_dev (through-focus sweep) added without a version change */

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
