/*
 * ort_oracle.c -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE)
 *
 * A plain-C restatement of the data-parallel hot path of Sagnac/OpticalRayTracing.jl
 * (pure Julia; Julia is not installed in this image, so the reference itself cannot
 * run here).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may call this; the product (libort_b200.so and the host
 * package) never links, imports or executes it.
 *
 * Parity pinning: see oracle/README.md.  The functions here are pinned against every
 * known-answer test the reference holds for this path (test/runtests.jl:53-60,
 * 62-113, 115-146, 231-239, 252-257, 260-286, 334-344, 355-372, 376-387) by
 * tests/test_oracle_*.py.  Quantities NO reference test pins (per-ray mask, r, theta,
 * output order, wavegrad, direction cosines, and the Optim.jl BFGS end points y1,y2)
 * are "parity unpinned": fidelity there is restatement fidelity only.
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math (see oracle/Makefile).  Julia never
 * contracts a*b+c into an FMA, so neither may this file; the one explicit fma() use
 * is the restatement of Julia Base's hypot, which calls fma itself.
 *
 * Every function cites the reference file:line (relative to /root/reference) it follows.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_API __attribute__((visibility("default")))

/* ---- flag bits shared with include/ort_b200.h (ORT_FLAG_*) ---- */
#define F_MISS   1u   /* sag discriminant < 0 -> NaN (PupilSampling.jl:9, RayTracing.jl:83) */
#define F_TIR    2u   /* refract! returned NaN, ray continues undeviated (PupilSampling.jl:27-30, :58) */
#define F_DOMAIN 4u   /* Julia would have thrown DomainError (sqrt/asin of out-of-range real) */
#define F_CLIP   8u   /* dropped by the stop-radius test (PupilSampling.jl:131-132) */

/* Julia Base sign(): sign(0)=0, sign(NaN)=NaN, sign(+-Inf)=+-1 */
static inline double jl_sign(double x) { return x < 0.0 ? -1.0 : (x > 0.0 ? 1.0 : x); }

/* ------------------------------------------------------------------------------------
 * EXTENSION: aspheric polynomial terms in COEFFICIENT form.  The reference's Layout carries
 * p::Vector{Polynomial} of Julia closures (src/Types.jl:21-27, 88-92), which cannot cross a C ABI;
 * here p_i(y) = sum_k coef[i][k] y^k (Horner, highest power first).  Where the reference uses p:
 * sag + p(y) (src/PupilSampling.jl:7, src/RayTracing.jl:82 -- p of the vertex-plane y only, and
 * ignored on a plane, :12 / :87) and tilt + dp_dy(p, .) with the complex-step derivative
 * dp_dy(p, y) = imag(p(complex(y, eps))) / eps, eps = sqrt(eps()) (src/RayTracing.jl:103).
 * The evaluation order of a user's closure is unknowable: parity unpinned.  State is process-
 * global (set before a batch, read-only during it).
 * ---------------------------------------------------------------------------------- */
#define ORC_MAX_POLY 18
static int g_poly_rows = 0, g_poly_n = 0;
static double g_poly[64 * ORC_MAX_POLY];

ORC_API int orc_set_poly(int rows, int ncoef, const double *coef)
{
    if (!coef || rows <= 0 || ncoef <= 0) { g_poly_rows = g_poly_n = 0; return 0; }
    if (rows > 64 || ncoef > ORC_MAX_POLY) return -1;
    g_poly_rows = rows; g_poly_n = ncoef;
    for (int i = 0; i < rows * ncoef; i++) g_poly[i] = coef[i];
    return 0;
}

static inline int poly_on(int row) { return g_poly_n > 0 && row < g_poly_rows; }

/* p_row(y); 0.0 (Julia's zero) without polynomials */
static inline double poly_eval(int row, double y)
{
    if (!poly_on(row)) return 0.0;
    const double *c = g_poly + (size_t)row * g_poly_n;
    double acc = c[g_poly_n - 1];
    for (int k = g_poly_n - 2; k >= 0; k--) acc = acc * y + c[k];
    return acc;
}

/* dp_dy(p_row, y) = imag(p(complex(y, eps))) / eps -- complex Horner with Julia's complex product
 * (a + bi)(c + di) = (ac - bd) + (ad + bc)i; 0.0 without polynomials */
static inline double poly_dpdy(int row, double y)
{
    if (!poly_on(row)) return 0.0;
    const double eps = 1.4901161193847656e-08;
    const double *c = g_poly + (size_t)row * g_poly_n;
    double re = c[g_poly_n - 1], im = 0.0;
    for (int k = g_poly_n - 2; k >= 0; k--) {
        double nre = re * y - im * eps + c[k];
        double nim = re * eps + im * y;
        re = nre; im = nim;
    }
    return im / eps;
}

/* Julia Base.Math._hypot for Float64 on an FMA-capable host (base/math.jl, not under
 * /root/reference).  Used by full_trace for the stop-radius mask, PupilSampling.jl:131.
 * The fma branch is correctly rounded, so the value equals any correctly rounded hypot. */
ORC_API double orc_hypot(double x, double y)
{
    double ax = fabs(x), ay = fabs(y);
    if (isinf(ax) || isinf(ay)) return INFINITY;
    if (ay > ax) { double tmp = ax; ax = ay; ay = tmp; }
    if (ay <= ax * 1.0536712127723509e-08 /* sqrt(eps/2) */) return ax; /* NaN falls through */
    double scale = 3.3121686421112381e-170; /* eps*sqrt(floatmin) */
    if (ax > 9.480751908109176e153 /* sqrt(floatmax/2) */) {
        ax *= scale; ay *= scale; scale = 1.0 / scale;
    } else if (ay < 1.4916681462400413e-154 /* sqrt(floatmin) */) {
        ax /= scale; ay /= scale;
    } else {
        scale = 1.0;
    }
    double h = sqrt(fma(ax, ax, ay * ay));
    double hsq = h * h, axsq = ax * ax;
    h -= (fma(-ay, ay, hsq - axsq) + fma(h, h, -hsq) - fma(ax, ax, -axsq)) / (2.0 * h);
    return h * scale;
}

/* ------------------------------------------------------------------------------------
 * Paraxial y-nu path
 * ---------------------------------------------------------------------------------- */

/* Lens(surfaces) -- src/RayTracing.jl:38-53.  Returns k (rows of the Lens matrix).
 * tau, phi must hold `rows` doubles.  Note :42 zeroes t[1] when it is not finite. */
ORC_API int orc_lens(int rows, const double *R, const double *t, const double *n,
                     double *tau, double *phi)
{
    for (int i = 0; i < rows; i++) {
        double ti = t[i];
        if (i == 0 && !isfinite(ti)) ti = 0.0;      /* t[1] *= isfinite(t[1])   :42 */
        tau[i] = ti / n[i];                          /* @. M[:,1] = t / n        :43 */
    }
    for (int i = 0; i + 1 < rows; i++)
        phi[i] = (n[i + 1] - n[i]) / R[i + 1];       /* :45 */
    double tend = (rows == 1 && !isfinite(t[0])) ? 0.0 : t[rows - 1];
    if (tend == 0.0 || !isfinite(tend)) return rows - 1;   /* :47-48 */
    phi[rows - 1] = 0.0;                             /* :50 */
    return rows;
}

/* transfer(y,w,tau) / refract(y,w,phi) -- src/RayTracing.jl:55-69 */
static inline double px_transfer(double y, double w, double tau)
{
    return isfinite(tau) ? y + w * tau : y;
}
static inline double px_refract(double y, double w, double phi) { return w - y * phi; }

/* raytrace(lens, y, w, a; clip) -- src/RayTracing.jl:127-143.
 * rt is (k+1) x 2 column-major (y column then nu column), as Julia stores it.
 * Returns the 1-based row index i at which the ray was clipped, 0 if not clipped. */
ORC_API int orc_paraxial_trace(int k, const double *tau, const double *phi, const double *a,
                               int clip, double y, double w, double *rt)
{
    int ld = k + 1;
    rt[0] = y; rt[ld] = w;
    for (int i = 0; i < k; i++) {
        y = px_transfer(y, w, tau[i]);
        w = px_refract(y, w, phi[i]);
        if (clip && a && fabs(y) - a[i] > 1e-13) {   /* :135 */
            for (int j = i + 1; j < ld; j++) { rt[j] = NAN; rt[ld + j] = NAN; }  /* :136 */
            return i + 1;
        }
        rt[i + 1] = y; rt[ld + i + 1] = w;
    }
    return 0;
}

/* Batched form used as oracle for ort_paraxial_batch: final (y, nu) and clip index only. */
ORC_API void orc_paraxial_batch(int k, const double *tau, const double *phi, const double *a,
                                int clip, int64_t N, const double *y0, const double *w0,
                                double *y_out, double *w_out, int32_t *clip_idx, int threads)
{
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel for schedule(static)
#endif
    for (int64_t r = 0; r < N; r++) {
        double y = y0[r], w = w0[r];
        int ci = 0;
        for (int i = 0; i < k; i++) {
            y = px_transfer(y, w, tau[i]);
            w = px_refract(y, w, phi[i]);
            if (clip && a && fabs(y) - a[i] > 1e-13) { ci = i + 1; y = NAN; w = NAN; break; }
        }
        y_out[r] = y; w_out[r] = w;
        if (clip_idx) clip_idx[r] = ci;
    }
}

/* ------------------------------------------------------------------------------------
 * Transfer matrix -- src/TransferMatrix.jl:1-17.  2x2 matrices are column-major
 * [m11 m21 m12 m22] exactly as Julia's Matrix{Float64} memory.
 * ---------------------------------------------------------------------------------- */
static void mm2(const double *A, const double *B, double *C)
{   /* generic 2x2 matmul as Julia's matmul2x2!: C[i,j] = A[i,1]*B[1,j] + A[i,2]*B[2,j] */
    double c11 = A[0] * B[0] + A[2] * B[1];
    double c21 = A[1] * B[0] + A[3] * B[1];
    double c12 = A[0] * B[2] + A[2] * B[3];
    double c22 = A[1] * B[2] + A[3] * B[3];
    C[0] = c11; C[1] = c21; C[2] = c12; C[3] = c22;
}

/* TransferMatrix(lens) -- :1-6: prod over i = k..1 (left fold): ((M_k*M_{k-1})*...)*M_1 */
ORC_API void orc_transfer_matrix(int k, const double *tau, const double *phi, double *M)
{
    double acc[4], Mi[4];
    for (int i = k - 1; i >= 0; i--) {
        Mi[0] = 1.0; Mi[1] = -phi[i]; Mi[2] = tau[i]; Mi[3] = 1.0 - tau[i] * phi[i];   /* :4 */
        if (i == k - 1) memcpy(acc, Mi, sizeof acc);
        else { double tmp[4]; mm2(acc, Mi, tmp); memcpy(acc, tmp, sizeof acc); }
    }
    memcpy(M, acc, sizeof acc);
}

/* extend(M, tau, taup) = [1 taup; 0 1] * M * [1 tau; 0 1] -- :8 (left-assoc product) */
ORC_API void orc_extend(const double *M, double tau, double taup, double *E)
{
    double L[4] = {1.0, 0.0, taup, 1.0}, Rm[4] = {1.0, 0.0, tau, 1.0}, T[4];
    mm2(L, M, T);
    mm2(T, Rm, E);
}

/* transfer(M, v, tau, taup) = extend(...) * v -- :10 */
ORC_API void orc_transfer(const double *M, double tau, double taup, const double *v, double *out)
{
    double E[4]; orc_extend(M, tau, taup, E);
    out[0] = E[0] * v[0] + E[2] * v[1];
    out[1] = E[1] * v[0] + E[3] * v[1];
}

/* reverse_transfer(M, v, taup, tau) = extend(M, tau, taup) \ v -- :13.  Julia's `\` on a
 * square dense matrix is LU with partial pivoting (after triangular checks that never
 * trigger for a system matrix with phi != 0); restated for 2x2. */
static void solve2(const double *E, const double *v, double *out)
{
    double a11 = E[0], a21 = E[1], a12 = E[2], a22 = E[3], b1 = v[0], b2 = v[1];
    if (a21 == 0.0) {            /* upper triangular: back substitution */
        double x2 = b2 / a22; out[1] = x2; out[0] = (b1 - a12 * x2) / a11; return;
    }
    if (a12 == 0.0) {            /* lower triangular: forward substitution */
        double x1 = b1 / a11; out[0] = x1; out[1] = (b2 - a21 * x1) / a22; return;
    }
    if (fabs(a21) > fabs(a11)) { /* pivot: swap rows */
        double t;
        t = a11; a11 = a21; a21 = t; t = a12; a12 = a22; a22 = t; t = b1; b1 = b2; b2 = t;
    }
    double l = a21 / a11;
    double u22 = a22 - l * a12;
    double y2 = b2 - l * b1;
    double x2 = y2 / u22;
    double x1 = (b1 - a12 * x2) / a11;
    out[0] = x1; out[1] = x2;
}
ORC_API void orc_reverse_transfer(const double *M, double taup, double tau, const double *v,
                                  double *out)
{
    double E[4]; orc_extend(M, tau, taup, E);
    solve2(E, v, out);
}

ORC_API void orc_transfer_batch(const double *M, double tau, double taup, int reverse,
                                int64_t N, const double *v_in, double *v_out, int threads)
{
    double E[4]; orc_extend(M, tau, taup, E);
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel for schedule(static)
#endif
    for (int64_t r = 0; r < N; r++) {
        if (reverse) solve2(E, v_in + 2 * r, v_out + 2 * r);
        else {
            double a = v_in[2 * r], b = v_in[2 * r + 1];
            v_out[2 * r] = E[0] * a + E[2] * b;
            v_out[2 * r + 1] = E[1] * a + E[3] * b;
        }
    }
}

/* ------------------------------------------------------------------------------------
 * 2-D meridional real-ray trace -- src/RayTracing.jl:75-103, 145-173
 * ---------------------------------------------------------------------------------- */

/* sag(y,U,R,K,p) with p == zero -- :75-88 */
static double sag2d(int row, double y, double U, double R, double K, unsigned *flags)
{
    if (isfinite(R)) {
        double beta = R - y * tan(U);
        double y2 = y * y;
        double sec = 1.0 / cos(U);
        double D = beta * beta - y2 * (sec * sec + K);
        if (D >= 0.0) return y2 / (beta + jl_sign(R) * sqrt(D)) + poly_eval(row, y);   /* + p(y) :82 */
        if (D < 0.0) *flags |= F_MISS;
        return NAN;
    }
    return 0.0;
}

/* raytrace(surfaces, y, U, RealRay; K, p) -- :145-169.
 * aspheric = 0: the AbstractMatrix / Layout{Spherical} method (K forced to zeros, p === zero
 *               -> asin(tilt(y,R)) branch, :162 and :101).
 * aspheric = 1: the Layout{Aspheric} method (:171-173): K from the layout and, because its
 *               p holds Polynomial(zero) which is not === zero, ALWAYS atan(tilt(y,R,K,p)) (:98).
 * rt is rows x 2 column-major [y U]; ts gets the sag-corrected thicknesses (rows). */
ORC_API unsigned orc_trace2d(int rows, const double *R, const double *t, const double *n,
                             const double *K, int aspheric, double y, double U,
                             double *rt, double *ts)
{
    unsigned flags = 0;
    for (int i = 0; i < rows; i++) ts[i] = t[i];
    rt[0] = y; rt[rows] = U;
    for (int i = 0; i + 1 < rows; i++) {
        y += tan(U) * ts[i];                                   /* :152 */
        double Rs = R[i + 1];
        double Ks = aspheric ? K[i + 1] : 0.0;
        double s = sag2d(i + 1, y, U, Rs, Ks, &flags);         /* :156 */
        y += s * tan(U);                                       /* :158 */
        ts[i] += s; ts[i + 1] -= s;                            /* :160-161 */
        double theta;
        /* iszero(Ks) && ps === zero  :162.  A Layout{Aspheric} fills p with Polynomial(zero), which is not === zero
         * (src/Types.jl:27, 91), so the choice is per layout: every surface of it takes atan, K = 0 spheres and
         * planes included. */
        if (!aspheric) {
            double q = y / Rs;                                 /* tilt(y,R) :101 */
            if (fabs(q) > 1.0) flags |= F_DOMAIN;              /* Julia asin throws */
            theta = asin(q);
        } else {
            double D = Rs * Rs - y * y * (1.0 + Ks);           /* tilt(y,R,K,p) :98 */
            if (D < 0.0) flags |= F_DOMAIN;                    /* Julia sqrt throws */
            theta = atan(jl_sign(Rs) * y / sqrt(D) + poly_dpdy(i + 1, y));   /* + dp_dy(p, y) :98 */
        }
        double sin_ip = n[i] * sin(U + theta) / n[i + 1];      /* :163 */
        if (fabs(sin_ip) <= 1.0) U = asin(sin_ip) - theta;     /* :164 */
        else { if (fabs(sin_ip) > 1.0) flags |= F_TIR; U = NAN; }
        rt[i + 1] = y; rt[rows + i + 1] = U;
    }
    return flags;
}

/* Batched form: y_out / U_out are rows x N column-major-per-ray? No: laid out [surface][ray]
 * (ray index fastest) so the GPU writes are coalesced; ts likewise.  Any pointer may be NULL. */
ORC_API void orc_trace2d_batch(int rows, const double *R, const double *t, const double *n,
                               const double *K, int aspheric, int64_t N,
                               const double *y0, const double *U0,
                               double *y_out, double *U_out, double *ts_out, uint8_t *flags_out,
                               int threads)
{
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel
#endif
    {
        double *rt = (double *)malloc(sizeof(double) * 3 * rows);
        double *ts = rt + 2 * rows;
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
        for (int64_t r = 0; r < N; r++) {
            unsigned f = orc_trace2d(rows, R, t, n, K, aspheric, y0[r], U0[r], rt, ts);
            for (int i = 0; i < rows; i++) {
                if (y_out) y_out[(int64_t)i * N + r] = rt[i];
                if (U_out) U_out[(int64_t)i * N + r] = rt[rows + i];
                if (ts_out) ts_out[(int64_t)i * N + r] = ts[i];
            }
            if (flags_out) flags_out[r] = (uint8_t)f;
        }
        free(rt);
    }
}

/* ------------------------------------------------------------------------------------
 * 3-D skew real-ray trace -- src/PupilSampling.jl:1-65
 * ---------------------------------------------------------------------------------- */

/* sag(y,x,u,v,R,K,p), p == zero -- :1-14 */
static inline double sag3d(int row, double y, double x, double u, double v, double R, double K,
                           unsigned *flags)
{
    if (isfinite(R)) {
        double beta = R - y * u - x * v;                        /* :3 */
        double r2 = x * x + y * y;                              /* :4 */
        double D = beta * beta - r2 * (1.0 + K + u * u + v * v);/* :5 */
        if (D >= 0.0) return r2 / (beta + jl_sign(R) * sqrt(D)) + poly_eval(row, y);   /* :7 (+ p(y)) */
        if (D < 0.0) *flags |= F_MISS;
        return NAN;                                             /* :9 */
    }
    return 0.0;                                                 /* :12 */
}

/* One ray through the whole prescription.  u, v are SLOPES (the reference's tan(U), tan(V),
 * :38-39 -- the caller applies tan so this routine is trig-free).  K may be NULL (zeros).
 * xv, yv: rows-1 entries each (may be NULL); kout: final direction cosines [kx ky kz] (may be NULL).
 * Returns flag bits. */
ORC_API unsigned orc_trace3d(int rows, const double *R, const double *t, const double *n,
                             const double *K, double y, double x, double u, double v,
                             double *xv, double *yv, double *kout)
{
    unsigned flags = 0;
    /* k = normalize!([v, u, 1.0]) :40-41.  LinearAlgebra.generic_norm2 (n < 32): sequential
     * sum of squares then sqrt; __normalize! multiplies by inv(nrm). */
    double k1 = v, k2 = u, k3 = 1.0;
    {
        double nrm = sqrt(k1 * k1 + k2 * k2 + k3 * k3);
        double inv = 1.0 / nrm;
        k1 *= inv; k2 *= inv; k3 *= inv;
    }
    double s_prev = 0.0; int have_prev = 0;
    for (int i = 0; i + 1 < rows; i++) {
        /* ts = copy(t); ts[i] was decremented by the previous sag (:55) */
        double ti = have_prev ? t[i] - s_prev : t[i];
        y += u * ti;                                            /* :46 */
        x += v * ti;                                            /* :47 */
        double Rs = R[i + 1], Ks = K ? K[i + 1] : 0.0;
        double s = sag3d(i + 1, y, x, u, v, Rs, Ks, &flags);    /* :51 */
        y += s * u;                                             /* :52 */
        x += s * v;                                             /* :53 */
        s_prev = s; have_prev = 1;                              /* :54-55 */
        /* m = normalize!([tilt(y,x,R,K,p); -1.0]) :16-19, :56-57; tilt returns (x-, y-) order */
        double D = Rs * Rs - (x * x + y * y) * (1.0 + Ks);      /* :17 */
        if (D < 0.0) flags |= F_DOMAIN;                         /* Julia sqrt would throw */
        double sq = sqrt(D);
        double m1 = jl_sign(Rs) * x / sq + poly_dpdy(i + 1, x);  /* :18, + dp_dy(p, x) */
        double m2 = jl_sign(Rs) * y / sq + poly_dpdy(i + 1, y);
        double m3 = -1.0;
        {
            double nrm = sqrt(m1 * m1 + m2 * m2 + m3 * m3);
            double inv = 1.0 / nrm;
            m1 *= inv; m2 *= inv; m3 *= inv;
        }
        /* refract!(k, m, n1, n2) :21-32.  k . m is a BLAS ddot on 3 elements in the reference;
         * OpenBLAS' scalar tail is dot = 0; dot += y[i]*x[i] (FMA use inside it is unknowable). */
        double eta = n[i] / n[i + 1];                           /* :22 */
        double dot = 0.0 + k1 * m1; dot += k2 * m2; dot += k3 * m3;
        double gam = -dot;                                      /* :23 */
        double Dr = 1.0 - eta * eta * (1.0 - gam * gam);        /* :24 */
        if (Dr >= 0.0) {
            double c = eta * gam - sqrt(Dr);                    /* :26 */
            k1 = eta * k1 + c * m1;
            k2 = eta * k2 + c * m2;
            k3 = eta * k3 + c * m3;
        } else if (Dr < 0.0) {
            flags |= F_TIR;     /* :27-30: returns NaN, k unchanged; caller ignores it (:58) */
        }
        u = k2 / k3;                                            /* :59 */
        v = k1 / k3;                                            /* :60 */
        if (xv) xv[i] = x;
        if (yv) yv[i] = y;
    }
    if (kout) { kout[0] = k1; kout[1] = k2; kout[2] = k3; }
    return flags;
}

/* Batch of arbitrary rays; outputs laid out [surface][ray] (ray fastest); kout is [3][N]. */
ORC_API void orc_trace3d_batch(int rows, const double *R, const double *t, const double *n,
                               const double *K, int64_t N, const double *y0, const double *x0,
                               const double *u0, const double *v0,
                               double *xv, double *yv, double *kout, uint8_t *flags_out,
                               int threads)
{
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel
#endif
    {
        double *bx = (double *)malloc(sizeof(double) * 2 * rows);
        double *by = bx + rows;
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
        for (int64_t r = 0; r < N; r++) {
            double kk[3];
            unsigned f = orc_trace3d(rows, R, t, n, K, y0[r], x0[r], u0[r], v0[r], bx, by, kk);
            for (int i = 0; i + 1 < rows; i++) {
                if (xv) xv[(int64_t)i * N + r] = bx[i];
                if (yv) yv[(int64_t)i * N + r] = by[i];
            }
            if (kout) { kout[r] = kk[0]; kout[N + r] = kk[1]; kout[2 * N + r] = kk[2]; }
            if (flags_out) flags_out[r] = (uint8_t)f;
        }
        free(bx);
    }
}


/* ------------------------------------------------------------------------------------
 * Extended-precision (x87 long double, 64-bit mantissa) evaluation of the same 3-D trace
 * (src/PupilSampling.jl:34-65).  NOT a restatement of the reference's rounding: it is the
 * "truth" used by tests to tell ill-conditioned rays (where the reference's own Float64
 * result is uncertain at the 1e-12 level) from kernel error.
 * ---------------------------------------------------------------------------------- */
ORC_API void orc_trace3d_ld(int rows, const double *R, const double *t, const double *n,
                            const double *K, double y0, double x0, double u0, double v0,
                            double *xv, double *yv, double *kout)
{
    long double y = y0, x = x0, u = u0, v = v0;
    long double k1 = v, k2 = u, k3 = 1.0L;
    { long double inv = 1.0L / sqrtl(k1 * k1 + k2 * k2 + k3 * k3); k1 *= inv; k2 *= inv; k3 *= inv; }
    long double s_prev = 0.0L;
    for (int i = 0; i + 1 < rows; i++) {
        long double ti = (long double)t[i] - s_prev;
        y += u * ti; x += v * ti;
        long double Rs = R[i + 1], Ks = K ? K[i + 1] : 0.0, s;
        if (isfinite(R[i + 1])) {
            long double beta = Rs - y * u - x * v, r2 = x * x + y * y;
            long double D = beta * beta - r2 * (1.0L + Ks + u * u + v * v);
            s = (D >= 0.0L) ? r2 / (beta + (long double)jl_sign(R[i + 1]) * sqrtl(D)) : (long double)NAN;
        } else s = 0.0L;
        y += s * u; x += s * v; s_prev = s;
        long double m1, m2, m3 = -1.0L;
        if (isfinite(R[i + 1])) {
            long double sq = sqrtl(Rs * Rs - (x * x + y * y) * (1.0L + Ks));
            m1 = (long double)jl_sign(R[i + 1]) * x / sq; m2 = (long double)jl_sign(R[i + 1]) * y / sq;
        } else { m1 = (x != x) ? x : 0.0L; m2 = (y != y) ? y : 0.0L; }
        { long double inv = 1.0L / sqrtl(m1 * m1 + m2 * m2 + m3 * m3); m1 *= inv; m2 *= inv; m3 *= inv; }
        long double eta = (long double)n[i] / (long double)n[i + 1];
        long double gam = -(k1 * m1 + k2 * m2 + k3 * m3);
        long double Dr = 1.0L - eta * eta * (1.0L - gam * gam);
        if (Dr >= 0.0L) {
            long double c = eta * gam - sqrtl(Dr);
            k1 = eta * k1 + c * m1; k2 = eta * k2 + c * m2; k3 = eta * k3 + c * m3;
        }
        u = k2 / k3; v = k1 / k3;
        if (xv) xv[i] = (double)x;
        if (yv) yv[i] = (double)y;
    }
    if (kout) { kout[0] = (double)k1; kout[1] = (double)k2; kout[2] = (double)k3; }
}

ORC_API void orc_trace3d_ld_batch(int rows, const double *R, const double *t, const double *n,
                                  const double *K, int64_t N, const double *y0, const double *x0,
                                  const double *u0, const double *v0, double *xv, double *yv,
                                  double *kout)
{
    double *bx = (double *)malloc(sizeof(double) * 2 * rows), *by = bx + rows;
    for (int64_t r = 0; r < N; r++) {
        double kk[3];
        orc_trace3d_ld(rows, R, t, n, K, y0[r], x0[r], u0[r], v0[r], bx, by, kk);
        for (int i = 0; i + 1 < rows; i++) { xv[(int64_t)i * N + r] = bx[i]; yv[(int64_t)i * N + r] = by[i]; }
        if (kout) { kout[r] = kk[0]; kout[N + r] = kk[1]; kout[2 * N + r] = kk[2]; }
    }
    free(bx);
}

/* ------------------------------------------------------------------------------------
 * Pupil grid driver -- src/PupilSampling.jl:115-138 (the hot loop).
 *
 * The caller has already done :85-114: appended the image plane [Inf 0 1] (K = 0) and set
 * t[end-1] = focus, so (R,t,n,K) here are the EXTENDED surfaces.  ys (ny) and xs (nx) are
 * collect(range(y1,y2,k)) and collect(range(0,y_EP,k/2)) (:121-122); loop order y outer,
 * x inner (:123).  mode 0 = System (collimated, slopes u,v given: u = tan(U), v = tan(0));
 * mode 1 = RayBasis (:124-127): U = (ybar - y)/z0, V = -x/z0, then u = tan(U), v = tan(V).
 * stop is the reference's 1-based system.stop (index into xv/yv).
 *
 * Full-grid outputs (any may be NULL): ex = xf, ey = yf - h', r = hypot at stop, theta =
 * atan(y_s, x_s), mask = 1 where the ray is KEPT (:132), flags = ORT_FLAG_* bits.
 * Returns the number kept.
 * ---------------------------------------------------------------------------------- */
ORC_API int64_t orc_grid_trace(int rows, const double *R, const double *t, const double *n,
                               const double *K, int mode, double u_in, double v_in,
                               double ybar, double z0, double h_prime,
                               int ny, const double *ys, int nx, const double *xs,
                               int stop, double a_stop,
                               double *ex, double *ey, double *r, double *theta,
                               uint8_t *mask, uint8_t *flags_out, int threads)
{
    int64_t kept = 0;
    int nsurf = rows - 1;
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel reduction(+ : kept)
#endif
    {
        double *bx = (double *)malloc(sizeof(double) * 2 * rows);
        double *by = bx + rows;
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
        for (int iy = 0; iy < ny; iy++) {
            for (int ix = 0; ix < nx; ix++) {
                int64_t idx = (int64_t)iy * nx + ix;
                double yi = ys[iy], xi = xs[ix];
                double u = u_in, v = v_in;
                if (mode == 1) {                       /* :124-127 then tan at :38-39 */
                    double U = (ybar - yi) / z0;
                    double V = -xi / z0;
                    u = tan(U); v = tan(V);
                }
                unsigned f = orc_trace3d(rows, R, t, n, K, yi, xi, u, v, bx, by, NULL);
                double xf = bx[nsurf - 1], yf = by[nsurf - 1];           /* :129-130 */
                double xs_ = bx[stop - 1], ys_ = by[stop - 1];
                double ri = orc_hypot(xs_, ys_);                         /* :131 */
                int drop = (ri > a_stop) || isnan(xf) || isnan(yf);      /* :132 */
                if (ri > a_stop) f |= F_CLIP;
                if (ex) ex[idx] = xf;                                    /* :135 */
                if (ey) ey[idx] = yf - h_prime;                          /* :134 */
                if (r) r[idx] = ri;                                      /* :136 */
                if (theta) theta[idx] = atan2(ys_, xs_);                 /* :133 */
                if (mask) mask[idx] = (uint8_t)!drop;
                if (flags_out) flags_out[idx] = (uint8_t)f;
                kept += !drop;
            }
        }
        free(bx);
    }
    return kept;
}


/* ------------------------------------------------------------------------------------
 * EXTENSION (no reference counterpart -- SURVEY.md section 8 rows f3/f4, "parity unpinned"):
 * the same 3-D trace (src/PupilSampling.jl:34-65, identical operations for x, y, k) that also
 *   - accumulates the optical path length  OPL = sum_i n[i] * dz_i / k3_i, where dz_i = ts[i] is
 *     the sag-corrected z-advance of leg i (:54-55) and k3 the z direction cosine on that leg;
 *   - tests every surface's clear aperture: hypot(x, y) > a[i] sets F_VIGN (the reference's real-ray
 *     tracer only tests the stop radius, :131-132; its paraxial tracer clips at every surface, :135).
 * opl0 is the start term (distance from the reference wavefront / object point to the start point).
 * If rr != 0 the OPL is closed on a reference sphere of radius rr centred at (xc, yc) on the last
 * plane: tau = -b - sign(rr) sqrt(b^2 - (|q|^2 - rr^2)), q = P - C, b = q.k;  OPL += n_last * tau.
 * Returns flags; *opl_out = OPL (NaN if the ray is NaN).
 * ---------------------------------------------------------------------------------- */
#define F_VIGN 16u
ORC_API unsigned orc_trace3d_ext(int rows, const double *R, const double *t, const double *n,
                                 const double *K, const double *a, double y, double x, double u, double v,
                                 double opl0, double xc, double yc, double rr,
                                 double *xv, double *yv, double *kout, double *opl_out)
{
    unsigned flags = 0;
    double k1 = v, k2 = u, k3 = 1.0;
    {
        double nrm = sqrt(k1 * k1 + k2 * k2 + k3 * k3);
        double inv = 1.0 / nrm;
        k1 *= inv; k2 *= inv; k3 *= inv;
    }
    double opl = opl0;
    double s_prev = 0.0; int have_prev = 0;
    for (int i = 0; i + 1 < rows; i++) {
        double ti = have_prev ? t[i] - s_prev : t[i];
        y += u * ti;
        x += v * ti;
        double Rs = R[i + 1], Ks = K ? K[i + 1] : 0.0;
        double s = sag3d(i + 1, y, x, u, v, Rs, Ks, &flags);
        y += s * u;
        x += s * v;
        s_prev = s; have_prev = 1;
        opl += n[i] * (ti + s) / k3;                             /* extension: OPL of leg i */
        if (a && orc_hypot(x, y) > a[i]) flags |= F_VIGN;        /* extension: clear aperture of surface i+1 */
        double D = Rs * Rs - (x * x + y * y) * (1.0 + Ks);
        if (D < 0.0) flags |= F_DOMAIN;
        double sq = sqrt(D);
        double m1 = jl_sign(Rs) * x / sq + poly_dpdy(i + 1, x);
        double m2 = jl_sign(Rs) * y / sq + poly_dpdy(i + 1, y);
        double m3 = -1.0;
        {
            double nrm = sqrt(m1 * m1 + m2 * m2 + m3 * m3);
            double inv = 1.0 / nrm;
            m1 *= inv; m2 *= inv; m3 *= inv;
        }
        double eta = n[i] / n[i + 1];
        double dot = 0.0 + k1 * m1; dot += k2 * m2; dot += k3 * m3;
        double gam = -dot;
        double Dr = 1.0 - eta * eta * (1.0 - gam * gam);
        if (Dr >= 0.0) {
            double c = eta * gam - sqrt(Dr);
            k1 = eta * k1 + c * m1;
            k2 = eta * k2 + c * m2;
            k3 = eta * k3 + c * m3;
        } else if (Dr < 0.0) flags |= F_TIR;
        u = k2 / k3;
        v = k1 / k3;
        if (xv) xv[i] = x;
        if (yv) yv[i] = y;
    }
    if (rr != 0.0) {                                             /* close on the reference sphere */
        double qx = x - xc, qy = y - yc;
        double b = qx * k1 + qy * k2;
        double cq = qx * qx + qy * qy - rr * rr;
        double tau = -b - jl_sign(rr) * sqrt(b * b - cq);
        opl += n[rows - 1] * tau;
    }
    if (kout) { kout[0] = k1; kout[1] = k2; kout[2] = k3; }
    if (opl_out) *opl_out = opl;
    return flags;
}

/* 80-bit evaluation of the same extension: "truth" for the OPL/OPD tolerance checks */
ORC_API void orc_trace3d_ext_ld(int rows, const double *R, const double *t, const double *n,
                                const double *K, double y0, double x0, double u0, double v0,
                                double opl0, double xc, double yc, double rr, double *opl_out)
{
    long double y = y0, x = x0, u = u0, v = v0, k1 = v, k2 = u, k3 = 1.0L, opl = opl0, s_prev = 0.0L;
    { long double inv = 1.0L / sqrtl(k1 * k1 + k2 * k2 + k3 * k3); k1 *= inv; k2 *= inv; k3 *= inv; }
    for (int i = 0; i + 1 < rows; i++) {
        long double ti = (long double)t[i] - s_prev;
        y += u * ti; x += v * ti;
        long double Rs = R[i + 1], Ks = K ? K[i + 1] : 0.0, s;
        if (isfinite(R[i + 1])) {
            long double beta = Rs - y * u - x * v, r2 = x * x + y * y;
            long double D = beta * beta - r2 * (1.0L + Ks + u * u + v * v);
            s = (D >= 0.0L) ? r2 / (beta + (long double)jl_sign(R[i + 1]) * sqrtl(D)) : (long double)NAN;
        } else s = 0.0L;
        y += s * u; x += s * v; s_prev = s;
        opl += (long double)n[i] * (ti + s) / k3;
        long double m1, m2, m3 = -1.0L;
        if (isfinite(R[i + 1])) {
            long double sq = sqrtl(Rs * Rs - (x * x + y * y) * (1.0L + Ks));
            m1 = (long double)jl_sign(R[i + 1]) * x / sq; m2 = (long double)jl_sign(R[i + 1]) * y / sq;
        } else { m1 = (x != x) ? x : 0.0L; m2 = (y != y) ? y : 0.0L; }
        { long double inv = 1.0L / sqrtl(m1 * m1 + m2 * m2 + m3 * m3); m1 *= inv; m2 *= inv; m3 *= inv; }
        long double eta = (long double)n[i] / (long double)n[i + 1];
        long double gam = -(k1 * m1 + k2 * m2 + k3 * m3);
        long double Dr = 1.0L - eta * eta * (1.0L - gam * gam);
        if (Dr >= 0.0L) {
            long double c = eta * gam - sqrtl(Dr);
            k1 = eta * k1 + c * m1; k2 = eta * k2 + c * m2; k3 = eta * k3 + c * m3;
        }
        u = k2 / k3; v = k1 / k3;
    }
    if (rr != 0.0) {
        long double qx = x - xc, qy = y - yc, b = qx * k1 + qy * k2, cq = qx * qx + qy * qy - (long double)rr * rr;
        opl += (long double)n[rows - 1] * (-b - (long double)jl_sign(rr) * sqrtl(b * b - cq));
    }
    *opl_out = (double)opl;
}

/* start term of the OPL: mode 0 (collimated): n0 (x k1 + y k2) -- the distance by which the start
 * point (x, y, 0) is ahead of the plane wavefront through the origin; mode 1 (object point at z0):
 * n0 (-z0) / k3.  k = normalize([v, u, 1]) exactly as :40-41. */
ORC_API double orc_opl_start(int mode, double n0, double y, double x, double u, double v, double z0)
{
    double k1 = v, k2 = u, k3 = 1.0;
    double nrm = sqrt(k1 * k1 + k2 * k2 + k3 * k3);
    double inv = 1.0 / nrm;
    k1 *= inv; k2 *= inv; k3 *= inv;
    if (mode == 1) return n0 * (-z0) / k3;
    return n0 * (x * k1 + y * k2);
}

/* Grid form of the extension: like orc_grid_trace plus per-surface apertures (a may be NULL), OPD
 * output  opd = (OPL - opl_ref) * opd_scale  and its mask semantics: kept = !(stop clip || vignetted
 * || NaN).  opd may be NULL. */
ORC_API int64_t orc_grid_trace_ext(int rows, const double *R, const double *t, const double *n,
                                   const double *K, const double *a, int mode, double u_in, double v_in,
                                   double ybar, double z0, double h_prime,
                                   double xc, double yc, double rr, double opl_ref, double opd_scale,
                                   int ny, const double *ys, int nx, const double *xs,
                                   int stop, double a_stop,
                                   double *ex, double *ey, double *opd, uint8_t *mask, uint8_t *flags_out,
                                   int threads)
{
    int64_t kept = 0;
    int nsurf = rows - 1;
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel reduction(+ : kept)
#endif
    {
        double *bx = (double *)malloc(sizeof(double) * 2 * rows);
        double *by = bx + rows;
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
        for (int iy = 0; iy < ny; iy++) {
            for (int ix = 0; ix < nx; ix++) {
                int64_t idx = (int64_t)iy * nx + ix;
                double yi = ys[iy], xi = xs[ix];
                double u = u_in, v = v_in;
                if (mode == 1) { u = tan((ybar - yi) / z0); v = tan(-xi / z0); }
                double opl0 = orc_opl_start(mode, n[0], yi, xi, u, v, z0), opl;
                unsigned f = orc_trace3d_ext(rows, R, t, n, K, a, yi, xi, u, v, opl0, xc, yc, rr, bx, by, NULL, &opl);
                double xf = bx[nsurf - 1], yf = by[nsurf - 1];
                double ri = orc_hypot(bx[stop - 1], by[stop - 1]);
                if (ri > a_stop) f |= F_CLIP;
                int drop = (ri > a_stop) || (f & F_VIGN) || isnan(xf) || isnan(yf);
                if (ex) ex[idx] = xf;
                if (ey) ey[idx] = yf - h_prime;
                if (opd) opd[idx] = (opl - opl_ref) * opd_scale;
                if (mask) mask[idx] = (uint8_t)!drop;
                if (flags_out) flags_out[idx] = (uint8_t)f;
                kept += !drop;
            }
        }
        free(bx);
    }
    return kept;
}


/* ------------------------------------------------------------------------------------
 * First-order solve + Seidel aberration sums of ONE prescription (SURVEY.md section 8 f2): what the
 * reference's optimize() evaluates per candidate (src/Optimization.jl:32-45).  Restates
 *   Lens(surfaces)                 src/RayTracing.jl:38-53
 *   trace_marginal_ray(lens, a)    src/RayTracing.jl:208-221   (y = 1, w = 0; stop = argmin a./y)
 *   trace_chief_ray(lens, ...)     src/RayTracing.jl:246-263   (y = 0, w = 1 basis ray)
 *   aberrations(surfaces, system, lambda, dn)   src/SeidelAberrations.jl:6-53
 * out[16] = f, EBFD, stop, H, W040, W131, W222, W220P, W311, W020, W111, W220, W220M, W220T,
 *           marginal nu[end], chief nu[1].   per[7][k] (optional): spherical, coma, astigmatism,
 * petzval, distortion, axial, lateral per surface.  dn may be NULL (zeros).  k = rows - 1 surfaces
 * (the prescription's last thickness must be 0 or Inf, as solve() requires).
 * ---------------------------------------------------------------------------------- */
ORC_API int orc_seidel(int rows, const double *R, const double *t, const double *n, const double *a,
                       double h_prime, double lambda, const double *dn, double *out, double *per)
{
    int k = rows - 1;
    if (k < 1 || k > 126) return -1;
    double tau[128], phi[128];
    if (orc_lens(rows, R, t, n, tau, phi) != k) return -2;
    /* pass 1: basis rays (1, 0) and (0, 1); stop = argmin a[i] / y[i] */
    double y1[129], w1[129], y2[129], w2[129];
    y1[0] = 1.0; w1[0] = 0.0; y2[0] = 0.0; w2[0] = 1.0;
    for (int i = 0; i < k; i++) {
        y1[i + 1] = px_transfer(y1[i], w1[i], tau[i]); w1[i + 1] = px_refract(y1[i + 1], w1[i], phi[i]);
        y2[i + 1] = px_transfer(y2[i], w2[i], tau[i]); w2[i + 1] = px_refract(y2[i + 1], w2[i], phi[i]);
    }
    double f = -(1.0 / w1[k]);                                   /* f = -inv(w[end])   :213 */
    double EBFD = y1[k] * f;
    int stop = 1; double s = a[0] / y1[1];
    for (int i = 1; i < k; i++) { double v = a[i] / y1[i + 1]; if (v < s) { s = v; stop = i + 1; } }   /* findmin :215-216 */
    /* marginal_ray *= s (:217); n extended by n[end] (Types.jl:39) */
    double ym[130], num[130], nx[130];
    for (int i = 0; i <= k; i++) { ym[i] = y1[i] * s; num[i] = w1[i] * s; }
    for (int i = 0; i < rows; i++) nx[i] = n[i];
    nx[rows] = n[rows - 1];
    double y_stop = ym[stop], y2_stop = y2[stop];
    double nub = -num[k] * h_prime / ym[1];                      /* :256  (marginal.nu[end] = extended row = num[k]) */
    double H = nub * ym[0];                                      /* _solve :316 */
    double W[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int i = 1; i <= k; i++) {                               /* surface i: row i+1 of the layout */
        double Ri = R[i];
        double y = ym[i];
        double yb = nub * (y2[i] - ym[i] * y2_stop / y_stop);    /* chief.y at surface i  :258 */
        double nu = num[i - 1], ni = nx[i - 1], ni1 = nx[i];
        double u0 = num[i - 1] / nx[i - 1], u1 = num[i] / nx[i];
        double A = nu + ni * y / Ri;                             /* SeidelAberrations.jl:17 */
        double Ab = (H + A * yb) / y;                            /* :18 */
        double yD = y * (u1 / ni1 - u0 / ni);                    /* :19, Delta :4 */
        double d0 = dn ? dn[i - 1] : 0.0, d1 = dn ? dn[i] : 0.0;
        double yd = y * (d1 / ni1 - d0 / ni);                    /* :20 */
        double in1 = 1.0 / ni1, in0 = 1.0 / ni;
        double Dn2 = in1 * in1 - in0 * in0;                      /* :21 */
        double P = (in1 - in0) / Ri;                             /* :22 */
        double sph = -(A * A) * yD / (8 * lambda);               /* :24 */
        double coma = -A * Ab * yD / (2 * lambda);               /* :25 */
        double ast = -(Ab * Ab) * yD / (2 * lambda);             /* :26 */
        double ptz = -(H * H) * P / (4 * lambda);                /* :27 */
        double dist = -Ab * (Ab * Ab * y * Dn2 - (H + Ab * y) * yb * P) / (2 * lambda);   /* :29 */
        double ax = A * yd / (2 * lambda);                       /* :30 */
        double lat = Ab * yd / lambda;                           /* :31 */
        double v[7] = {sph, coma, ast, ptz, dist, ax, lat};
        for (int j = 0; j < 7; j++) { W[j] += v[j]; if (per) per[j * k + (i - 1)] = v[j]; }
    }
    out[0] = f; out[1] = EBFD; out[2] = (double)stop; out[3] = H;
    out[4] = W[0]; out[5] = W[1]; out[6] = W[2]; out[7] = W[3]; out[8] = W[4]; out[9] = W[5]; out[10] = W[6];
    out[11] = W[3] + 0.5 * W[2]; out[12] = W[3] + W[2]; out[13] = W[3] + 1.5 * W[2];     /* :41-43 */
    out[14] = num[k]; out[15] = nub;
    return 0;
}

ORC_API void orc_seidel_candidates(int rows, int64_t C, const double *RtnK, const double *a, double h_prime,
                                   double lambda, const double *dn, double *out, int threads)
{
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel for schedule(static)
#endif
    for (int64_t c = 0; c < C; c++) {
        const double *Rc = RtnK + c * 4 * rows;
        if (orc_seidel(rows, Rc, Rc + rows, Rc + 2 * rows, a, h_prime, lambda, dn, out + 16 * c, NULL) != 0)
            for (int j = 0; j < 16; j++) out[16 * c + j] = NAN;
    }
}

/* Ordered compaction: the reference's push! order (:134-137).  Returns count. */
ORC_API int64_t orc_compact(int64_t N, const uint8_t *mask, const double *in, double *out)
{
    int64_t c = 0;
    for (int64_t i = 0; i < N; i++) if (mask[i]) out[c++] = in[i];
    return c;
}

/* Julia Base pairwise sum (mapreduce_impl, blksize 1024) -- used by sigma :171-172.
 * The base case in Julia is an @simd loop whose lane order is CPU-dependent; restated
 * sequentially (last-ulp differences vs real Julia are unknowable). */
static double pairwise_sum(const double *a, int64_t lo, int64_t hi /* inclusive */)
{
    if (lo == hi) return a[lo];
    if (hi - lo < 1024) {
        double v = a[lo] + a[lo + 1];
        for (int64_t i = lo + 2; i <= hi; i++) v += a[i];
        return v;
    }
    int64_t mid = lo + ((hi - lo) >> 1);
    return pairwise_sum(a, lo, mid) + pairwise_sum(a, mid + 1, hi);
}
ORC_API double orc_sum(int64_t n, const double *a) { return n > 0 ? pairwise_sum(a, 0, n - 1) : 0.0; }

/* sigma(ex, ey) -- src/PupilSampling.jl:169-173 (two-pass, pairwise sums) */
ORC_API double orc_sigma(int64_t n, const double *ex, const double *ey)
{
    if (n <= 0) return NAN;
    double mux = orc_sum(n, ex) / (double)n, muy = orc_sum(n, ey) / (double)n;
    double *d = (double *)malloc(sizeof(double) * (size_t)n);
    for (int64_t i = 0; i < n; i++) { double q = ex[i] - mux; d[i] = q * q; }
    double sx = orc_sum(n, d);
    for (int64_t i = 0; i < n; i++) { double q = ey[i] - muy; d[i] = q * q; }
    double sy = orc_sum(n, d);
    free(d);
    return sqrt((sx + sy) / (double)n);
}

/* Symmetry + statistics -- src/PupilSampling.jl:139-146.  Inputs are the n compacted
 * half-pupil vectors; outputs hold 2n entries each:
 *   ey2 = [ey; ey], ex2 = [ex; -ex], rho2 = [r; r]/maximum(r), th2 = [theta; pi .- theta].
 * Returns RMS = sigma(ex2, ey2). */
ORC_API double orc_mirror_stats(int64_t n, const double *ex, const double *ey, const double *r,
                                const double *theta, double *ex2, double *ey2, double *rho2,
                                double *th2)
{
    double rmax = -INFINITY;
    for (int64_t i = 0; i < n; i++) if (r[i] > rmax) rmax = r[i];   /* maximum(r) */
    for (int64_t i = 0; i < n; i++) {
        ey2[i] = ey[i]; ey2[n + i] = ey[i];                /* :140 */
        ex2[i] = ex[i]; ex2[n + i] = -ex[i];               /* :141 */
        double rho = r[i] / rmax;                          /* :142 */
        rho2[i] = rho; rho2[n + i] = rho;                  /* :143 */
        th2[i] = theta[i]; th2[n + i] = M_PI - theta[i];   /* :144 */
    }
    return orc_sigma(2 * n, ex2, ey2);                     /* :146 */
}

/* wavegrad -- src/PupilSampling.jl:165-167: eps * nu / lambda (left-assoc: (eps*nu)/lambda) */
ORC_API void orc_wavegrad(int64_t n, const double *e, double nu, double lambda, double *out)
{
    for (int64_t i = 0; i < n; i++) out[i] = e[i] * nu / lambda;
}

/* Candidate-batched merit (BASELINE config 5; no reference counterpart -- a synthetic batch of
 * the 3-D tracer): C prescriptions, each rows x 4 [R t n K] stored as RtnK[c][4][rows]; fixed
 * full-pupil entrance grid ys (ny) x xs (nx); per candidate: n_kept, mean_x, mean_y, RMS about
 * the centroid (two-pass). out is C x 4 doubles. */
ORC_API void orc_candidates(int rows, int64_t C, const double *RtnK, double u, double v,
                            double h_prime, int ny, const double *ys, int nx, const double *xs,
                            int stop, double a_stop, double *out, int threads)
{
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#pragma omp parallel
#endif
    {
        int64_t NN = (int64_t)ny * nx;
        double *bx = (double *)malloc(sizeof(double) * (2 * rows + 2 * NN));
        double *by = bx + rows, *kx = by + rows, *ky = kx + NN;
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 16)
#endif
        for (int64_t c = 0; c < C; c++) {
            const double *Rc = RtnK + c * 4 * rows, *tc = Rc + rows, *nc = tc + rows, *Kc = nc + rows;
            int64_t m = 0;
            for (int iy = 0; iy < ny; iy++)
                for (int ix = 0; ix < nx; ix++) {
                    orc_trace3d(rows, Rc, tc, nc, Kc, ys[iy], xs[ix], u, v, bx, by, NULL);
                    double xf = bx[rows - 2], yf = by[rows - 2];
                    double ri = orc_hypot(bx[stop - 1], by[stop - 1]);
                    if ((ri > a_stop) || isnan(xf) || isnan(yf)) continue;
                    kx[m] = xf; ky[m] = yf - h_prime; m++;
                }
            double *o = out + 4 * c;
            o[0] = (double)m;
            if (m == 0) { o[1] = o[2] = o[3] = NAN; continue; }
            o[1] = orc_sum(m, kx) / (double)m;
            o[2] = orc_sum(m, ky) / (double)m;
            o[3] = orc_sigma(m, kx, ky);
        }
        free(bx);
    }
}

ORC_API int orc_max_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
