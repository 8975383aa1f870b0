// kern_first_order.cu -- the batched 2-D meridional real-ray trace (K2), the paraxial y-nu trace
// (K3), the transfer-matrix apply (K4) and the FP64 peak microbenchmark (sm_100a).
#include <stdlib.h>

#include "kern.cuh"

// ------------------------------------------------------------------------------------------
// K2: raytrace(surfaces, y, U, RealRay)  src/RayTracing.jl:145-173 (sag :75-88, tilt :98-101)
// One thread per ray.  The arithmetic keeps the reference's order (never contracted); tan / cos /
// asin / sin / atan are CUDA's double-precision libm (<= 2 ulp; Julia's own libm differs in the
// last ulp too), so parity here is 1e-12 relative, not bit-exact.
// ------------------------------------------------------------------------------------------
// one iteration of the surface loop of src/RayTracing.jl:151-167; returns ts[i] (:160).
// `aspheric` selects the method: 0 = AbstractMatrix / Layout{Spherical} (K forced to 0, asin(tilt(y, R)) :162, :101),
// 1 = Layout{Aspheric} (K from the layout, atan(tilt(y, R, K, p)) on EVERY surface, :98, :171-173).  The reference tests
// iszero(Ks) && ps === zero, and a Layout{Aspheric} holds Polynomial(zero) in p, which is not === zero (src/Types.jl:27,
// 91), so the branch is chosen per layout, never per surface.  `pc` is non-null only with aspheric = 1.
template <class SurfT>
__device__ __forceinline__ double trace2d_step(const SurfT& S, int aspheric, double& y, double& U, double& sprev,
                                               unsigned& flags, const double* pc = nullptr, int npoly = 0)
{
    const double tU = tan(U);
    const double ti = SS(S.t, sprev);                        // ts[i] (:148, :161)
    y = SA(y, SM(tU, ti));                                   // :152
    const double Ks = aspheric ? S.K : 0.0;
    double sg;
    if (isfinite(S.R)) {                                     // sag :75-88
        double beta = SS(S.R, SM(y, tU));
        double y2 = SM(y, y);
        double sec = SD(1.0, cos(U));
        double D = SS(SM(beta, beta), SM(y2, SA(SM(sec, sec), Ks)));
        if (D >= 0.0) sg = SA(SD(y2, SA(beta, SM(S.sgnR, SQ(D)))), pc ? poly_eval(pc, npoly, y) : 0.0);       // + p(y) :82
        else { if (D < 0.0) flags |= ORT_FLAG_MISS; sg = CUDART_NAN; }
    } else sg = 0.0;
    y = SA(y, SM(sg, tU));                                   // :158
    sprev = sg;                                              // ts[i+1] -= s :161
    double theta;
    if (!aspheric) {                                         // asin(tilt(y, R))  :162, :101
        double q = SD(y, S.R);
        if (fabs(q) > 1.0) flags |= ORT_FLAG_DOMAIN;
        theta = asin(q);
    } else {                                                 // atan(tilt(y, R, K, p))  :98
        double D2 = SS(SM(S.R, S.R), SM(SM(y, y), SA(1.0, Ks)));
        if (D2 < 0.0) flags |= ORT_FLAG_DOMAIN;
        theta = atan(SA(SD(SM(S.sgnR, y), SQ(D2)), pc ? poly_dpdy(pc, npoly, y) : 0.0));                     // + dp_dy(p, y) :98
    }
    const double sin_ip = SD(SM(S.n1, sin(SA(U, theta))), S.n2);   // :163
    if (fabs(sin_ip) <= 1.0) U = SS(asin(sin_ip), theta);          // :164
    else { if (fabs(sin_ip) > 1.0) flags |= ORT_FLAG_TIR; U = CUDART_NAN; }
    return SA(ti, sg);                                       // ts[i] += s  :160
}

__global__ void __launch_bounds__(256)
k_trace2d(const __grid_constant__ Presc P, Trace2dArgs A)
{
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= A.N) return;
    const long long N = A.N;
    double y = A.y0[i], U = A.U0[i];
    unsigned flags = 0;
    double sprev = 0.0;
    if (A.y_out) A.y_out[i] = y;
    if (A.U_out) A.U_out[i] = U;
    const int nsurf = P.nsurf;
    for (int s = 0; s < nsurf; s++) {
        const double ts = trace2d_step(P.s[s], A.aspheric, y, U, sprev, flags,     // the caller's layout type
                                       (A.aspheric && P.poly) ? P.poly + (size_t)s * P.npoly : nullptr, P.npoly);
        if (A.ts_out) A.ts_out[(size_t)s * N + i] = ts;
        if (A.y_out) A.y_out[(size_t)(s + 1) * N + i] = y;
        if (A.U_out) A.U_out[(size_t)(s + 1) * N + i] = U;
    }
    if (A.ts_out) A.ts_out[(size_t)nsurf * N + i] = SS(P.t_last, sprev);
    if (A.flags) A.flags[i] = (uint8_t)flags;
}

// ------------------------------------------------------------------------------------------
// Ray aiming on the device (SURVEY.md section 8 f1): the secant loops of trace_marginal_ray / trace_chief_ray
// (src/RayTracing.jl:223-240, 265-296; stop_loss :117-125) and of the edge-ray search
// (src/PupilSampling.jl:67-83), one thread per solve, every function evaluation = a 2-D trace to the stop.
// ------------------------------------------------------------------------------------------
// The two root finders of the prelude, generic over the function evaluation `f(x)` = height at the stop surface of the
// meridional ray parametrised by x (a functor: prescription in the constant bank for k_aim2d, in the candidate's RtnK
// block for k_aim_candidates).  Returns the iteration count, negative when the iteration left the domain.
//   secant_reference: x <- x - f eps / (f(x + eps) - f) until |f| <= tol, eps = sqrt(eps())   (src/RayTracing.jl:229-233, 282-286)
//   secant_polish:    same step with a relative eps, run to the rounding floor (the roots of the reference's BFGS-on-abs,
//                     src/PupilSampling.jl:67-83)
template <class F>
__device__ __forceinline__ int secant_reference(F f, double& x, double tgt, double tol, bool* finite = nullptr)
{
    const double eps = 1.4901161193847656e-08;                 // sqrt(eps())  src/RayTracing.jl:1
    int it = 0;
    double v = SS(f(x), tgt);
    while (fabs(v) > tol) {                                     // :229, :282
        if (++it > 100 || !isfinite(v)) return -(it + 1);
        const double ve = SS(f(SA(x, eps)), tgt);
        x = SS(x, SD(SM(v, eps), SS(ve, v)));                   // :231, :284
        v = SS(f(x), tgt);
    }
    if (finite) *finite = isfinite(v);      // a NaN height ends the reference's `while abs(f) > atol` too (no error there)
    return it;
}

template <class F>
__device__ __forceinline__ int secant_polish(F f, double& x, double tgt, double scale)
{
    const double eps = 1.4901161193847656e-08;
    double v_prev = 0.0;
    int it = 0;
    for (;; it++) {
        if (it >= 60) break;
        const double h = SM(eps, fmax(1.0, fabs(x)));
        const double v = SS(f(x), tgt);
        const double vh = SS(f(SA(x, h)), tgt);
        if (!isfinite(v)) return -(it + 1);
        bool done = fabs(v) <= SM(4e-16, scale);
        if (it > 0) done = done || (fabs(v) >= fabs(v_prev) && fabs(v_prev) <= SM(1e-13, scale));
        if (done) break;
        x = SS(x, SD(SM(v, h), SS(vh, v)));
        v_prev = v;
    }
    return it;
}

// The same two iterations with the two function evaluations of a step -- f(x) and f(x + eps) -- taken SIDE BY SIDE by the two
// lanes of a pair (even lane: x, odd lane: x + eps; one shuffle each way).  Same operations on the same operands, so the
// same bits and the same iteration counts as the one-thread forms; the chain of serial 2-D traces is half as long (the
// f(x + eps) of the last step is wasted).  The loop is warp-uniform: pairs that have converged idle until the last one has.
// Every lane of the warp must call these together.
template <class F>
__device__ __forceinline__ int secant_reference_pair(F f, double& x, double tgt, double tol, bool* finite, int odd)
{
    const double eps = 1.4901161193847656e-08;                 // sqrt(eps())  src/RayTracing.jl:1
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    int it = 0, ret = 0;
    bool active = true;
    double val = SS(f(odd ? SA(x, eps) : x), tgt);
    double v = __shfl_sync(full, val, lane & ~1), ve = __shfl_sync(full, val, lane | 1);
    for (;;) {
        bool go = active && fabs(v) > tol;                      // :229, :282
        if (go && (++it > 100 || !isfinite(v))) { ret = -(it + 1); active = false; go = false; }
        if (active && !go) { active = false; ret = it; if (finite) *finite = isfinite(v); }
        if (!__any_sync(full, go)) break;
        if (go) {
            x = SS(x, SD(SM(v, eps), SS(ve, v)));               // :231, :284
            val = SS(f(odd ? SA(x, eps) : x), tgt);
            active = true;
        }
        v = __shfl_sync(full, val, lane & ~1); ve = __shfl_sync(full, val, lane | 1);
    }
    return ret;
}

template <class F>
__device__ __forceinline__ int secant_polish_pair(F f, double& x, double tgt, double scale, int odd)
{
    const double eps = 1.4901161193847656e-08;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    double v_prev = 0.0;
    int it = 0, ret = 0;
    bool active = true;
    for (;;) {
        if (active && it >= 60) { active = false; ret = it; }
        if (!__any_sync(full, active)) break;
        const double h = SM(eps, fmax(1.0, fabs(x)));
        double val = 0.0;
        if (active) val = SS(f(odd ? SA(x, h) : x), tgt);
        const double v = __shfl_sync(full, val, lane & ~1), vh = __shfl_sync(full, val, lane | 1);
        if (active) {
            if (!isfinite(v)) { active = false; ret = -(it + 1); }
            else {
                bool done = fabs(v) <= SM(4e-16, scale);
                if (it > 0) done = done || (fabs(v) >= fabs(v_prev) && fabs(v_prev) <= SM(1e-13, scale));
                if (done) { active = false; ret = it; }
                else { x = SS(x, SD(SM(v, h), SS(vh, v))); v_prev = v; it++; }
            }
        }
    }
    return ret;
}

__device__ __forceinline__ double aim_eval(const Presc& P, const AimArgs& A, double x, double other)
{
    double y = A.vary_u ? other : x, U = A.vary_u ? x : other, sprev = 0.0;
    unsigned flags = 0;
    for (int s = 0; s < A.stop; s++)                       // aspheric: the layout type of the system being aimed
        trace2d_step(P.s[s], A.aspheric, y, U, sprev, flags, (A.aspheric && P.poly) ? P.poly + (size_t)s * P.npoly : nullptr, P.npoly);
    return y;
}

__global__ void __launch_bounds__(64)
k_aim2d(const __grid_constant__ Presc P, AimArgs A)
{
    const long long j = (long long)blockIdx.x * 64 + threadIdx.x;
    if (j >= A.N) return;
    double x = A.x0[j];
    const double other = A.other[j], tgt = A.target[j];
    auto f = [&](double xx) { return aim_eval(P, A, xx, other); };
    const int it = (A.mode == 0) ? secant_reference(f, x, tgt, A.tol) : secant_polish(f, x, tgt, A.tol);
    A.x_out[j] = x;
    if (A.iters) A.iters[j] = it;
}

// ------------------------------------------------------------------------------------------
// K3: raytrace(lens, y, w, a; clip)  src/RayTracing.jl:127-143 with transfer/refract :55-69.
// 4 rays per thread, row loop in convergent control flow so the Lens rows are read through the
// uniform datapath (constant bank -> uniform registers) once per row for all 4 rays.
// STRICT = reference order (mul, add: never contracted); FAST = DFMA.  32 B of HBM traffic per ray
// (+4 B with clip indices): FAST is HBM-bound, STRICT sits at the FP64-issue / HBM crossover.
// Clip test `abs(y) - a[i] > 1e-13` (:135): an integer pre-filter on the exponent/mantissa high
// word skips the exact FP64 test for rays that are not within 2^-19 of the aperture edge.
// ------------------------------------------------------------------------------------------
#ifndef PX_RPT
#define PX_RPT 4
#endif
// The one-argument form of __launch_bounds__ on purpose: with a minimum-blocks argument (whatever its value) ptxas feeds the
// per-row constants through predicated LDC loads into vector registers instead of uniform registers, +30 % kernel time.
#if defined(PX_MINB)
#define PX_BOUNDS __launch_bounds__(256, PX_MINB)
#else
#define PX_BOUNDS __launch_bounds__(256)
#endif

// Clip test of :135 for final-only output (no per-row table), one FFMA + one SHF per ray and row plus one shared FMNMX,
// all off the FP64 pipe (which the 2 DFMA per ray and row already keep ~75 % busy):
//   The high word of a double, read as a float, orders like |y| itself (IEEE bit patterns of positive numbers are
//   monotonic), and FP32 instructions take |.| for free.  Per row the host prepares S = 1 / ulp_float(T) and M = T S for
//   T = float(high word of a[row]): z = fma(|hf|, S, -M) is then EXACTLY the distance k = hi(|y|) - hi(a) in high-word units
//   (2^-20 relative) whenever |y| is near the aperture.  k <= -1 means |y| < a (not clipped), k >= 2 means
//   |y| - a > a 2^-21 > 1e-13 (clipped; rows with a <= 2.2e-7 take the exact path), k in {0, 1} is undecided.
//     sign(z) goes into a 32-row bit mask with one funnel shift  -> first row with k >= 0 by clz at the end of the chunk
//     amb = min(amb, |z|) over all rows and the thread's rays     -> amb < 1.5 iff some |k| <= 1 occurred
//   A thread with an undecided row (or a non-finite ray) re-traces its rays from the inputs with the exact FP64 test --
//   same arithmetic, so the same values: a few threads in a million.  A clipped ray simply keeps running; its outputs
//   are NaN (:136) and its clip row is the first mask bit.
struct ParaxOne { double y, w; int ci; };
template <int ARITH>
__device__ __noinline__ ParaxOne paraxial_exact_clip(const LensK& L, double yy, double ww)
{
    const int k = L.k;
    int c = 0;
    for (int row = 0; row < k; row++) {
        const double tau = L.tau[row], phi = L.phi[row];
        if (isfinite(tau)) yy = (ARITH == ORT_ARITH_STRICT) ? SA(yy, SM(ww, tau)) : fma(ww, tau, yy);   // :62
        ww = (ARITH == ORT_ARITH_STRICT) ? SS(ww, SM(yy, phi)) : fma(-yy, phi, ww);                      // :67
        if (c == 0 && SS(fabs(yy), L.a[row]) > 1e-13) c = row + 1;                                      // :135
    }
    ParaxOne o; o.y = yy; o.w = ww; o.ci = c;
    return o;
}

template <int ARITH, bool TABLE, bool CLIP>
__global__ void PX_BOUNDS
k_paraxial(const __grid_constant__ LensK L, ParaxArgs A)
{
    // Persistent CTAs, tile-strided, with a software prefetch: the loads of tile k+1 are issued before the
    // 40-row arithmetic of tile k, so HBM latency hides behind the FP64 work instead of in front of it.
    const long long N = A.N;
    const long long per = 256 * PX_RPT;
    const long long ntiles = (N + per - 1) / per;
    const int k = L.k;
    constexpr bool MASKCLIP = CLIP && !TABLE;
    double yn[PX_RPT], wn[PX_RPT];
    long long tile = blockIdx.x;
    if (tile < ntiles) {
#pragma unroll
        for (int j = 0; j < PX_RPT; j++) {
            const long long i = min(tile * per + (long long)j * 256 + threadIdx.x, N - 1);
            yn[j] = __ldcs(A.y0 + i); wn[j] = __ldcs(A.w0 + i);
        }
    }
    for (; tile < ntiles; tile += gridDim.x) {
        double y[PX_RPT], w[PX_RPT];
        int ci[PX_RPT];
        long long idx[PX_RPT];
        bool valid[PX_RPT];
#pragma unroll
        for (int j = 0; j < PX_RPT; j++) {
            const long long i = tile * per + (long long)j * 256 + threadIdx.x;
            valid[j] = i < N;
            idx[j] = valid[j] ? i : N - 1;           // padded lanes redo the last ray: warp stays convergent
            y[j] = yn[j]; w[j] = wn[j];
            ci[j] = 0;
        }
        const long long nxt = tile + gridDim.x;
        if (nxt < ntiles) {                          // prefetch the next tile of this CTA
#pragma unroll
            for (int j = 0; j < PX_RPT; j++) {
                const long long i = min(nxt * per + (long long)j * 256 + threadIdx.x, N - 1);
                yn[j] = __ldcs(A.y0 + i); wn[j] = __ldcs(A.w0 + i);
            }
        }
        if (TABLE) {
#pragma unroll
            for (int j = 0; j < PX_RPT; j++) {
                if (!valid[j]) continue;
                if (A.y_all) A.y_all[idx[j]] = y[j];
                if (A.w_all) A.w_all[idx[j]] = w[j];
            }
        }
        if (MASKCLIP) {
            float amb = 4.0f;
            unsigned msk[PX_RPT];
#pragma unroll
            for (int j = 0; j < PX_RPT; j++) msk[j] = 0xFFFFFFFFu;
            // one flat row loop (the shape ptxas unrolls and feeds from uniform registers); the 32-row mask is folded
            // into the clip row in a uniform branch every 32nd row and once behind the loop
#define PX_FOLD(BASE, C)                                                                                      \
            {                                                                                                 \
                const unsigned live = ((C) == 32) ? 0xFFFFFFFFu : ((1u << (C)) - 1u);                         \
                _Pragma("unroll") for (int j = 0; j < PX_RPT; j++) {                                          \
                    const unsigned over = ~msk[j] & live;     /* bit (C - 1 - i): row BASE + i had k >= 0 */  \
                    if (ci[j] == 0 && over) ci[j] = (BASE) + (C) - 31 + __clz(over);                          \
                    msk[j] = 0xFFFFFFFFu;                                                                     \
                }                                                                                             \
            }
#pragma unroll 4
            for (int row = 0; row < k; row++) {
                const double tau = L.tau[row], phi = L.phi[row];
                const float2 csm = L.csm[row]; const float cs = csm.x, ncm = csm.y;
                const bool fin = isfinite(tau);                      // uniform (:62)
                if (fin) {
#pragma unroll
                    for (int j = 0; j < PX_RPT; j++)
                        y[j] = (ARITH == ORT_ARITH_STRICT) ? SA(y[j], SM(w[j], tau)) : fma(w[j], tau, y[j]);
                }
#pragma unroll
                for (int j = 0; j < PX_RPT; j++) {
                    w[j] = (ARITH == ORT_ARITH_STRICT) ? SS(w[j], SM(y[j], phi)) : fma(-y[j], phi, w[j]);   // :67
                    const float z = fmaf(fabsf(__int_as_float(__double2hiint(y[j]))), cs, ncm);
                    msk[j] = __funnelshift_l(__float_as_uint(z), msk[j], 1);
                    amb = fminf(amb, fabsf(z));
                }
                if ((row & 31) == 31) PX_FOLD(row - 31, 32)
            }
            if (k & 31) PX_FOLD(k & ~31, k & 31)
#undef PX_FOLD
            bool slow = !(amb >= 1.5f);
#pragma unroll
            for (int j = 0; j < PX_RPT; j++) slow = slow || !isfinite(y[j]) || !isfinite(w[j]);
            if (slow) {
#pragma unroll
                for (int j = 0; j < PX_RPT; j++) {
                    const ParaxOne o = paraxial_exact_clip<ARITH>(L, A.y0[idx[j]], A.w0[idx[j]]);
                    y[j] = o.y; w[j] = o.w; ci[j] = o.ci;
                }
            }
        } else {
        for (int row = 0; row < k; row++) {
            const double tau = L.tau[row], phi = L.phi[row];
            const bool fin = isfinite(tau);                  // uniform (:62)
            const double a = CLIP ? L.a[row] : 0.0;
            const int a_hi = CLIP ? (__double2hiint(a) - 1) : 0;
            if (fin) {                                       // uniform branch, not a per-ray select
#pragma unroll
                for (int j = 0; j < PX_RPT; j++)
                    y[j] = (ARITH == ORT_ARITH_STRICT) ? SA(y[j], SM(w[j], tau)) : fma(w[j], tau, y[j]);   // :62
            }
#pragma unroll
            for (int j = 0; j < PX_RPT; j++)
                w[j] = (ARITH == ORT_ARITH_STRICT) ? SS(w[j], SM(y[j], phi)) : fma(-y[j], phi, w[j]);       // :67
            if (CLIP) {
                // (table output) One integer pre-filter for the thread's rays: only if some |y| >= a (1 - 2^-20) by high
                // word (or is NaN) run the exact test of :135.  A clipped ray continues as (0, 0) -- finite, so it never
                // re-enters the exact test -- and is written out as NaN (:136).
                int mx = 0;
#pragma unroll
                for (int j = 0; j < PX_RPT; j++) mx = max(mx, __double2hiint(y[j]) & 0x7FFFFFFF);
                if (mx >= a_hi) {
#pragma unroll
                    for (int j = 0; j < PX_RPT; j++)
                        if (ci[j] == 0 && SS(fabs(y[j]), a) > 1e-13) { ci[j] = row + 1; y[j] = 0.0; w[j] = 0.0; }
                }
            }
            if (TABLE) {
#pragma unroll
                for (int j = 0; j < PX_RPT; j++) {
                    if (!valid[j]) continue;                         // rt[i+1,:] (NaN after the clip row, :136)
                    if (A.y_all) A.y_all[(size_t)(row + 1) * N + idx[j]] = ci[j] ? CUDART_NAN : y[j];
                    if (A.w_all) A.w_all[(size_t)(row + 1) * N + idx[j]] = ci[j] ? CUDART_NAN : w[j];
                }
            }
        }
        }
#pragma unroll
        for (int j = 0; j < PX_RPT; j++) {
            if (!valid[j]) continue;
            if (A.y) __stcs(A.y + idx[j], ci[j] ? CUDART_NAN : y[j]);
            if (A.w) __stcs(A.w + idx[j], ci[j] ? CUDART_NAN : w[j]);
            if (A.clip_idx) A.clip_idx[idx[j]] = ci[j];
        }
    }
}

// ------------------------------------------------------------------------------------------
// K3, the streaming form: final (y, nu) only (no per-row table), every tau finite (Lens(surfaces) guarantees it:
// src/RayTracing.jl:42 zeroes an infinite t[1]), apertures "nice" (LensK::clip_nice).  Everything else runs k_paraxial above.
// ncu on k_paraxial showed the plain kernel issue-bound (82 % of the issue slots, 10.6 non-FP64 instructions per row for
// 8 DFMA) and the clip kernel latency-bound at 33 instructions per row.  Here a row of PX2_RPT rays costs 2 uniform loads +
// 2 PX2_RPT DFMA, plus per ray FADD + SHF + half an FMNMX3 when clipping:
//   hf = the high word of y read as a float, T[row] = the high word of a[row] read as a float (host): z = |hf| - T is the
//   distance between |y| and a in float ulps of T (= 2^-20-relative units of the doubles), exact when they are close.
//   sign(z) -> one bit of a 32-row mask per ray (funnel shift); amb = min |z| over rows and the thread's rays.
//   With U = the largest ulp(T[row]) (host, LensK::amb_thr = 1.5 U): amb >= 1.5 U means every |z| was at least two units,
//   i.e. every decision was clear of the 1e-13 threshold of :135 (k <= -2: |y| < a; k >= 2: |y| - a > a 2^-21 > 1e-13 for
//   a > 2.2e-7) and the first clear bit of the mask is the clip row.  Otherwise (a few threads in a million), or when a
//   ray went non-finite, the thread re-traces its rays with the exact FP64 test -- same arithmetic, same values.
// ------------------------------------------------------------------------------------------
// Rays per thread: 8 without the clip test (5.67 ms per 1e9 rays against 6.03 at 4: fewer warps, more loads in flight per
// thread), 4 with it (11.4 ms against 12.8 at 8; the clip kernel is bound by issue slots, not by HBM -- DESIGN.md section 3).
#ifndef PX2_RPT
#define PX2_RPT 8
#endif
#ifndef PX2_RPT_CLIP
#define PX2_RPT_CLIP 4
#endif
template <int ARITH, bool CLIP>
__global__ void __launch_bounds__(256)
k_paraxial_final(const __grid_constant__ LensK L, ParaxArgs A)
{
    constexpr int R = CLIP ? PX2_RPT_CLIP : PX2_RPT;
    const long long N = A.N;
    const long long per = 256 * R;
    const long long ntiles = (N + per - 1) / per;
    const int k = L.k;
    double yn[R], wn[R];
    long long tile = blockIdx.x;
    if (tile < ntiles) {
#pragma unroll
        for (int j = 0; j < R; j++) {
            const long long i = min(tile * per + (long long)j * 256 + threadIdx.x, N - 1);
            yn[j] = __ldcs(A.y0 + i); wn[j] = __ldcs(A.w0 + i);
        }
    }
    for (; tile < ntiles; tile += gridDim.x) {
        const long long i0 = tile * per + threadIdx.x;
        double y[R], w[R];
#pragma unroll
        for (int j = 0; j < R; j++) { y[j] = yn[j]; w[j] = wn[j]; }
        const long long nxt = tile + gridDim.x;
        if (nxt < ntiles) {                          // prefetch the next tile of this CTA behind this tile's arithmetic
#pragma unroll
            for (int j = 0; j < R; j++) {
                const long long i = min(nxt * per + (long long)j * 256 + threadIdx.x, N - 1);
                yn[j] = __ldcs(A.y0 + i); wn[j] = __ldcs(A.w0 + i);
            }
        }
        unsigned msk[R];
        int ci[R];
        float amb = CUDART_INF_F;
#pragma unroll
        for (int j = 0; j < R; j++) { msk[j] = 0xFFFFFFFFu; ci[j] = 0; }
#define PX2_ROW(ROWIDX)                                                                                              \
        {                                                                                                             \
            const double tau = L.tau[ROWIDX], phi = L.phi[ROWIDX];                                                    \
            const float tf = CLIP ? L.ctf[ROWIDX] : 0.0f;                                                             \
            _Pragma("unroll") for (int j = 0; j < R; j++) {                                                           \
                y[j] = (ARITH == ORT_ARITH_STRICT) ? SA(y[j], SM(w[j], tau)) : fma(w[j], tau, y[j]);     /* :62 */    \
                w[j] = (ARITH == ORT_ARITH_STRICT) ? SS(w[j], SM(y[j], phi)) : fma(-y[j], phi, w[j]);    /* :67 */    \
                if (CLIP) {                                                                                           \
                    const float z = fabsf(__int_as_float(__double2hiint(y[j]))) - tf;                                 \
                    msk[j] = __funnelshift_l(__float_as_uint(z), msk[j], 1);                                          \
                    amb = fminf(amb, fabsf(z));                                                                       \
                }                                                                                                     \
            }                                                                                                         \
        }
#define PX2_FOLD(BASE, C)                                                                                             \
        {                                                                                                             \
            const unsigned live = ((C) == 32) ? 0xFFFFFFFFu : ((1u << (C)) - 1u);                                     \
            _Pragma("unroll") for (int j = 0; j < R; j++) {                                                           \
                const unsigned over = ~msk[j] & live;         /* bit (C - 1 - i): |y| >= a at row BASE + i */          \
                if (ci[j] == 0 && over) ci[j] = (BASE) + (C) - 31 + __clz(over);                                      \
                msk[j] = 0xFFFFFFFFu;                                                                                 \
            }                                                                                                         \
        }
        if (CLIP) {
            int row = 0;
            for (; row + 32 <= k; row += 32) {
#pragma unroll 4
                for (int i = 0; i < 32; i++) PX2_ROW(row + i)
                PX2_FOLD(row, 32)
            }
            if (row < k) {
                const int c = k - row;
#pragma unroll 4
                for (int i = 0; i < c; i++) PX2_ROW(row + i)
                PX2_FOLD(row, c)
            }
            bool slow = !(amb >= L.amb_thr);
#pragma unroll
            for (int j = 0; j < R; j++) slow = slow || !isfinite(y[j]) || !isfinite(w[j]);
            if (slow) {
#pragma unroll
                for (int j = 0; j < R; j++) {
                    const long long i = min(i0 + (long long)j * 256, N - 1);
                    const ParaxOne o = paraxial_exact_clip<ARITH>(L, A.y0[i], A.w0[i]);
                    y[j] = o.y; w[j] = o.w; ci[j] = o.ci;
                }
            }
        } else {
#pragma unroll 4
            for (int row = 0; row < k; row++) PX2_ROW(row)
        }
#undef PX2_ROW
#undef PX2_FOLD
#pragma unroll
        for (int j = 0; j < R; j++) {
            const long long i = i0 + (long long)j * 256;
            if (i >= N) continue;
            if (A.y) __stcs(A.y + i, (CLIP && ci[j]) ? CUDART_NAN : y[j]);
            if (A.w) __stcs(A.w + i, (CLIP && ci[j]) ? CUDART_NAN : w[j]);
            if (A.clip_idx) __stcs(A.clip_idx + i, CLIP ? ci[j] : 0);      // 0 = not clipped (also without the clip test)
        }
    }
}

// ------------------------------------------------------------------------------------------
// K4: transfer(M, v, tau, taup) = extend(M, tau, taup) * v and reverse_transfer = extend \ v
// src/TransferMatrix.jl:8-17.  Pure HBM streaming: 16 B in, 16 B out per ray, 128-bit accesses.
// The reverse path restates the 2x2 partially pivoted LU that Julia's `\` performs.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 transfer_one(const TransferArgs& A, double2 v)
{
    const double a11 = A.E[0], a21 = A.E[1], a12 = A.E[2], a22 = A.E[3];
    double2 o;
    if (!A.reverse) {
        o.x = SA(SM(a11, v.x), SM(a12, v.y));
        o.y = SA(SM(a21, v.x), SM(a22, v.y));
    } else if (a21 == 0.0) {
        o.y = SD(v.y, a22); o.x = SD(SS(v.x, SM(a12, o.y)), a11);
    } else if (a12 == 0.0) {
        o.x = SD(v.x, a11); o.y = SD(SS(v.y, SM(a21, o.x)), a22);
    } else {
        double p11 = a11, p12 = a12, p21 = a21, p22 = a22, b1 = v.x, b2 = v.y;
        if (fabs(a21) > fabs(a11)) { p11 = a21; p12 = a22; p21 = a11; p22 = a12; b1 = v.y; b2 = v.x; }
        const double l = SD(p21, p11);
        const double u22 = SS(p22, SM(l, p12));
        const double y2 = SS(b2, SM(l, b1));
        o.y = SD(y2, u22);
        o.x = SD(SS(b1, SM(p12, o.y)), p11);
    }
    return o;
}

__global__ void __launch_bounds__(256) k_transfer(TransferArgs A)
{
    // grid-stride, 4 independent 128-bit loads in flight per thread
    const long long stride = (long long)gridDim.x * 256;
    long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    for (; i + 3 * stride < A.N; i += 4 * stride) {
        const double2 v0 = __ldcs(A.v_in + i), v1 = __ldcs(A.v_in + i + stride);
        const double2 v2 = __ldcs(A.v_in + i + 2 * stride), v3 = __ldcs(A.v_in + i + 3 * stride);
        __stcs(A.v_out + i, transfer_one(A, v0));
        __stcs(A.v_out + i + stride, transfer_one(A, v1));
        __stcs(A.v_out + i + 2 * stride, transfer_one(A, v2));
        __stcs(A.v_out + i + 3 * stride, transfer_one(A, v3));
    }
    for (; i < A.N; i += stride) __stcs(A.v_out + i, transfer_one(A, __ldcs(A.v_in + i)));
}

// ------------------------------------------------------------------------------------------
// First-order solve shared by the per-candidate kernels (k_seidel, k_vignetting, k_aim_candidates): Lens(surfaces)
// src/RayTracing.jl:38-53 and the two fundamental paraxial rays (1, 0) and (0, 1) traced together :55-69, :127-143,
// stop = argmin a ./ y and the marginal scale s :213-217.  Reference operation order throughout (never contracted),
// so every kernel that starts from it holds the same bits as the CPU restatement.
// ------------------------------------------------------------------------------------------
struct FirstOrder {
    double y1, w1, y2, w2;      // both rays after the last surface (unscaled)
    double s;                   // min a[i] / y[i]: scale of the marginal ray
    double ys1, ys2;            // both rays at the stop (unscaled)
    double yfirst;              // ray 1 at the first surface (unscaled)
    double zsum;                // cumsum of the real thicknesses t = tau .* n (Types.jl:41-46)
    int stop;                   // 1-based
};

// one Lens row: (tau, phi) of surface i+1 from the candidate's R, t, n
__device__ __forceinline__ void lens_row(const double* R, const double* t, const double* n, int i, double& tau, double& phi)
{
    double ti = t[i];
    if (i == 0 && !isfinite(ti)) ti = 0.0;                           // :42
    tau = SD(ti, n[i]);                                              // :43
    phi = SD(SS(n[i + 1], n[i]), R[i + 1]);                          // :45
}

// transfer(y, w, tau) then refract(y, w, phi) for both fundamental rays (:55-69)
__device__ __forceinline__ void lens_step(double tau, double phi, double& y1, double& w1, double& y2, double& w2)
{
    if (isfinite(tau)) { y1 = SA(y1, SM(w1, tau)); y2 = SA(y2, SM(w2, tau)); }     // :62
    w1 = SS(w1, SM(y1, phi)); w2 = SS(w2, SM(y2, phi));                            // :67
}

__device__ __forceinline__ FirstOrder first_order(const double* R, const double* t, const double* n, int k, const double* a)
{
    FirstOrder o;
    o.y1 = 1.0; o.w1 = 0.0; o.y2 = 0.0; o.w2 = 1.0;
    o.s = CUDART_INF; o.ys1 = o.ys2 = o.yfirst = o.zsum = 0.0; o.stop = 1;
    for (int i = 0; i < k; i++) {
        double tau, phi;
        lens_row(R, t, n, i, tau, phi);
        const double tz = SM(tau, n[i]);
        o.zsum = (i == 0) ? tz : SA(o.zsum, tz);
        lens_step(tau, phi, o.y1, o.w1, o.y2, o.w2);
        const double v = SD(a[i], o.y1);
        if (i == 0) o.yfirst = o.y1;
        if (i == 0 || v < o.s) { o.s = v; o.stop = i + 1; o.ys1 = o.y1; o.ys2 = o.y2; }     // findmin :215-216
    }
    return o;
}

// ------------------------------------------------------------------------------------------
// K7 (SURVEY.md section 8 f2): first-order solve + Seidel sums, one thread per candidate prescription.
// Lens(surfaces) src/RayTracing.jl:38-53; trace_marginal_ray(lens, a) :208-221; trace_chief_ray(lens, ...)
// :246-263; aberrations() src/SeidelAberrations.jl:6-53.  Two passes over the surfaces (the stop --
// argmin a./y, :215-216 -- must be known before the chief ray can be combined), no per-thread arrays:
// pass 2 recomputes the two basis rays with the same operations, hence the same bits.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_seidel(const __grid_constant__ SeidelArgs A)
{
    const long long c = (long long)blockIdx.x * 128 + threadIdx.x;
    if (c >= A.C) return;
    const int rows = A.rows, k = rows - 1;
    const double* R = A.RtnK + (size_t)c * 4 * rows;
    const double* t = R + rows;
    const double* n = t + rows;
    double* out = A.out + (size_t)c * ORT_SEIDEL_NOUT;
    const double tl = t[rows - 1];
    if (!(tl == 0.0 || !isfinite(tl))) {             // Lens() keeps the last row: solve() cannot use it
        for (int j = 0; j < ORT_SEIDEL_NOUT; j++) out[j] = CUDART_NAN;
        return;
    }
    // ---- pass 1
    const FirstOrder fo = first_order(R, t, n, k, A.a);
    double y1 = fo.y1, w1 = fo.w1, y2 = fo.y2, w2 = fo.w2;
    const double s = fo.s, ys1 = fo.ys1, ys2 = fo.ys2;
    const int stop = fo.stop;
    const double f = -SD(1.0, w1);                                   // :213
    const double EBFD = SM(y1, f);
    const double numk = SM(w1, s);                                   // marginal.nu[end]
    const double y_stop = SM(ys1, s), y2_stop = ys2;
    const double ym1 = SM(1.0, s);                                   // marginal.y[begin]: the start height 1.0 scaled by s (:217)
    // ---- pass 2
    y1 = 1.0; w1 = 0.0; y2 = 0.0; w2 = 1.0;
    double W[7] = {0, 0, 0, 0, 0, 0, 0};
    double nub = 0.0, H = 0.0;
    for (int i = 0; i < k; i++) {
        double tau, phi;
        lens_row(R, t, n, i, tau, phi);
        const double w1_prev = w1;
        lens_step(tau, phi, y1, w1, y2, w2);
        const double ym = SM(y1, s);                                 // marginal y at surface i+1
        if (i == 0) {
            nub = SD(SM(-numk, A.h_prime), ym);                      // :256  -marginal.nu[end] * h' / y[1]
            H = SM(nub, ym1);                                        // _solve :316  nu_bar * marginal.y[begin]
        }
        const double Ri = R[i + 1];
        const double ni = n[i], ni1 = (i + 1 < rows) ? n[i + 1] : n[rows - 1];
        const double yb = SM(nub, SS(y2, SD(SM(ym, y2_stop), y_stop)));               // :258
        const double nu = SM(w1_prev, s), nu1 = SM(w1, s);
        const double u0 = SD(nu, ni), u1 = SD(nu1, ni1);
        const double Aa = SA(nu, SD(SM(ni, ym), Ri));                                  // SeidelAberrations.jl:17
        const double Ab = SD(SA(H, SM(Aa, yb)), ym);                                   // :18
        const double yD = SM(ym, SS(SD(u1, ni1), SD(u0, ni)));                         // :19
        const double yd = SM(ym, SS(SD(A.dn[i + 1], ni1), SD(A.dn[i], ni)));           // :20
        const double in1 = SD(1.0, ni1), in0 = SD(1.0, ni);
        const double Dn2 = SS(SM(in1, in1), SM(in0, in0));                             // :21
        const double P = SD(SS(in1, in0), Ri);                                         // :22
        const double l8 = SM(8.0, A.lambda), l2 = SM(2.0, A.lambda), l4 = SM(4.0, A.lambda);
        double v[7];
        v[0] = SD(SM(-SM(Aa, Aa), yD), l8);                                            // :24
        v[1] = SD(SM(SM(-Aa, Ab), yD), l2);                                            // :25
        v[2] = SD(SM(-SM(Ab, Ab), yD), l2);                                            // :26
        v[3] = SD(SM(-SM(H, H), P), l4);                                               // :27
        v[4] = SD(SM(-Ab, SS(SM(SM(SM(Ab, Ab), ym), Dn2), SM(SM(SA(H, SM(Ab, ym)), yb), P))), l2);   // :29
        v[5] = SD(SM(Aa, yd), l2);                                                     // :30
        v[6] = SD(SM(Ab, yd), A.lambda);                                               // :31
#pragma unroll
        for (int j = 0; j < 7; j++) {
            W[j] = SA(W[j], v[j]);
            if (A.per) A.per[((size_t)c * 7 + j) * k + i] = v[j];
        }
    }
    out[0] = f; out[1] = EBFD; out[2] = (double)stop; out[3] = H;
    out[4] = W[0]; out[5] = W[1]; out[6] = W[2]; out[7] = W[3]; out[8] = W[4]; out[9] = W[5]; out[10] = W[6];
    out[11] = SA(W[3], SM(0.5, W[2])); out[12] = SA(W[3], W[2]); out[13] = SA(W[3], SM(1.5, W[2]));
    out[14] = numk; out[15] = nub;
}

// ------------------------------------------------------------------------------------------
// vignetting(system, a) per candidate (SURVEY.md section 8 f3; src/Vignetting.jl:1-30): semi-diameter table
// [a, limited = |y|, unvignetted = |y| + |ybar|, half = |ybar|, full = |ybar| - |y|] (the last two NaN where
// < |y|, :12-13), the three maximum fields of view (:20-26), and the limit / partial / full classification
// (:27-29) as a per-surface code.  Same two-pass first-order solve as k_seidel (bit-identical rays).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool jl_isapprox(double x, double y)
{   // isapprox(x, y): x == y || (isfinite(x) && isfinite(y) && |x - y| <= sqrt(eps) * max(|x|, |y|))
    if (x == y) return true;
    if (!isfinite(x) || !isfinite(y)) return false;
    return fabs(SS(x, y)) <= SM(1.4901161193847656e-08, fmax(fabs(x), fabs(y)));
}

__global__ void __launch_bounds__(128) k_vignetting(const __grid_constant__ VigArgs A)
{
    const long long c = (long long)blockIdx.x * 128 + threadIdx.x;
    if (c >= A.C) return;
    const int rows = A.rows, k = rows - 1;
    const double* R = A.RtnK + (size_t)c * 4 * rows;
    const double* t = R + rows;
    const double* n = t + rows;
    double* M = A.out + (size_t)c * (6 * k + ORT_VIG_TAIL);
    double* tail = M + 6 * k;
    const double tl = t[rows - 1];
    if (!(tl == 0.0 || !isfinite(tl))) {
        for (int j = 0; j < 6 * k + ORT_VIG_TAIL; j++) M[j] = CUDART_NAN;
        return;
    }
    // ---- pass 1: stop, scale, marginal nu[end]
    const FirstOrder fo = first_order(R, t, n, k, A.a_solve);
    double y1 = fo.y1, w1 = fo.w1, y2 = fo.y2, w2 = fo.w2;
    const double s = fo.s, ys1 = fo.ys1, ys2 = fo.ys2, yfirst = fo.yfirst;
    const int stop = fo.stop;
    const double f = -SD(1.0, w1);
    const double numk = SM(w1, s);
    const double nub = SD(SM(-numk, A.h_prime), SM(yfirst, s));
    const double y_stop = SM(ys1, s);
    // ---- pass 2: the table and the three minima
    y1 = 1.0; w1 = 0.0; y2 = 0.0; w2 = 1.0;
    double min_un = CUDART_INF, min_half = CUDART_INF, min_full = CUDART_INF;
    bool un = true, nan_un = false, nan_half = false, nan_full = false;
    for (int i = 0; i < k; i++) {
        double tau, phi;
        lens_row(R, t, n, i, tau, phi);
        lens_step(tau, phi, y1, w1, y2, w2);
        const double ym = SM(y1, s);
        const double yb = fabs(SM(nub, SS(y2, SD(SM(ym, ys2), y_stop))));     // |chief y|  (src/RayTracing.jl:258)
        const double y = fabs(ym);
        const double a = A.a_vig[i];
        const double unv = SA(y, yb);
        double half = yb, full = SS(yb, y);
        if (half < y) half = CUDART_NAN;                                       // :12
        if (full < y) full = CUDART_NAN;                                       // :13
        const bool a_unvig = a >= unv || jl_isapprox(a, unv);                  // :14
        un = un && a_unvig;
        const bool is_limit = a < y && !jl_isapprox(a, unv);                   // :27
        const bool is_full = a <= full;                                        // :28 (NaN compares false)
        const bool is_partial = !a_unvig && !is_full;                          // :29
        M[0 * k + i] = a; M[1 * k + i] = y; M[2 * k + i] = unv; M[3 * k + i] = half; M[4 * k + i] = full;
        M[5 * k + i] = (double)((is_limit ? 1 : 0) | (is_partial ? 2 : 0) | (is_full ? 4 : 0));
        // minimum(...) propagates NaN in Julia; fmin would drop it
        if (i != stop - 1) { const double q = SD(SS(a, y), yb); nan_un |= isnan(q); if (q < min_un) min_un = q; }   // :17
        { const double q = SD(a, yb); nan_half |= isnan(q); if (q < min_half) min_half = q; }                       // :18
        { const double q = SD(SA(a, y), yb); nan_full |= isnan(q); if (q < min_full) min_full = q; }                // :19
    }
    if (nan_un) min_un = CUDART_NAN;
    if (nan_half) min_half = CUDART_NAN;
    if (nan_full) min_full = CUDART_NAN;
    const double u0 = SD(nub, n[0]);                                           // chief.u[1] = nu_bar / n[1]
    const double mins[3] = {min_un, min_half, min_full};
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const double ub = fabs(SM(u0, mins[j]));                               // :22
        tail[3 * j + 0] = SM(2.0, SM(atan(ub), 57.29577951308232));            // 2 atand(u_bar)  :23
        tail[3 * j + 1] = ub;
        tail[3 * j + 2] = fabs(SM(A.h_prime, mins[j]));                        // chief.y[end] = h'  :25
    }
    tail[9] = un ? 1.0 : 0.0; tail[10] = (double)stop; tail[11] = f;
}

// ------------------------------------------------------------------------------------------
// Per-candidate prelude of full_trace (SURVEY.md section 8 f1, src/PupilSampling.jl:85-108): first-order solve
// (src/RayTracing.jl:208-221, 246-263), real chief ray traced backwards through the reversed prescription
// (:265-296), real marginal ray (:223-240), edge rays (src/PupilSampling.jl:67-83; the two roots of the
// reference's BFGS-on-abs, by secant).  One thread per candidate prescription; every function evaluation is
// a 2-D meridional trace with the surface rows read straight from the candidate's RtnK block.
// ------------------------------------------------------------------------------------------
struct Surf2 { double R, K, t, n1, n2, sgnR; };
struct CandView { const double *R, *t, *n, *K; int rows; double bfd; };

template <bool REV>
__device__ __forceinline__ Surf2 cand_surf(const CandView& V, int j)
{
    Surf2 S;
    if (!REV) { S.R = V.R[j + 1]; S.K = V.K[j + 1]; S.t = V.t[j]; S.n1 = V.n[j]; S.n2 = V.n[j + 1]; }
    else {      // rev_R = -[Inf; R[end:-1:2]], rev_t = t[end:-1:1] with rev_t[1] = BFD, reverse(K) (:267-274)
        const int r = V.rows - 1 - j;
        S.R = -V.R[r]; S.K = V.K[r - 1]; S.t = (j == 0) ? V.bfd : V.t[r]; S.n1 = V.n[r]; S.n2 = V.n[r - 1];
    }
    S.sgnR = (S.R < 0.0) ? -1.0 : ((S.R > 0.0) ? 1.0 : S.R);
    return S;
}

template <bool REV>
__device__ __noinline__ double cand_height(const CandView& V, int upto, int aspheric, double y, double U)
{
    double sprev = 0.0; unsigned fl = 0;
    for (int j = 0; j < upto; j++) { const Surf2 S = cand_surf<REV>(V, j); trace2d_step(S, aspheric, y, U, sprev, fl); }   // caller's flag
    return y;
}

// The prelude of one candidate is a chain of serial root finds, so the kernel is latency-bound (0.21 ms for 8192 candidates,
// 0.30 ms for 65 536 in the one-thread form).  Two splits shorten the chain.  (1) The two independent links run side by
// side in the two halves of a CTA: half 0 aims the chief ray (secant + the final reversed trace), half 1 the marginal
// ray; after one exchange through shared memory half 0 polishes the upper edge ray, half 1 the lower one.  (2) Inside a
// half, a PAIR of lanes works on one candidate: the two function evaluations of every secant step are taken side by side
// (secant_*_pair).  Every quantity is computed with the operations it always had, so the records are bit-identical to
// the one-thread-per-candidate form.
#define AIM_CPB 32                                       // candidates per CTA
#define AIM_PAIR_MAX_C 24576                             // populations up to this size take the lane-pair form
// PAIR = false: one lane per candidate and half (2 warps per CTA) -- half the work, twice the chain: the form for large
// populations, where the kernel is throughput-bound (65 536 candidates: 0.28 ms against 0.30 ms; 8192: 0.139 against 0.094).
template <bool PAIR>
__global__ void __launch_bounds__((PAIR ? 4 : 2) * AIM_CPB) k_aim_candidates(const __grid_constant__ AimCandArgs A)
{
    __shared__ double s_x[3][AIM_CPB];                   // Ubar, EP_t (half 0) | y_m (half 1)
    __shared__ double s_e2[AIM_CPB];
    __shared__ int s_st[2][AIM_CPB];
    const int role = threadIdx.x / ((PAIR ? 2 : 1) * AIM_CPB), odd = PAIR ? (threadIdx.x & 1) : 0;
    const int lane = PAIR ? ((threadIdx.x & (2 * AIM_CPB - 1)) >> 1) : (threadIdx.x & (AIM_CPB - 1));   // candidate within the CTA
    const long long craw = (long long)blockIdx.x * AIM_CPB + lane;
    const bool live = craw < A.C;
    const long long c = live ? craw : A.C - 1;           // idle lanes shadow the last candidate (no stores)
    const int rows = A.rows, k = rows - 1;
    CandView V;
    V.R = A.RtnK + (A.n_fields > 0 ? 0 : (size_t)c * 4 * rows);       // fields of one system share its prescription
    V.t = V.R + rows; V.n = V.t + rows; V.K = V.n + rows; V.rows = rows; V.bfd = 0.0;
    const double Hrel = A.n_fields > 0 ? A.Hs[c] : A.H;
    double* out = A.out + (size_t)c * ORT_AIM_NOUT;
    const double tl = V.t[rows - 1];
    const bool lastrow_ok = (tl == 0.0 || !isfinite(tl));             // else Lens() would keep the last row
    // ---- first-order solve: both fundamental rays (:209, :252), stop = argmin a ./ y (:215-216)  [both warps]
    const FirstOrder fo = first_order(V.R, V.t, V.n, k, A.a);
    const double y1 = fo.y1, w1 = fo.w1, w2 = fo.w2, s = fo.s, ys1 = fo.ys1, ys2 = fo.ys2, yfirst = fo.yfirst, zsum = fo.zsum;
    const int stop = fo.stop;
    const double f = -SD(1.0, w1);
    const double nlast = V.n[rows - 1];
    const double ymk = SM(y1, s), numk = SM(w1, s);                   // marginal (y, nu) after the last surface
    const double bfd = SS(SA(zsum, SD(-ymk, SD(numk, nlast))), zsum); // marginal.z[end] - marginal.z[end-1]  (Types.jl:44-46)
    const double nub = SD(SM(-numk, A.h_prime), SM(yfirst, s));       // :256
    const double nuck = SM(nub, SS(w2, SD(SM(numk, ys2), SM(ys1, s))));   // chief nu after the last surface :258
    V.bfd = bfd;
    const int stop_c = stop < 1 ? 1 : (stop > k ? k : stop);          // a degenerate solve must not index outside the prescription
    const double a_stop_signed = A.a[stop_c - 1];
    const double a_stop = fabs(a_stop_signed);
    const double tol = 1.4901161193847656e-08;
    int status = 0;
    bool fin = true;
    if (role == 0) {
        // ---- real chief ray, backwards (:265-296).  aspheric = 1 whatever A.aspheric: full_trace reaches trace_chief_ray with
        // a Layout (src/PupilSampling.jl:85), so the reversed system is always built as a Layout{Aspheric} (:272-277)
        const double ybp = A.h_prime;
        double ubp = -SD(nuck, nlast);
        const int rstop = rows - stop_c;
        auto fc = [&](double uu) { return cand_height<true>(V, rstop, 1, ybp, uu); };
        if ((PAIR ? secant_reference_pair(fc, ubp, 0.0, tol, &fin, odd) : secant_reference(fc, ubp, 0.0, tol, &fin)) < 0 || !fin) status |= 1;
        double y = ybp, U = ubp, sprev = 0.0, csum = 0.0; unsigned fl = 0;
        for (int j = 0; j < k; j++) {
            const Surf2 S = cand_surf<true>(V, j);
            const double ts = trace2d_step(S, 1, y, U, sprev, fl);     // reversed Layout{Aspheric}, as above
            csum = (j == 0) ? ts : SA(csum, ts);                       // z = cumsum(ts)  (Types.jl:61-63)
        }
        const double ts_last = SS(V.t[0], sprev);
        const double z1 = SS(SA(csum, ts_last), csum);                 // z[2] = ray.z[end] - ray.z[end-1]  :292
        const double Ubar = -U;                                        // u_bar[1] = -ray.u[end]  :289
        s_x[0][lane] = Ubar;
        s_x[1][lane] = SA(SD(-y, tan(Ubar)), z1);                      // EP_t  :293
    } else {
        // ---- real marginal ray (:223-240)
        double ym = SM(1.0, s);
        auto fm = [&](double yy) { return cand_height<false>(V, stop_c, A.aspheric, yy, 0.0); };   // the system's layout type
        if ((PAIR ? secant_reference_pair(fm, ym, a_stop_signed, tol, &fin, odd) : secant_reference(fm, ym, a_stop_signed, tol, &fin)) < 0 || !fin) status |= 2;
        s_x[2][lane] = ym;
    }
    s_st[role][lane] = status;
    __syncthreads();
    const double Ubar = s_x[0][lane], EP_t = s_x[1][lane], ym = s_x[2][lane];
    const double y_EP = fabs(ym);
    // ---- field point and edge rays (src/PupilSampling.jl:92-100): warp 0 the upper one, warp 1 the lower one
    const double U = SM(fabs(Hrel), Ubar);
    const double u = tan(U);
    double e = role == 0 ? SS(y_EP, SM(u, EP_t)) : SS(-y_EP, SM(u, EP_t));
    auto edge = [&](double yy) { return cand_height<false>(V, stop_c, A.aspheric, yy, U); };    // the system's layout type
    int st2 = 0;
    if ((PAIR ? secant_polish_pair(edge, e, role == 0 ? a_stop : -a_stop, a_stop, odd) : secant_polish(edge, e, role == 0 ? a_stop : -a_stop, a_stop)) < 0) st2 = 4;
    if (role == 1) { s_e2[lane] = e; s_st[1][lane] |= st2; }
    __syncthreads();
    if (role == 0 && live && !odd) {
        status = s_st[0][lane] | s_st[1][lane] | st2;
        for (int j = 0; j < ORT_AIM_NOUT; j++) out[j] = CUDART_NAN;
        if (!lastrow_ok) { out[11] = 8.0; return; }
        out[0] = e; out[1] = s_e2[lane]; out[2] = y_EP; out[3] = u; out[4] = SM(u, f); out[5] = bfd;
        out[6] = (double)stop; out[7] = a_stop; out[8] = EP_t; out[9] = Ubar; out[10] = f; out[11] = (double)status;
        out[12] = numk; out[13] = U; out[14] = 0.0; out[15] = 0.0;     // 14..23: k_aim_edges
    }
}

// ------------------------------------------------------------------------------------------
// FP64 roofline denominator: 8 independent DFMA chains per thread, register resident.
// ------------------------------------------------------------------------------------------
#define PEAK_CHAINS 8
#define PEAK_UNROLL 16
__global__ void __launch_bounds__(512) k_fp64_peak(double* sink, long long iters)
{
    double a[PEAK_CHAINS];
#pragma unroll
    for (int j = 0; j < PEAK_CHAINS; j++) a[j] = 1.0 + 1e-9 * (threadIdx.x + j);
    const double b = 0.9999999, c = 1e-7;
    for (long long it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < PEAK_UNROLL; u++)
#pragma unroll
            for (int j = 0; j < PEAK_CHAINS; j++) a[j] = fma(a[j], b, c);
    }
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < PEAK_CHAINS; j++) s += a[j];
    if (s == 123456.789) sink[0] = s;       // never true; defeats dead-code elimination
}

// ------------------------------------------------------------------------------------------
// Self-test of xdiv / xsqrt (ort_internal.cuh) against the library's __ddiv_rn / __dsqrt_rn: wherever the deferred-slow-path
// forms do NOT raise their flag, the result must be the intrinsic's bit for bit.  Four operand classes per thread and
// iteration: raw 64-bit patterns; moderate magnitudes (2^-80 .. 2^80: no flag expected unless the numerator is zero);
// every exponent with random mantissas; special values (zeros, denormals, the ends of the range, Inf, NaN) against the rest.
// out: [0] divisions tested, [1] flagged, [2] kept-and-different; [3..5] the same for square roots; [6], [7] flags raised
// in the moderate class (division, square root).
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long& x)
{
    unsigned long long z = (x += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ double selftest_operand(int cls, unsigned long long& st)
{
    const unsigned long long z = splitmix64(st);
    const unsigned long long mant = z & 0x000FFFFFFFFFFFFFull, sign = z & 0x8000000000000000ull;
    if (cls == 0) return __longlong_as_double((long long)z);
    if (cls == 1) return __longlong_as_double((long long)(sign | ((1023ull - 80ull + (z >> 52) % 161ull) << 52) | mant));
    if (cls == 2) return __longlong_as_double((long long)(sign | (((z >> 52) % 2047ull) << 52) | mant));
    const unsigned long long special[16] = {0x0ull, 0x8000000000000000ull, 0x7FF0000000000000ull, 0xFFF0000000000000ull,
                                            0x7FF8000000000000ull, 0x1ull, 0x000FFFFFFFFFFFFFull, 0x0010000000000000ull,
                                            0x7FEFFFFFFFFFFFFFull, 0x3FF0000000000000ull, 0xBFF0000000000000ull,
                                            0x0360000000000000ull, 0x035FFFFFFFFFFFFFull, 0x0350000000000000ull,
                                            0x7FD0000000000000ull, 0x7F90000000000000ull};
    return __longlong_as_double((long long)special[(z >> 56) & 15]);
}
__global__ void __launch_bounds__(256) k_selftest_exact(long long iters, unsigned long long seed, unsigned long long* out)
{
    unsigned long long st = seed + 0x632BE59BD9B4E019ull * ((unsigned long long)blockIdx.x * 256 + threadIdx.x + 1);
    unsigned long long c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (long long it = 0; it < iters; it++) {
        const int cls = (int)(it & 3);
        const double a = selftest_operand(cls, st);
        const double b = selftest_operand(cls == 3 ? (int)(splitmix64(st) & 3) : cls, st);
        int bad = 0;
        const double q = xdiv(a, b, bad), q0 = __ddiv_rn(a, b);
        c[0]++; c[1] += bad; c[2] += (!bad && __double_as_longlong(q) != __double_as_longlong(q0)) ? 1 : 0;
        if (cls == 1) c[6] += bad;
        int bad0 = 0;                                            // the zero-numerator form: (+-0) / normal b kept as +-0
        const double qz = xdiv0(a, b, bad0);
        c[2] += (!bad0 && __double_as_longlong(qz) != __double_as_longlong(q0)) ? 1 : 0;
        if (a == 0.0 && !bad0) c[0]++;                           // (counted twice: zero numerators that stay on the fast path)
        const double aa = (cls == 1) ? fabs(a) : a;
        int bad2 = 0;
        const double g = xsqrt(aa, bad2), g0 = __dsqrt_rn(aa);
        c[3]++; c[4] += bad2; c[5] += (!bad2 && __double_as_longlong(g) != __double_as_longlong(g0)) ? 1 : 0;
        if (cls == 1) c[7] += bad2;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        unsigned long long v = c[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(out + k, v);
    }
}
cudaError_t launch_selftest_exact(long long n, unsigned long long seed, unsigned long long* d_out, int sm_count, cudaStream_t st)
{
    const int blocks = sm_count * 4;
    long long iters = (n + (long long)blocks * 256 - 1) / ((long long)blocks * 256);
    if (iters < 4) iters = 4;
    k_selftest_exact<<<blocks, 256, 0, st>>>(iters, seed, d_out);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
cudaError_t launch_trace2d(const Presc& P, const Trace2dArgs& A, cudaStream_t st)
{
    const unsigned nb = (unsigned)((A.N + 255) / 256);
    if (nb == 0) return cudaSuccess;
    k_trace2d<<<nb, 256, 0, st>>>(P, A);
    return cudaGetLastError();
}

cudaError_t launch_paraxial(const LensK& L, const ParaxArgs& A, int arith, cudaStream_t st)
{
    const bool table = A.y_all || A.w_all;
    const bool clip = L.clip != 0;
    // ORT_PX_GRID = CTAs per SM of the persistent grids (tuning)
    static const int per_sm = [] { const char* e = getenv("ORT_PX_GRID"); const int v = e ? atoi(e) : 8; return v < 1 ? 1 : v; }();
    if (!table && L.tau_finite && (!clip || L.clip_nice)) {       // the streaming form
        const long long per = 256 * (clip ? PX2_RPT_CLIP : PX2_RPT), ntl = (A.N + per - 1) / per;
        if (ntl == 0) return cudaSuccess;
        const unsigned nb = (unsigned)(ntl < 148LL * per_sm ? ntl : 148LL * per_sm);
        if (arith == ORT_ARITH_FAST) { if (clip) k_paraxial_final<ORT_ARITH_FAST, true><<<nb, 256, 0, st>>>(L, A); else k_paraxial_final<ORT_ARITH_FAST, false><<<nb, 256, 0, st>>>(L, A); }
        else                         { if (clip) k_paraxial_final<ORT_ARITH_STRICT, true><<<nb, 256, 0, st>>>(L, A); else k_paraxial_final<ORT_ARITH_STRICT, false><<<nb, 256, 0, st>>>(L, A); }
        return cudaGetLastError();
    }
    const long long per = 256 * PX_RPT;
    const long long ntl = (A.N + per - 1) / per;
    if (ntl == 0) return cudaSuccess;
    // 1.6 waves of the 5 resident CTAs/SM; whole-wave grids measured slower (DESIGN.md section 3)
    const unsigned nb = (unsigned)(ntl < 148LL * per_sm ? ntl : 148LL * per_sm);
#define PX_LAUNCH(AR, TB, CL) k_paraxial<AR, TB, CL><<<nb, 256, 0, st>>>(L, A)
    if (arith == ORT_ARITH_FAST) {
        if (table) { if (clip) PX_LAUNCH(ORT_ARITH_FAST, true, true); else PX_LAUNCH(ORT_ARITH_FAST, true, false); }
        else       { if (clip) PX_LAUNCH(ORT_ARITH_FAST, false, true); else PX_LAUNCH(ORT_ARITH_FAST, false, false); }
    } else {
        if (table) { if (clip) PX_LAUNCH(ORT_ARITH_STRICT, true, true); else PX_LAUNCH(ORT_ARITH_STRICT, true, false); }
        else       { if (clip) PX_LAUNCH(ORT_ARITH_STRICT, false, true); else PX_LAUNCH(ORT_ARITH_STRICT, false, false); }
    }
#undef PX_LAUNCH
    return cudaGetLastError();
}

cudaError_t launch_transfer(const TransferArgs& A, cudaStream_t st)
{
    if (A.N == 0) return cudaSuccess;
    long long nb = (A.N + 255) / 256;
    if (nb > 148 * 32) nb = 148 * 32;
    k_transfer<<<(unsigned)nb, 256, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t launch_aim2d(const Presc& P, const AimArgs& A, cudaStream_t st)
{
    if (A.N == 0) return cudaSuccess;
    k_aim2d<<<(unsigned)((A.N + 63) / 64), 64, 0, st>>>(P, A);
    return cudaGetLastError();
}

cudaError_t launch_seidel(const SeidelArgs& A, cudaStream_t st)
{
    if (A.C == 0) return cudaSuccess;
    k_seidel<<<(unsigned)((A.C + 127) / 128), 128, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t launch_vignetting(const VigArgs& A, cudaStream_t st)
{
    if (A.C == 0) return cudaSuccess;
    k_vignetting<<<(unsigned)((A.C + 127) / 128), 128, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t launch_aim_candidates(const AimCandArgs& A, cudaStream_t st)
{
    if (A.C == 0) return cudaSuccess;
    // lane pairs halve the chain of serial traces and double the work: worth it while the kernel is latency-bound
    static const int pair_env = [] { const char* e = getenv("ORT_AIM_PAIR"); return e ? atoi(e) : -1; }();
    const bool pair = pair_env >= 0 ? pair_env != 0 : A.C <= AIM_PAIR_MAX_C;
    if (pair) k_aim_candidates<true><<<(unsigned)((A.C + AIM_CPB - 1) / AIM_CPB), 4 * AIM_CPB, 0, st>>>(A);
    else k_aim_candidates<false><<<(unsigned)((A.C + AIM_CPB - 1) / AIM_CPB), 2 * AIM_CPB, 0, st>>>(A);
    return cudaGetLastError();
}

cudaError_t launch_fp64_peak(double* d_sink, int sm_count, long long iters, cudaStream_t st,
                             long long* dfma_per_launch)
{
    const int blocks = sm_count * 2;
    k_fp64_peak<<<blocks, 512, 0, st>>>(d_sink, iters);
    if (dfma_per_launch) *dfma_per_launch = (long long)blocks * 512 * iters * PEAK_UNROLL * PEAK_CHAINS;
    return cudaGetLastError();
}
