// kern_zernike.cu -- Zernike fit of the ray-traced wavefront (ort_wavefront_zernike_dev, include/ort_b200.h).
//
// The fit is the least-squares fit of the mirrored wavefront; under the mirror only the terms symmetric in x survive
// (header), one per (n, |m|) pair: cos |m|theta for even m, sin |m|theta for odd m.  Their J_s columns are numbered in
// ANSI order ("fitted terms" below).  Four launches, whatever n, n_max and the number of sets:
//
//   k_zern_gram     per CTA: tiles of ZT rays; each of the first ZT threads evaluates the fitted terms of one ray into
//                   shared memory, row [z_0 .. z_{J_s-1}, W, 0 ..] of jp = J_s + 1 rounded up to 4 doubles; then the CTA
//                   does the rank-ZT update of the upper triangle of that row's outer product.  Each thread owns one
//                   4 x 4 block of it in registers for a fixed subset of the tile's rays (DFMA, 16 per 4 LDS.128), so the
//                   column W gives b = sum z W next to G = sum z z^T.  The ray groups are folded in group order; one
//                   partial record per CTA, plus a flag for a kept ray with a non-finite opd.
//   k_zern_solve    one CTA per set: folds the records in CTA order, Cholesky factorisation of G and the two triangular
//                   solves in shared memory; writes coef (ANSI order, antisymmetric terms 0.0) and status.
//   k_zern_resid    the rays again: opd - sum c_k Z_k per kept ray; per CTA the sum of squares, the minimum and maximum.
//   k_zern_finish   one thread per set: folds those in CTA order into resid = (RMS, PV).
//
// No floating-point atomics and fixed fold orders: the results are bit-identical run to run on one device.
#include "kern.cuh"

namespace {

constexpr int ZT = 192;                      // rays per tile of k_zern_gram
constexpr int ZB = 384;                      // threads of k_zern_gram (at most: nblk * R)
constexpr int ZR_THREADS = 256;              // threads of k_zern_resid
constexpr int ZJP_MAX = 52;                  // jp at ORT_ZERN_MAX_ORDER: J_s = 49 fitted terms, W, padding
constexpr int ZJS_MAX = 49;
constexpr double ZERN_PIVOT = 1e-10;         // Cholesky: the pivot must exceed this times the diagonal of G

// sqrt(k), correctly rounded: the normalisation sqrt(2(n+1)) or sqrt(n+1)
__constant__ double kSqrt[27] = {0.0, 1.0, 1.4142135623730951, 1.7320508075688772, 2.0, 2.23606797749979,
                              2.449489742783178, 2.6457513110645907, 2.8284271247461903, 3.0, 3.1622776601683795,
                              3.3166247903554, 3.4641016151377544, 3.605551275463989, 3.7416573867739413,
                              3.872983346207417, 4.0, 4.123105625617661, 4.242640687119285, 4.358898943540674,
                              4.47213595499958, 4.58257569495584, 4.69041575982343, 4.795831523312719,
                              4.898979485566356, 5.0, 5.0990195135927845};

// column of the fitted term (n, |m|): rows n' < n hold n'/2 + 1 terms each; within row n the ANSI order is ascending m,
// i.e. |m| = 0, 2, .., n for even n and |m| = n, n-2, .., 1 (m = -n .. -1) for odd n
__host__ __device__ constexpr int zoff(int n) { return (n / 2) * (n / 2 + 1) + ((n & 1) ? n / 2 + 1 : 0); }
__host__ __device__ constexpr int zcol(int n, int am) { return zoff(n) + ((n & 1) ? (n - am) / 2 : am / 2); }

__device__ __forceinline__ double znorm(int n, int am) { return am ? kSqrt[2 * (n + 1)] : kSqrt[n + 1]; }

// emit(k, Z_k(rho, theta)) for every fitted term of order <= n_max.  cos / sin of m theta by the Chebyshev recurrence
// from sincos(theta); the radial polynomials per m by Kintner's three-term recurrence in n from R_m^m = rho^m and
// R_{m+2}^m = rho^m ((m+2) rho^2 - (m+1)), which keeps the digits the factorial sum loses near rho = 1 at high order.
template <class F>
__device__ __forceinline__ void zern_eval(int n_max, double rho, double theta, F&& emit)
{
    double s1, c1;
    sincos(theta, &s1, &c1);
    const double r2 = rho * rho, c2 = c1 + c1;
    double cm = 1.0, cq = c1, sm = 0.0, sq = -s1;    // cos, sin of m theta and of (m - 1) theta
    double rm = 1.0;                                 // rho^m
#pragma unroll
    for (int m = 0; m <= ORT_ZERN_MAX_ORDER; m++) {
        if (m > n_max) break;
        if (m) {
            const double cn = fma(c2, cm, -cq), sn = fma(c2, sm, -sq);
            cq = cm; cm = cn; sq = sm; sm = sn;
            rm *= rho;
        }
        const double ang = (m & 1) ? sm : cm;
        emit(zcol(m, m), znorm(m, m) * (rm * ang));
        double Rq = 0.0, Rn = rm;                    // R_{n-4}^m, R_{n-2}^m
#pragma unroll
        for (int n = m + 2; n <= ORT_ZERN_MAX_ORDER; n += 2) {
            if (n > n_max) break;
            double Rt;
            if (n == m + 2) {
                Rt = rm * fma((double)(m + 2), r2, -(double)(m + 1));
            } else {
                const double K1 = (double)((n + m) * (n - m) * (n - 2)) / 2.0;
                const double K2 = 2.0 * n * (n - 1) * (n - 2);
                const double K3 = -(double)(m * m * (n - 1)) - (double)(n * (n - 1) * (n - 2));
                const double K4 = -(double)(n * (n + m - 2) * (n - m - 2)) / 2.0;
                Rt = fma(K2 / K1, r2, K3 / K1) * Rn + (K4 / K1) * Rq;
            }
            Rq = Rn; Rn = Rt;
            emit(zcol(n, m), znorm(n, m) * (Rn * ang));
        }
    }
}

__device__ __forceinline__ long long set_len(const ZernArgs& A, int s)
{
    return A.mask ? A.stride : min((long long)A.stats[s].n_kept, A.stride);
}

__device__ __forceinline__ double set_rnorm(const ZernArgs& A, int s)
{
    return A.r_norm > 0.0 ? A.r_norm : A.stats[s].r_max;
}

__global__ void __launch_bounds__(ZB, 2) k_zern_gram(const __grid_constant__ ZernArgs A)
{
    extern __shared__ double z_tile[];       // [ZT][jp]; at the end [R][nblk * 16] for the fold of the ray groups
    const int s = blockIdx.y, t = threadIdx.x, jp = A.jp, js = A.js, nblk = A.nblk, R = A.R;
    const int blk = t % nblk, grp = t / nblk;
    const bool active = grp < R;
    int bi = 0, rem = blk;                   // block (bi, bj), bi <= bj, of the jp/4 x jp/4 upper block triangle
    while (rem >= jp / 4 - bi) { rem -= jp / 4 - bi; bi++; }
    const int bj = bi + rem;
    const size_t o = (size_t)s * A.stride;
    const double *opd = A.opd + o, *r = A.r + o, *th = A.theta + o;
    const uint8_t* mask = A.mask ? A.mask + o : nullptr;
    const long long len = set_len(A, s);
    const double rn = set_rnorm(A, s);
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.0;
    int bad = 0;
    for (long long t0 = (long long)blockIdx.x * ZT; t0 < len; t0 += (long long)gridDim.x * ZT) {
        __syncthreads();
        if (t < ZT) {
            double* row = z_tile + t * jp;
            const long long i = t0 + t;
            int k0 = 0;
            if (i < len && (!mask || mask[i] == 1)) {
                const double w = opd[i];
                bad |= !isfinite(w);
                zern_eval(A.n_max, r[i] / rn, th[i], [&](int k, double v) { row[k] = v; });
                row[js] = w;
                k0 = js + 1;
            }
            for (int k = k0; k < jp; k++) row[k] = 0.0;
        }
        __syncthreads();
        if (active) {
            const int nt = (int)min((long long)ZT, len - t0);
            for (int u = grp; u < nt; u += R) {
                const double2* zr = (const double2*)(z_tile + u * jp);
                const double2 a0 = zr[2 * bi], a1 = zr[2 * bi + 1], b0 = zr[2 * bj], b1 = zr[2 * bj + 1];
                const double a[4] = {a0.x, a0.y, a1.x, a1.y}, b[4] = {b0.x, b0.y, b1.x, b1.y};
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) acc[i][j] = fma(a[i], b[j], acc[i][j]);
            }
        }
    }
    bad = __syncthreads_or(bad);
    if (active)
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) z_tile[((size_t)grp * nblk + blk) * 16 + i * 4 + j] = acc[i][j];
    __syncthreads();
    const int rs = nblk * 16 + 1;
    double* out = A.gpart + ((size_t)s * gridDim.x + blockIdx.x) * rs;
    for (int e = t; e < nblk * 16; e += blockDim.x) {
        double v = 0.0;
        for (int g = 0; g < R; g++) v += z_tile[(size_t)g * nblk * 16 + e];
        out[e] = v;
    }
    if (t == 0) out[nblk * 16] = bad ? 1.0 : 0.0;
}

__global__ void __launch_bounds__(256) k_zern_solve(const __grid_constant__ ZernArgs A)
{
    __shared__ double sG[ZJP_MAX * ZJP_MAX];   // G and b (column js); L in the lower triangle
    __shared__ double sD[ZJS_MAX], sY[ZJS_MAX];
    __shared__ int s_status;
    const int s = blockIdx.x, t = threadIdx.x, jp = A.jp, js = A.js, nblk = A.nblk, rs = nblk * 16 + 1;
    const double* P = A.gpart + (size_t)s * A.gx * rs;
    for (int e = t; e < nblk * 16; e += blockDim.x) {
        double v = 0.0;
        for (int c = 0; c < A.gx; c++) v += P[(size_t)c * rs + e];
        int bi = 0, rem = e / 16;
        while (rem >= jp / 4 - bi) { rem -= jp / 4 - bi; bi++; }
        const int row = 4 * bi + (e % 16) / 4, col = 4 * (bi + rem) + e % 4;
        sG[row * jp + col] = v;
        sG[col * jp + row] = v;
    }
    if (t == 0) {
        bool bad = false;
        for (int c = 0; c < A.gx; c++) bad |= P[(size_t)c * rs + nblk * 16] != 0.0;
        s_status = A.stats[s].n_kept < js ? 1 : bad ? 3 : 0;
    }
    __syncthreads();
    if (t < js) sD[t] = sG[t * jp + t];
    __syncthreads();
    const bool factor = s_status == 0;
    for (int k = 0; factor && k < js; k++) {
        if (t == 0) {
            double d = sG[k * jp + k];
            for (int p = 0; p < k; p++) d -= sG[k * jp + p] * sG[k * jp + p];
            if (d > ZERN_PIVOT * sD[k]) sG[k * jp + k] = sqrt(d);
            else s_status = 2;
        }
        __syncthreads();
        if (s_status) break;
        const double lkk = sG[k * jp + k];
        for (int i = k + 1 + t; i < js; i += blockDim.x) {
            double v = sG[i * jp + k];
            for (int p = 0; p < k; p++) v -= sG[i * jp + p] * sG[k * jp + p];
            sG[i * jp + k] = v / lkk;
        }
        __syncthreads();
    }
    if (t) return;
    const int st = s_status;
    double* csym = A.csym + (size_t)s * ZJS_MAX;
    if (st == 0) {
        for (int k = 0; k < js; k++) {                                   // L y = b
            double v = sG[k * jp + js];
            for (int p = 0; p < k; p++) v -= sG[k * jp + p] * sY[p];
            sY[k] = v / sG[k * jp + k];
        }
        for (int k = js - 1; k >= 0; k--) {                              // L^T c = y
            double v = sY[k];
            for (int p = k + 1; p < js; p++) v -= sG[p * jp + k] * sY[p];
            sY[k] = v / sG[k * jp + k];
        }
    }
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    double* coef = A.coef + (size_t)s * ((A.n_max + 1) * (A.n_max + 2) / 2);
    for (int n = 0, j = 0; n <= A.n_max; n++)
        for (int m = -n; m <= n; m += 2, j++) {
            const int am = m < 0 ? -m : m;
            const bool sym = (am & 1) ? m < 0 : m >= 0;
            coef[j] = st ? nan : sym ? sY[zcol(n, am)] : 0.0;
        }
    for (int k = 0; k < js; k++) csym[k] = st ? nan : sY[k];
    A.status[s] = st;
}

__global__ void __launch_bounds__(ZR_THREADS) k_zern_resid(const __grid_constant__ ZernArgs A)
{
    __shared__ double sc[ZJS_MAX];
    __shared__ double s_red[ZR_THREADS / 32][3];
    const int s = blockIdx.y, t = threadIdx.x;
    if (A.status[s] != 0) return;
    if (t < A.js) sc[t] = A.csym[(size_t)s * ZJS_MAX + t];
    __syncthreads();
    const size_t o = (size_t)s * A.stride;
    const double *opd = A.opd + o, *r = A.r + o, *th = A.theta + o;
    const uint8_t* mask = A.mask ? A.mask + o : nullptr;
    const long long len = set_len(A, s);
    const double rn = set_rnorm(A, s);
    double ssq = 0.0, mn = INFINITY, mx = -INFINITY;
    for (long long i = (long long)blockIdx.x * ZR_THREADS + t; i < len; i += (long long)gridDim.x * ZR_THREADS) {
        if (mask && mask[i] != 1) continue;
        double fit = 0.0;
        zern_eval(A.n_max, r[i] / rn, th[i], [&](int k, double v) { fit = fma(sc[k], v, fit); });
        const double e = opd[i] - fit;
        ssq = fma(e, e, ssq);
        mn = fmin(mn, e); mx = fmax(mx, e);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        ssq += __shfl_xor_sync(0xffffffffu, ssq, d);
        mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, d));
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    }
    if ((t & 31) == 0) { s_red[t >> 5][0] = ssq; s_red[t >> 5][1] = mn; s_red[t >> 5][2] = mx; }
    __syncthreads();
    if (t) return;
    for (int w = 1; w < ZR_THREADS / 32; w++) {
        ssq += s_red[w][0]; mn = fmin(mn, s_red[w][1]); mx = fmax(mx, s_red[w][2]);
    }
    double* out = A.rpart + ((size_t)s * gridDim.x + blockIdx.x) * 3;
    out[0] = ssq; out[1] = mn; out[2] = mx;
}

__global__ void k_zern_finish(const __grid_constant__ ZernArgs A)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= A.n_sets) return;
    double* res = A.resid + (size_t)s * 2;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (A.status[s] != 0) { res[0] = res[1] = nan; return; }
    double ssq = 0.0, mn = INFINITY, mx = -INFINITY;
    const double* P = A.rpart + (size_t)s * A.gx_resid * 3;
    for (int c = 0; c < A.gx_resid; c++) { ssq += P[3 * c]; mn = fmin(mn, P[3 * c + 1]); mx = fmax(mx, P[3 * c + 2]); }
    res[0] = sqrt(ssq / (double)A.stats[s].n_kept);
    res[1] = mx - mn;
}

size_t gram_smem(const ZernArgs& A)
{
    const size_t tile = (size_t)ZT * A.jp, fold = (size_t)A.R * A.nblk * 16;
    return sizeof(double) * (tile > fold ? tile : fold);
}

}  // namespace

int zern_fitted_terms(int n_max) { return zoff(n_max + 1); }

cudaError_t zern_dims(ZernArgs& A, int sm_count)
{
    A.js = zern_fitted_terms(A.n_max);
    A.jp = (A.js + 1 + 3) / 4 * 4;
    A.nblk = (A.jp / 4) * (A.jp / 4 + 1) / 2;
    A.R = ZB / A.nblk;
    cudaError_t e = cudaFuncSetAttribute(k_zern_gram, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(sizeof(double) * (ZT * ZJP_MAX > ZB * 16 ? ZT * ZJP_MAX : ZB * 16)));
    if (e != cudaSuccess) return e;
    int occ = 0, occ_r = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_zern_gram, A.nblk * A.R, gram_smem(A))) != cudaSuccess)
        return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_r, k_zern_resid, ZR_THREADS, 0)) != cudaSuccess) return e;
    // one wave of resident CTAs over all sets, no more CTAs per set than it has tiles
    const long long tiles = (A.stride + ZT - 1) / ZT, tiles_r = (A.stride + ZR_THREADS - 1) / ZR_THREADS;
    long long gx = (long long)sm_count * (occ > 0 ? occ : 1) / A.n_sets;
    long long gr = (long long)sm_count * (occ_r > 0 ? occ_r : 1) / A.n_sets;
    A.gx = (int)(gx < 1 ? 1 : gx > tiles ? tiles : gx);
    A.gx_resid = (int)(gr < 1 ? 1 : gr > tiles_r ? tiles_r : gr);
    return cudaSuccess;
}

size_t zern_gram_record(const ZernArgs& A) { return (size_t)A.nblk * 16 + 1; }

cudaError_t launch_zernike(const ZernArgs& A, cudaStream_t st, int* launches)
{
    k_zern_gram<<<dim3((unsigned)A.gx, (unsigned)A.n_sets), A.nblk * A.R, gram_smem(A), st>>>(A);
    k_zern_solve<<<A.n_sets, 256, 0, st>>>(A);
    k_zern_resid<<<dim3((unsigned)A.gx_resid, (unsigned)A.n_sets), ZR_THREADS, 0, st>>>(A);
    k_zern_finish<<<1, 32, 0, st>>>(A);
    *launches = 4;
    return cudaGetLastError();
}
