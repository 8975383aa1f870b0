// kern_mtf.cu -- diffraction MTF of the ray-traced wavefront (ort_wavefront_mtf_dev, include/ort_b200.h).
//
// The OTF is the normalised autocorrelation of the mirrored pupil amplitude A (column x = 0 doubled), evaluated as direct
// lag sums at the lattice lags the requested frequencies need: slot 2f + e of an azimuth holds lag floor(q_f) + e
// (q_f = nu_f / (s d)), slot 2 n_freq lag 0.  Four launches, whatever the sizes:
//
//   k_mtf_pupil  Ah = mask exp(2 pi i W), column 0 doubled, from opd by sincospi: stored row-major (the sagittal rows) and,
//                through a 32 x 32 shared-memory tile, transposed (the tangential columns).  One non-finite flag per tile.
//   k_mtf_sag    per row, C(k) = [k even] |Ah[k/2]|^2 + 2 sum_{j > -k/2}^{nx-1-k} Re Ah[|j+k|] conj Ah[|j|]: the pairs of
//                the mirrored row taken once each (j and -j-k are conjugate terms), 2 DFMA per product.  Each lag walks
//                its own j range, so every product loads both operands (2 loads, no range tests).
//   k_mtf_tan    per column, w_ix sum_iy Ah[iy+k] conj Ah[iy] (w_0 = 1: Ah is already doubled there, w = 2 for the
//                mirrored pair of every other column), 4 DFMA per product.
//                Both lag kernels: a CTA takes one block of <= LB lag slots over a group of rows, one accumulator per
//                slot and thread.  k_mtf_tan reads Ah[i] once per lag block and walks the union of the lags' ranges (all
//                start at 0), so a product costs one 16-byte load.  A row of up to
//                LMAX elements is staged in shared memory by cp.async and read from there (two CTAs per SM: one
//                stages while the other multiplies); a longer row is read through L1 from global memory.  The CTAs of
//                one row group and different lag blocks are adjacent in the grid and share the rows in L2.
//   k_mtf_fold   one CTA per set: the row-group partials folded in group order, OTF(k) = C(k) / C(0), interpolated
//                between the two lags of each frequency, and the status.
//
// No floating-point atomics and fixed fold orders: the results are bit-identical run to run on one device.
#include <climits>

#include "kern.cuh"

namespace {

constexpr int MT = 256;     // threads of every MTF kernel
constexpr int LB = 16;      // lag slots per block of k_mtf_sag / k_mtf_tan (accumulators per thread)
constexpr int TW = 32;      // k_mtf_pupil tile side
constexpr int LMAX = 6144;  // longest row staged in shared memory (96 KB: two CTAs per SM)

__device__ __forceinline__ void cp_async16(void* smem, const void* g)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(g));
}

// row r of Ah (at g + r len) for the lag sums, called for r = r0 .. r1 - 1 in order.  SM: staged in shared memory by
// cp.async (barriers on both sides of the copy); otherwise read in place.
template <bool SM>
__device__ __forceinline__ const double2* stage_row(const double2* g, int r, int len, double2* row)
{
    g += (size_t)r * len;
    if (!SM) return g;
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += blockDim.x) cp_async16(row + i, g + i);
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();
    return row;
}

__device__ __forceinline__ double mtf_nan() { return __longlong_as_double(0x7ff8000000000000ll); }

// the signed lattice step of azimuth az: dx = xs[nx-1] / (nx-1), dy_s = (ys_s[ny-1] - ys_s[0]) / (ny-1)
__device__ __forceinline__ double lattice_step(const MtfArgs& A, int s, int az)
{
    if (az == 0) return A.xs[A.nx - 1] / (double)(A.nx - 1);
    const double* ys = A.ys + (size_t)s * A.ys_stride;
    return (ys[A.ny - 1] - ys[0]) / (double)(A.ny - 1);
}

__device__ __forceinline__ int last_lag(const MtfArgs& A, int az) { return az == 0 ? 2 * (A.nx - 1) : A.ny - 1; }

// q = nu / (s d) of frequency f at step |d| (d finite and > 0)
__device__ __forceinline__ double lag_q(const MtfArgs& A, int f, double d)
{
    const double nu = A.freqs[f];
    return nu == 0.0 ? 0.0 : nu / (A.scale * d);
}

// the lag of slot l at step |d|, or -1: past the last lag kmax, or d not a usable step (status 4 of the fold)
__device__ __forceinline__ int slot_lag(const MtfArgs& A, int l, double d, int kmax)
{
    if (!(d > 0.0 && d < INFINITY)) return -1;
    if (l == 2 * A.n_freq) return 0;
    const double q = lag_q(A, l >> 1, d);
    if (!(q < (double)kmax + 1.0)) return -1;
    const int k = (int)floor(q) + (l & 1);
    return k <= kmax ? k : -1;
}

__global__ void __launch_bounds__(MT) k_mtf_pupil(const __grid_constant__ MtfArgs A)
{
    __shared__ double2 tile[TW][TW + 1];
    const int s = blockIdx.y, t = threadIdx.x, lane = t % TW, w = t / TW;
    const int x0 = (blockIdx.x % A.tiles_x) * TW, y0 = (blockIdx.x / A.tiles_x) * TW;
    const size_t o = (size_t)s * A.stride;
    bool bad = false;
#pragma unroll
    for (int q = 0; q < TW / (MT / TW); q++) {
        const int iy = y0 + w + (MT / TW) * q, ix = x0 + lane;
        double2 p = make_double2(0.0, 0.0);
        if (iy < A.ny && ix < A.nx) {
            const size_t i = o + (size_t)iy * A.nx + ix;
            if (A.mask[i] == 1) {
                const double v = A.opd[i];
                bad |= !isfinite(v);
                sincospi(2.0 * v, &p.y, &p.x);
                if (ix == 0) { p.x *= 2.0; p.y *= 2.0; }
            }
            A.P[i] = p;
        }
        tile[w + (MT / TW) * q][lane] = p;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < TW / (MT / TW); q++) {
        const int ix = x0 + w + (MT / TW) * q, iy = y0 + lane;
        if (iy < A.ny && ix < A.nx) A.PT[o + (size_t)ix * A.ny + iy] = tile[lane][w + (MT / TW) * q];
    }
    bad = __syncthreads_or(bad);
    if (t == 0) A.bad[(size_t)s * A.tiles + blockIdx.x] = bad ? 1 : 0;
}

// the per-thread accumulators of one lag block folded in a fixed order (lanes, then warps); thread l < nl gets slot l
template <int NV>
__device__ __forceinline__ void fold_block(double (&acc)[LB][NV], double (*red)[LB][NV], int nl, double (&out)[NV])
{
    const int t = threadIdx.x;
#pragma unroll
    for (int l = 0; l < LB; l++)
#pragma unroll
        for (int v = 0; v < NV; v++) {
#pragma unroll
            for (int d = 16; d; d >>= 1) acc[l][v] += __shfl_xor_sync(0xffffffffu, acc[l][v], d);
            if ((t & 31) == 0) red[t >> 5][l][v] = acc[l][v];
        }
    __syncthreads();
#pragma unroll
    for (int v = 0; v < NV; v++) out[v] = 0.0;
    if (t < nl)
        for (int q = 0; q < MT / 32; q++)
#pragma unroll
            for (int v = 0; v < NV; v++) out[v] += red[q][t][v];
}

template <bool SM>
__global__ void __launch_bounds__(MT) k_mtf_sag(const __grid_constant__ MtfArgs A)
{
    __shared__ double red[MT / 32][LB][1];
    extern __shared__ double2 mtf_row[];
    const int s = blockIdx.z, t = threadIdx.x, nx = A.nx, kmax = 2 * (nx - 1);
    const int l0 = blockIdx.x * A.lb, nl = min(A.lb, A.n_slot - l0);
    const double dx = lattice_step(A, s, 0);
    // per slot: the lag and the range j in [-jneg, jpos] of its terms, j > -k/2 (one term of each conjugate pair
    // (j, -j-k); jneg = floor((k-1)/2), -1 at k = 0) and j <= nx-1-k; the part j < 0 is walked as i = -j, where
    // Ah[|j|] = Ah[i] and Ah[|j+k|] = Ah[k-i]
    int k[LB], jneg[LB], jpos[LB];
#pragma unroll
    for (int l = 0; l < LB; l++) {
        k[l] = l < nl ? slot_lag(A, l0 + l, dx, kmax) : -1;
        jneg[l] = k[l] >= 0 ? (k[l] - 1) >> 1 : 0;
        jpos[l] = k[l] >= 0 ? nx - 1 - k[l] : -1;
    }
    const int kt = t < nl ? slot_lag(A, l0 + t, dx, kmax) : -1;   // the slot whose self-conjugate term thread t adds
    double acc[LB][1], fix = 0.0;
#pragma unroll
    for (int l = 0; l < LB; l++) acc[l][0] = 0.0;
    const int r0 = blockIdx.y * A.rl_s, r1 = min(A.ny, r0 + A.rl_s);
    for (int r = r0; r < r1; r++) {
        const double2* p = stage_row<SM>(A.P + (size_t)s * A.stride, r, nx, mtf_row);
#pragma unroll
        for (int l = 0; l < LB; l++) {
            if (k[l] < 0) continue;
            double c = acc[l][0];
#pragma unroll 1
            for (int j = max(0, -jneg[l]) + t; j <= jpos[l]; j += MT) {      // k = 0 starts at j = 1
                const double2 a = p[j], b = p[j + k[l]];
                c = fma(b.x, a.x, fma(b.y, a.y, c));
            }
#pragma unroll 1
            for (int i = max(1, -jpos[l]) + t; i <= jneg[l]; i += MT) {
                const double2 a = p[i], b = p[k[l] - i];
                c = fma(b.x, a.x, fma(b.y, a.y, c));
            }
            acc[l][0] = c;
        }
        if (kt >= 0 && (kt & 1) == 0) {
            const double2 c = p[kt >> 1];
            fix = fma(c.x, c.x, fma(c.y, c.y, fix));
        }
    }
    double out[1];
    fold_block<1>(acc, red, nl, out);
    if (t < nl) A.psag[((size_t)s * A.rg_s + blockIdx.y) * A.n_slot + l0 + t] = fma(2.0, out[0], fix);
}

template <bool SM>
__global__ void __launch_bounds__(MT) k_mtf_tan(const __grid_constant__ MtfArgs A)
{
    __shared__ double red[MT / 32][LB][2];
    extern __shared__ double2 mtf_row[];
    const int s = blockIdx.z, t = threadIdx.x, ny = A.ny, kmax = ny - 1;
    const int l0 = blockIdx.x * A.lb, nl = min(A.lb, A.n_slot - l0);
    const double dy = fabs(lattice_step(A, s, 1));
    int k[LB], hi[LB];
    int imax = INT_MIN;
#pragma unroll
    for (int l = 0; l < LB; l++) {
        k[l] = l < nl ? slot_lag(A, l0 + l, dy, kmax) : -1;
        hi[l] = k[l] >= 0 ? ny - 1 - k[l] : -1;
        imax = max(imax, hi[l]);
    }
    double acc[LB][2];
#pragma unroll
    for (int l = 0; l < LB; l++) acc[l][0] = acc[l][1] = 0.0;
    const int c0 = blockIdx.y * A.rl_t, c1 = min(A.nx, c0 + A.rl_t);
    for (int c = c0; c < c1; c++) {
        const double2* p = stage_row<SM>(A.PT + (size_t)s * A.stride, c, ny, mtf_row);
        const double wc = c == 0 ? 1.0 : 2.0;           // column 0 is doubled in Ah; every other column has a mirror twin
        for (int i = t; i <= imax; i += MT) {
            double2 a = p[i];
            a.x *= wc; a.y *= wc;
#pragma unroll
            for (int l = 0; l < LB; l++)
                if (i <= hi[l]) {
                    const double2 b = p[i + k[l]];
                    acc[l][0] = fma(b.x, a.x, fma(b.y, a.y, acc[l][0]));
                    acc[l][1] = fma(b.y, a.x, fma(-b.x, a.y, acc[l][1]));
                }
        }
    }
    double out[2];
    fold_block<2>(acc, red, nl, out);
    if (t < nl) A.ptan[((size_t)s * A.rg_t + blockIdx.y) * A.n_slot + l0 + t] = make_double2(out[0], out[1]);
}

// C of slot l of azimuth az, its row-group partials folded in group order
__device__ double2 slot_sum(const MtfArgs& A, int s, int az, int l)
{
    double2 c = make_double2(0.0, 0.0);
    if (az == 0) {
        const double* p = A.psag + (size_t)s * A.rg_s * A.n_slot + l;
        for (int g = 0; g < A.rg_s; g++) c.x += p[(size_t)g * A.n_slot];
    } else {
        const double2* p = A.ptan + (size_t)s * A.rg_t * A.n_slot + l;
        for (int g = 0; g < A.rg_t; g++) { const double2 v = p[(size_t)g * A.n_slot]; c.x += v.x; c.y += v.y; }
    }
    return c;
}

__global__ void __launch_bounds__(MT) k_mtf_fold(const __grid_constant__ MtfArgs A)
{
    const int s = blockIdx.x, t = threadIdx.x;
    bool bad = false;
    for (int i = t; i < A.tiles; i += MT) bad |= A.bad[(size_t)s * A.tiles + i] != 0;
    bad = __syncthreads_or(bad);
    const double dx = lattice_step(A, s, 0), dy = lattice_step(A, s, 1);
    const bool lattice = A.xs[0] == 0.0 && isfinite(dx) && dx > 0.0 && isfinite(dy) && dy != 0.0;
    const int st = A.stats[s].n_kept <= 0 ? 1 : bad ? 3 : !lattice ? 4 : 0;
    double* otf = A.otf + (size_t)s * 2 * A.n_freq * 2;
    for (int e = t; e < 2 * A.n_freq; e += MT) {
        const int az = e / A.n_freq, f = e % A.n_freq;
        double2 v = make_double2(mtf_nan(), mtf_nan());
        if (st == 0) {
            const double d = az == 0 ? dx : fabs(dy);
            const int kmax = last_lag(A, az);
            const double c0 = slot_sum(A, s, az, 2 * A.n_freq).x;
            const int k0 = slot_lag(A, 2 * f, d, kmax), k1 = slot_lag(A, 2 * f + 1, d, kmax);
            v = make_double2(0.0, 0.0);
            if (k0 >= 0) {
                const double q = lag_q(A, f, d), fr = q - floor(q);
                // OTF(k) = C(k) / C(0); OTF(0) = 1 exactly; OTF(k) = 0 past the last lag
                double2 o0 = make_double2(1.0, 0.0), o1 = make_double2(0.0, 0.0);
                if (k0 > 0) { const double2 c = slot_sum(A, s, az, 2 * f); o0 = make_double2(c.x / c0, c.y / c0); }
                if (k1 > 0) { const double2 c = slot_sum(A, s, az, 2 * f + 1); o1 = make_double2(c.x / c0, c.y / c0); }
                v.x = fma(fr, o1.x, (1.0 - fr) * o0.x);
                v.y = fma(fr, o1.y, (1.0 - fr) * o0.y);
                if (az == 0) v.y = 0.0;                 // the sagittal OTF is real (the mirror)
                else if (dy < 0.0) v.y = -v.y;          // ys descending: nu > 0 pairs iy with iy + k as conj C(k)
            }
        }
        otf[(size_t)e * 2] = v.x;
        otf[(size_t)e * 2 + 1] = v.y;
    }
    if (t == 0) A.status[s] = st;
}

size_t sag_smem(const MtfArgs& A) { return sizeof(double2) * (size_t)A.nx; }
size_t tan_smem(const MtfArgs& A) { return sizeof(double2) * (size_t)A.ny; }

// row groups of a lag kernel over `rows` rows per set: about four CTAs per resident slot, a whole number of rows each
void groups(int rows, int n_sets, int nlb, int slots, int& rg, int& rl)
{
    long long g = (4LL * slots + (long long)n_sets * nlb - 1) / ((long long)n_sets * nlb);
    g = g < 1 ? 1 : g > rows ? rows : g;
    rl = (int)((rows + g - 1) / g);
    rg = (rows + rl - 1) / rl;
}

}  // namespace

cudaError_t mtf_occupancy(int (&occ)[2][2])
{
    // the staged kernels at the largest stage: registers, not shared memory, bound them below it
    const int smem = (int)(sizeof(double2) * LMAX);
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_mtf_sag<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_mtf_tan<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[0][1], k_mtf_sag<true>, MT, smem)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[0][0], k_mtf_sag<false>, MT, 0)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[1][1], k_mtf_tan<true>, MT, smem)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ[1][0], k_mtf_tan<false>, MT, 0)) != cudaSuccess)
        return e;
    for (auto& o : occ)
        for (int& v : o) v = v > 0 ? v : 1;
    return cudaSuccess;
}

cudaError_t mtf_dims(MtfArgs& A, int sm_count, const int (&occ)[2][2])
{
    A.n_slot = 2 * A.n_freq + 1;
    A.nlb = (A.n_slot + LB - 1) / LB;
    A.lb = (A.n_slot + A.nlb - 1) / A.nlb;
    A.tiles_x = (A.nx + TW - 1) / TW;
    A.tiles = A.tiles_x * ((A.ny + TW - 1) / TW);
    groups(A.ny, A.n_sets, A.nlb, sm_count * occ[0][A.nx <= LMAX], A.rg_s, A.rl_s);
    groups(A.nx, A.n_sets, A.nlb, sm_count * occ[1][A.ny <= LMAX], A.rg_t, A.rl_t);
    return cudaSuccess;
}

cudaError_t launch_mtf(const MtfArgs& A, cudaStream_t st, int* launches)
{
    k_mtf_pupil<<<dim3((unsigned)A.tiles, (unsigned)A.n_sets), MT, 0, st>>>(A);
    const dim3 gs((unsigned)A.nlb, (unsigned)A.rg_s, (unsigned)A.n_sets), gt((unsigned)A.nlb, (unsigned)A.rg_t, (unsigned)A.n_sets);
    if (A.nx <= LMAX) k_mtf_sag<true><<<gs, MT, sag_smem(A), st>>>(A);
    else k_mtf_sag<false><<<gs, MT, 0, st>>>(A);
    if (A.ny <= LMAX) k_mtf_tan<true><<<gt, MT, tan_smem(A), st>>>(A);
    else k_mtf_tan<false><<<gt, MT, 0, st>>>(A);
    k_mtf_fold<<<A.n_sets, MT, 0, st>>>(A);
    *launches = 4;
    return cudaGetLastError();
}
