// kern_psf.cu -- diffraction PSF and Strehl ratio of the ray-traced wavefront (ort_wavefront_psf_dev, include/ort_b200.h).
//
// A matrix Fourier transform of the pupil function P = mask exp(2 pi i W) on the sweep's own grid (not an FFT: the image
// sampling is free of the pupil sampling).  The PSF is even in xi (the mirrored set), so only the nuh = ceil(n_u / 2)
// columns with xi >= 0 are computed and written to both mirrored pixels.  Five launches, whatever the sizes:
//
//   k_psf_table  C[ix][j] = 2 cos(2 pi s x_ix xi_j), shared by every set; columns nuh .. nup - 1 are 0.
//   k_psf_x      stage A, T_s[iy][j] = sum_ix P_s[iy][ix] C[ix][j]: a real x complex GEMM over (2 ny x nx)(nx x nup).
//                P is generated from opd and mask (sincospi) while a tile is staged in shared memory, never stored.  CTA
//                tile BM complex rows x BN columns, 4 x 8 per thread in registers (64 DFMA per 8 LDS.128 and k).  The
//                ix range may be split into kx chunks (partial T per chunk) to even out the last CTA wave.  The thread
//                that generates P also adds it up: sum_ix P, the weight-1 column of strehl_ref, costs no GEMM column.
//   k_psf_y      stage B, E_s[iv][j] = sum_iy Y_s[iv][iy] T_s[iy][j], Y = exp(2 pi i s (y - ybar) eta): a complex GEMM,
//                Y generated and T summed over its kx chunks while a tile is staged.  64 x 64 CTA tile, 4 x 4 complex
//                per thread; the iy range split into ky chunks (one partial E per chunk) to even out the last CTA wave.
//   k_psf_fold   per pixel: the ky partial E folded in chunk order, |E|^2 / (2n)^2 into both mirrored columns; per CTA
//                the maximum and its lowest grid index.
//   k_psf_peak   one CTA per set: strehl_ref from the sum_ix P records, the maximum and peak, the status.
//
// No floating-point atomics and fixed fold orders: the results are bit-identical run to run on one device.
#include <climits>

#include "kern.cuh"

namespace {

constexpr int PT = 256;     // threads of every PSF kernel but k_psf_table
constexpr int BK = 16;      // contraction depth of one shared-memory tile (ix in stage A, iy in stage B)
constexpr int YB = 64;      // stage B tile: 64 iv x 64 j, 16 x 16 threads
constexpr int MAX_KX = 4;   // stage A chunks of the ix range
constexpr int MAX_KY = 64;  // stage B chunks of the iy range

__device__ __forceinline__ double psf_nan() { return __longlong_as_double(0x7ff8000000000000ll); }

// xi of computed column j (pixel iu = n_u - nuh + j), eta of pixel row iv: (i - (n - 1)/2) d, the half-integer exact
__device__ __forceinline__ double pix(int i, int n, double d) { return (double)(2 * i - (n - 1)) * 0.5 * d; }

__device__ __forceinline__ void cp_async8(void* smem, const void* g)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(g));
}
__device__ __forceinline__ void cp_async16(void* smem, const void* g)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(g));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

__device__ __forceinline__ int set_status(const PsfArgs& A, int s, bool bad)
{
    return A.stats[s].n_kept <= 0 ? 1 : bad ? 3 : 0;
}

__global__ void k_psf_table(const __grid_constant__ PsfArgs A)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)A.nx * A.nup) return;
    const int ix = (int)(e / A.nup), j = (int)(e % A.nup);
    double c = 0.0;
    if (j < A.nuh) c = 2.0 * cospi(2.0 * A.scale * A.xs[ix] * pix(A.n_u - A.nuh + j, A.n_u, A.du));
    A.ctab[e] = c;
}

// stage A.  TX threads along the columns (8 columns each, as 4 double2 at stride TX), PT / TX along the rows (4 complex
// rows each, at stride PT / TX).  Shared memory: As [2][BK][BM + 1] double2 (the +1 spreads the transposing stores over the
// banks), Bs [2][BK][BN] double.
template <int TX>
__global__ void __launch_bounds__(PT, 1) k_psf_x(const __grid_constant__ PsfArgs A)
{
    constexpr int TY = PT / TX, BM = 4 * TY, BN = 8 * TX, AP = BM + 1;
    constexpr int NQ = BM * BK / PT;            // P elements staged per thread and tile
    constexpr int NB = BK * BN / 2 / PT;        // double2 of C staged per thread and tile
    extern __shared__ double2 psf_smem[];
    double2* As = psf_smem;
    double* Bs = (double*)(psf_smem + 2 * BK * AP);
    const int t = threadIdx.x, tx = t % TX, ty = t / TX;
    const int s = blockIdx.z / A.kx, kc = blockIdx.z % A.kx;
    const int row0 = blockIdx.x * BM, col0 = blockIdx.y * BN;
    const int ix0 = kc * A.kx_len, ix1 = min(A.nx, ix0 + A.kx_len);
    const int nk = (ix1 - ix0 + BK - 1) / BK;
    const size_t o = (size_t)s * A.stride;
    const double* opd = A.opd + o;
    const uint8_t* mask = A.mask + o;
    const int lk = t % BK, lr = t / BK;         // the loader's k and first row (rows lr + (PT / BK) q)
    uint8_t m[NQ];                              // mask of the staged elements (0 outside the grid)
    double2 rs = make_double2(0.0, 0.0);
    bool bad = false;

    // stage tile kt into buffer buf: opd into the .x of its P slots and C by cp.async, the mask into m
    auto issue = [&](int kt, int buf) {
        double2* as = As + buf * BK * AP + lk * AP;
        const int ix = ix0 + kt * BK + lk;
#pragma unroll
        for (int q = 0; q < NQ; q++) {
            const int iy = row0 + lr + (PT / BK) * q;
            m[q] = 0;
            if (ix < ix1 && iy < A.ny) {
                const size_t i = (size_t)iy * A.nx + ix;
                m[q] = mask[i];
                cp_async8(&as[lr + (PT / BK) * q].x, opd + i);
            }
        }
        double2* bs = (double2*)(Bs + buf * BK * BN);
#pragma unroll
        for (int q = 0; q < NB; q++) {
            const int e = t + PT * q, k = e / (BN / 2), c2 = e % (BN / 2), ixb = ix0 + kt * BK + k;
            if (ixb < ix1) cp_async16(bs + e, A.ctab + (size_t)ixb * A.nup + col0 + 2 * c2);
            else bs[e] = make_double2(0.0, 0.0);
        }
        cp_async_commit();
    };
    // after the copies of this thread landed: its opd slots of buffer buf become P = mask exp(2 pi i opd)
    auto convert = [&](int buf) {
        cp_async_wait_all();
        double2* as = As + buf * BK * AP + lk * AP;
#pragma unroll
        for (int q = 0; q < NQ; q++) {
            double2 p = make_double2(0.0, 0.0);
            if (m[q] == 1) {
                const double w = as[lr + (PT / BK) * q].x;
                bad |= !isfinite(w);
                sincospi(2.0 * w, &p.y, &p.x);
                rs.x += p.x; rs.y += p.y;
            }
            as[lr + (PT / BK) * q] = p;
        }
    };

    double acc[4][4][4];                        // [row r][column pair c][re x C_even, im x C_even, re x C_odd, im x C_odd]
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int c = 0; c < 4; c++)
#pragma unroll
            for (int h = 0; h < 4; h++) acc[r][c][h] = 0.0;

    if (nk > 0) { issue(0, 0); convert(0); }
    __syncthreads();
    for (int kt = 0; kt < nk; kt++) {
        const int cur = kt & 1;
        if (kt + 1 < nk) issue(kt + 1, cur ^ 1);
        const double2* as = As + cur * BK * AP;
        const double2* bs = (const double2*)(Bs + cur * BK * BN);
#pragma unroll 4
        for (int k = 0; k < BK; k++) {
            double2 a[4], b[4];
#pragma unroll
            for (int r = 0; r < 4; r++) a[r] = as[k * AP + ty + TY * r];
#pragma unroll
            for (int c = 0; c < 4; c++) b[c] = bs[k * (BN / 2) + tx + TX * c];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    acc[r][c][0] = fma(a[r].x, b[c].x, acc[r][c][0]);
                    acc[r][c][1] = fma(a[r].y, b[c].x, acc[r][c][1]);
                    acc[r][c][2] = fma(a[r].x, b[c].y, acc[r][c][2]);
                    acc[r][c][3] = fma(a[r].y, b[c].y, acc[r][c][3]);
                }
        }
        if (kt + 1 < nk) convert(cur ^ 1);
        __syncthreads();
    }

    double2* T = A.T + ((size_t)(s * A.kx + kc) * A.ny) * A.nup;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const int iy = row0 + ty + TY * r;
        if (iy >= A.ny) continue;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int j = col0 + 2 * (tx + TX * c);
            T[(size_t)iy * A.nup + j] = make_double2(acc[r][c][0], acc[r][c][1]);
            T[(size_t)iy * A.nup + j + 1] = make_double2(acc[r][c][2], acc[r][c][3]);
        }
    }

    // sum_ix P of this CTA's rows and ix chunk, folded in a fixed order: lanes, then warps
    bad = __syncthreads_or(bad);
    if (blockIdx.y != 0) return;
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        rs.x += __shfl_xor_sync(0xffffffffu, rs.x, d);
        rs.y += __shfl_xor_sync(0xffffffffu, rs.y, d);
    }
    __shared__ double2 s_rs[PT / 32];
    if ((t & 31) == 0) s_rs[t >> 5] = rs;
    __syncthreads();
    if (t) return;
    for (int q = 1; q < PT / 32; q++) { rs.x += s_rs[q].x; rs.y += s_rs[q].y; }
    double* rec = A.rsum + (((size_t)s * A.rt + blockIdx.x) * A.kx + kc) * 3;
    rec[0] = rs.x; rec[1] = rs.y; rec[2] = bad ? 1.0 : 0.0;
}

// stage B.  16 x 16 threads, each 4 iv rows (stride 16) x 4 complex columns (stride 16).  Shared memory: Ys [2][BK][YB + 1],
// Ts [2][BK][YB] double2, and Tr [kx][BK][YB] double2, where the kx partials of the next T tile land by cp.async; the
// thread that copied a slot also folds it (in chunk order), so Tr needs no second buffer and no barrier of its own.
__global__ void __launch_bounds__(PT, 1) k_psf_y(const __grid_constant__ PsfArgs A)
{
    constexpr int YP = YB + 1;
    extern __shared__ double2 psf_smem[];
    double2* Ys = psf_smem;
    double2* Ts = psf_smem + 2 * BK * YP;
    double2* Tr = Ts + 2 * BK * YB;
    const int t = threadIdx.x, tx = t % 16, ty = t / 16;
    const int s = blockIdx.z, v0 = (blockIdx.x / A.jt) * YB, j0 = (blockIdx.x % A.jt) * YB;
    const int iy0 = blockIdx.y * A.ky_len, iy1 = min(A.ny, iy0 + A.ky_len);
    const int nk = (iy1 - iy0 + BK - 1) / BK;
    const double* ys = A.ys + (size_t)s * A.ys_stride;
    const double ybar = 0.5 * (ys[0] + ys[A.ny - 1]);
    const int lk = t % BK, lr = t / BK;         // the Y loader's k and first row (rows lr + 16 q)
    double eta2s[4];
#pragma unroll
    for (int q = 0; q < 4; q++) eta2s[q] = 2.0 * A.scale * pix(v0 + lr + 16 * q, A.n_v, A.dv);
    double yv = 0.0;
    bool yin = false;
    bool tin[4];

    // stage tile kt: the kx partials of T into Tr by cp.async, y of this thread's k into yv
    auto issue = [&](int kt) {
        const int iy = iy0 + kt * BK + lk;
        yin = iy < iy1;
        if (yin) yv = ys[iy];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = t + PT * q, k = e / YB, c = e % YB, iyb = iy0 + kt * BK + k;
            tin[q] = iyb < iy1;
            if (tin[q])
                for (int kc = 0; kc < A.kx; kc++)
                    cp_async16(Tr + kc * BK * YB + e, A.T + ((size_t)(s * A.kx + kc) * A.ny + iyb) * A.nup + j0 + c);
        }
        cp_async_commit();
    };
    // after this thread's copies landed: Y of its slots and the folded T into buffer buf
    auto convert = [&](int buf) {
        cp_async_wait_all();
        double2* ysm = Ys + buf * BK * YP + lk * YP;
        const double dy = yv - ybar;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            double2 y = make_double2(0.0, 0.0);
            if (yin) sincospi(dy * eta2s[q], &y.y, &y.x);
            ysm[lr + 16 * q] = y;
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = t + PT * q;
            double2 v = make_double2(0.0, 0.0);
            if (tin[q])
                for (int kc = 0; kc < A.kx; kc++) {
                    const double2 p = Tr[kc * BK * YB + e];
                    v.x += p.x; v.y += p.y;
                }
            Ts[buf * BK * YB + e] = v;
        }
    };

    double2 acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[r][c] = make_double2(0.0, 0.0);

    if (nk > 0) { issue(0); convert(0); }
    __syncthreads();
    for (int kt = 0; kt < nk; kt++) {
        const int cur = kt & 1;
        if (kt + 1 < nk) issue(kt + 1);
        const double2* ysm = Ys + cur * BK * YP;
        const double2* tsm = Ts + cur * BK * YB;
#pragma unroll 4
        for (int k = 0; k < BK; k++) {
            double2 a[4], b[4];
#pragma unroll
            for (int r = 0; r < 4; r++) a[r] = ysm[k * YP + ty + 16 * r];
#pragma unroll
            for (int c = 0; c < 4; c++) b[c] = tsm[k * YB + tx + 16 * c];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    acc[r][c].x = fma(a[r].x, b[c].x, acc[r][c].x);
                    acc[r][c].x = fma(-a[r].y, b[c].y, acc[r][c].x);
                    acc[r][c].y = fma(a[r].x, b[c].y, acc[r][c].y);
                    acc[r][c].y = fma(a[r].y, b[c].x, acc[r][c].y);
                }
        }
        if (kt + 1 < nk) convert(cur ^ 1);
        __syncthreads();
    }

    double2* E = A.E + ((size_t)s * A.ky + blockIdx.y) * A.n_v * A.nuh;
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const int iv = v0 + ty + 16 * r;
        if (iv >= A.n_v) continue;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int j = j0 + tx + 16 * c;
            if (j < A.nuh) E[(size_t)iv * A.nuh + j] = acc[r][c];
        }
    }
}

// the status of set s from its k_psf_x records (every CTA of the set reads them: a few hundred flags)
__device__ int fold_status(const PsfArgs& A, int s)
{
    const int nrec = A.rt * A.kx;
    const double* rec = A.rsum + (size_t)s * nrec * 3;
    bool bad = false;
    for (int i = threadIdx.x; i < nrec; i += blockDim.x) bad |= rec[3 * i + 2] != 0.0;
    return set_status(A, s, __syncthreads_or(bad));
}

__device__ __forceinline__ bool better(double v, int i, double bv, int bi) { return v > bv || (v == bv && i < bi); }

__global__ void __launch_bounds__(PT) k_psf_fold(const __grid_constant__ PsfArgs A)
{
    __shared__ double s_v[PT];
    __shared__ int s_i[PT];
    const int s = blockIdx.y, t = threadIdx.x;
    const int st = fold_status(A, s);
    const long long n = A.stats[s].n_kept;
    const double norm = 4.0 * (double)n * (double)n;
    const int npix = A.n_v * A.nuh;
    const double2* E = A.E + (size_t)s * A.ky * npix;
    double* psf = A.psf + (size_t)s * A.n_v * A.n_u;
    double bv = -INFINITY;
    int bi = INT_MAX;
    for (int p = blockIdx.x * PT + t; p < npix; p += gridDim.x * PT) {
        const int iv = p / A.nuh, j = p % A.nuh;
        const int iu = A.n_u - A.nuh + j, iu_m = A.n_u - 1 - iu;
        double v = psf_nan();
        if (st == 0) {
            double er = 0.0, ei = 0.0;
            for (int k = 0; k < A.ky; k++) { const double2 e = E[(size_t)k * npix + p]; er += e.x; ei += e.y; }
            v = (er * er + ei * ei) / norm;
            const int idx = iv * A.n_u + iu_m;
            if (better(v, idx, bv, bi)) { bv = v; bi = idx; }
        }
        psf[(size_t)iv * A.n_u + iu] = v;
        psf[(size_t)iv * A.n_u + iu_m] = v;
    }
    s_v[t] = bv; s_i[t] = bi;
    __syncthreads();
    if (t) return;
    for (int q = 1; q < PT; q++)
        if (better(s_v[q], s_i[q], bv, bi)) { bv = s_v[q]; bi = s_i[q]; }
    A.bval[(size_t)s * gridDim.x + blockIdx.x] = bv;
    A.bidx[(size_t)s * gridDim.x + blockIdx.x] = bi;
}

__global__ void __launch_bounds__(PT) k_psf_peak(const __grid_constant__ PsfArgs A)
{
    __shared__ double2 s_rs[PT];
    const int s = blockIdx.x, t = threadIdx.x;
    const int st = fold_status(A, s);
    const int nrec = A.rt * A.kx;
    const double* rec = A.rsum + (size_t)s * nrec * 3;
    double2 rs = make_double2(0.0, 0.0);
    for (int i = t; i < nrec; i += PT) { rs.x += rec[3 * i]; rs.y += rec[3 * i + 1]; }
    s_rs[t] = rs;
    __syncthreads();
    if (t) return;
    for (int q = 1; q < PT; q++) { rs.x += s_rs[q].x; rs.y += s_rs[q].y; }
    double bv = -INFINITY;
    int bi = INT_MAX;
    for (int b = 0; b < A.fb; b++) {
        const double v = A.bval[(size_t)s * A.fb + b];
        const int i = A.bidx[(size_t)s * A.fb + b];
        if (better(v, i, bv, bi)) { bv = v; bi = i; }
    }
    const double n = (double)A.stats[s].n_kept;
    A.strehl[2 * s] = st ? psf_nan() : (rs.x * rs.x + rs.y * rs.y) / (n * n);
    A.strehl[2 * s + 1] = st ? psf_nan() : bv;
    A.peak[s] = st ? -1 : bi;
    A.status[s] = st;
}

template <int TX>
size_t x_smem() { return sizeof(double2) * 2 * BK * (4 * (PT / TX) + 1) + sizeof(double) * 2 * BK * 8 * TX; }
size_t y_smem(int kx) { return sizeof(double2) * (2 * BK * (2 * YB + 1) + (size_t)kx * BK * YB); }

// the chunk count in [1, max_chunks] that least lengthens the last CTA wave of `tiles` x chunks CTAs; ties to fewer chunks
int chunks(long long tiles, int slots, int max_chunks)
{
    int best = 1;
    double best_t = 1e300;
    for (int c = 1; c <= max_chunks; c++) {
        const double waves = (double)((tiles * c + slots - 1) / slots) / c;
        if (waves < 0.95 * best_t) { best_t = waves; best = c; }
    }
    return best;
}

}  // namespace

cudaError_t psf_dims(PsfArgs& A, int sm_count)
{
    A.nuh = (A.n_u + 1) / 2;
    A.tx = A.nuh <= 64 ? 8 : 16;
    const int BM = 4 * (PT / A.tx), BN = 8 * A.tx;
    A.nup = (A.nuh + BN - 1) / BN * BN;
    A.rt = (A.ny + BM - 1) / BM;
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_psf_x<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)x_smem<8>())) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_psf_x<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)x_smem<16>())) != cudaSuccess ||
        (e = cudaFuncSetAttribute(k_psf_y, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)y_smem(MAX_KX))) != cudaSuccess)
        return e;
    int occ_x = 0, occ_y = 0;
    if (A.tx == 8) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_x, k_psf_x<8>, PT, x_smem<8>());
    else e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_x, k_psf_x<16>, PT, x_smem<16>());
    if (e != cudaSuccess) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_y, k_psf_y, PT, y_smem(MAX_KX))) != cudaSuccess) return e;
    const int slots_x = sm_count * (occ_x > 0 ? occ_x : 1), slots_y = sm_count * (occ_y > 0 ? occ_y : 1);
    // stage A: chunks of the ix range, each a whole number of tiles and none empty
    const int kt_x = (A.nx + BK - 1) / BK;
    int kx = chunks((long long)A.rt * (A.nup / BN) * A.n_sets, slots_x, kt_x < MAX_KX ? kt_x : MAX_KX);
    A.kx_len = (kt_x + kx - 1) / kx * BK;
    A.kx = (A.nx + A.kx_len - 1) / A.kx_len;
    // stage B: chunks of the iy range, as for stage A
    A.jt = (A.nuh + YB - 1) / YB;
    A.vt = (A.n_v + YB - 1) / YB;
    const int kt_y = (A.ny + BK - 1) / BK;
    const int ky = chunks((long long)A.vt * A.jt * A.n_sets, slots_y, kt_y < MAX_KY ? kt_y : MAX_KY);
    A.ky_len = (kt_y + ky - 1) / ky * BK;
    A.ky = (A.ny + A.ky_len - 1) / A.ky_len;
    // fold: about two CTAs per SM over all sets
    const long long fb = (2LL * sm_count + A.n_sets - 1) / A.n_sets, fmax = ((long long)A.n_v * A.nuh + PT - 1) / PT;
    A.fb = (int)(fb < fmax ? fb : fmax);
    return cudaSuccess;
}

cudaError_t launch_psf(const PsfArgs& A, cudaStream_t st, int* launches)
{
    const long long nt = (long long)A.nx * A.nup;
    k_psf_table<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(A);
    const dim3 gx((unsigned)A.rt, (unsigned)(A.nup / (8 * A.tx)), (unsigned)(A.n_sets * A.kx));
    if (A.tx == 8) k_psf_x<8><<<gx, PT, x_smem<8>(), st>>>(A);
    else k_psf_x<16><<<gx, PT, x_smem<16>(), st>>>(A);
    k_psf_y<<<dim3((unsigned)(A.vt * A.jt), (unsigned)A.ky, (unsigned)A.n_sets), PT, y_smem(A.kx), st>>>(A);
    k_psf_fold<<<dim3((unsigned)A.fb, (unsigned)A.n_sets), PT, 0, st>>>(A);
    k_psf_peak<<<A.n_sets, PT, 0, st>>>(A);
    *launches = 5;
    return cudaGetLastError();
}
