// kern_energy.cu -- geometric encircled / ensquared energy of the spot (ort_spot_energy_dev, include/ort_b200.h).
//
// Every kept ray of a set has a distance d from the centre.  The curve counts d <= radii[k]; the energy radius is the
// k-th smallest d, found by an exact radix select on 63-bit keys: the bit pattern of d with the sign bit cleared, which
// orders non-negative doubles like uint64 and puts a NaN after +Inf.  Six digits, high to low:
//
//   pass  key bits   buckets   reads
//   0     62..51     4096      the sweep outputs (ex, ey and the mask or the compacted count); also bins the radii
//   1     50..40     2048      per fraction: the candidate list if one was written, else the sweep outputs again
//   2..4  39..7      2048      the same
//   5     6..0        128      the same
//
// After each pass k_energy_select picks, per (set, fraction), the bucket that holds the remaining rank.  It then knows
// how many keys the next pass keeps -- the sum of the picked buckets -- and, when that fits the candidate list
// (energy_cand_cap), the next pass appends exactly those keys to it, so the passes after it read 8 bytes per candidate
// instead of the sweep outputs.  A set of at most `cap` kept rays writes all its keys in pass 0.  Nothing comes back to
// the host: the launch sequence is fixed (13 kernels) and the state lives in device scratch.  Integer atomics only, so
// every result is bit-reproducible.
#include "kern.cuh"

namespace {

constexpr int EN_THREADS = 256;
constexpr int EN_UNROLL = 4;                        // rays per thread per tile
constexpr int EN_TILE = EN_THREADS * EN_UNROLL;
constexpr int EN_PASSES = 6;
constexpr int EN_BUCKETS0 = 4096;                   // pass 0: one histogram per set, shared by the fractions
constexpr int EN_BUCKETS = 2048;                    // passes 1..5: one histogram per (set, fraction)
constexpr unsigned long long EN_KEY = 0x7fffffffffffffffull;

struct EnergyRadii { double r[ORT_MAX_RADII]; };

// key bits [lo, hi) are pass p's digit; the prefix already selected is key >> hi
__device__ __forceinline__ int pass_lo(int p) { return p == 0 ? 51 : max(51 - 11 * p, 0); }
__device__ __forceinline__ int pass_hi(int p) { return p == 0 ? 63 : pass_lo(p - 1); }

__device__ __forceinline__ size_t hist_words(int n_fracs)
{
    return (size_t)max(EN_BUCKETS0, n_fracs * EN_BUCKETS);
}

// the distance of the header, operation for operation (no contraction)
__device__ __forceinline__ double energy_d(double ex, double ey, double cy, int metric)
{
    const double dy = __dadd_rn(ey, -cy);
    if (metric == ORT_ENERGY_CIRCLE) return __dsqrt_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(dy, dy)));
    const double a = fabs(ex), b = fabs(dy);
    return (a >= b || a != a) ? a : b;              // numpy.maximum: NaN if either is
}

__device__ __forceinline__ unsigned long long energy_key(double d)
{
    return (unsigned long long)__double_as_longlong(d) & EN_KEY;
}

__device__ __forceinline__ double set_centre(const EnergyArgs& A, int s)
{
    return A.center == ORT_CENTER_CENTROID ? A.stats[s].mean_y : 0.0;
}

// rays of set s this CTA owns: f(key, d, kept) for EN_UNROLL rays per thread and tile.  Every thread of the CTA takes the
// same steps, so f may use warp-collective operations.
template <class F>
__device__ __forceinline__ void for_each_ray(const EnergyArgs& A, int s, long long len, F&& f)
{
    const double* ex = A.ex + (size_t)s * A.stride;
    const double* ey = A.ey + (size_t)s * A.stride;
    const uint8_t* mask = A.mask ? A.mask + (size_t)(s / A.sets_per_mask) * A.stride : nullptr;
    const double cy = set_centre(A, s);
    for (long long t0 = (long long)blockIdx.x * EN_TILE; t0 < len; t0 += (long long)gridDim.x * EN_TILE) {
        bool kept[EN_UNROLL];
        double x[EN_UNROLL], y[EN_UNROLL];
#pragma unroll
        for (int u = 0; u < EN_UNROLL; u++) {
            const long long i = t0 + u * EN_THREADS + threadIdx.x;
            kept[u] = i < len && (!mask || mask[i] == 1);
        }
#pragma unroll
        for (int u = 0; u < EN_UNROLL; u++) {
            const long long i = t0 + u * EN_THREADS + threadIdx.x;
            x[u] = kept[u] ? ex[i] : 0.0;
            y[u] = kept[u] ? ey[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < EN_UNROLL; u++) {
            const double d = energy_d(x[u], y[u], cy, A.metric);
            f(energy_key(d), d, kept[u]);
        }
    }
}

// the same over a candidate list of n keys
template <class F>
__device__ __forceinline__ void for_each_cand(const unsigned long long* list, unsigned n, F&& f)
{
    for (long long t0 = (long long)blockIdx.x * EN_TILE; t0 < n; t0 += (long long)gridDim.x * EN_TILE) {
        unsigned long long k[EN_UNROLL];
#pragma unroll
        for (int u = 0; u < EN_UNROLL; u++) {
            const long long i = t0 + u * EN_THREADS + threadIdx.x;
            k[u] = i < n ? list[i] : 0ull;
        }
#pragma unroll
        for (int u = 0; u < EN_UNROLL; u++) f(k[u], 0.0, t0 + u * EN_THREADS + threadIdx.x < n);
    }
}

// warp-aggregated append of the keys with `want` to a candidate list (order is irrelevant: only counts are taken from it).
// The select kernel sized the list from the histograms; `cap` only guards against statistics that disagree with the mask.
__device__ __forceinline__ void append(unsigned long long* list, unsigned* cnt, unsigned cap, unsigned long long key,
                                       bool want)
{
    const unsigned b = __ballot_sync(0xffffffffu, want);
    if (!b) return;
    const int lane = threadIdx.x & 31, first = __ffs(b) - 1;
    unsigned base = 0;
    if (lane == first) base = atomicAdd(cnt, (unsigned)__popc(b));
    base = __shfl_sync(0xffffffffu, base, first);
    const unsigned i = base + __popc(b & ((1u << lane) - 1u));
    if (want && i < cap) list[i] = key;
}

// one CTA per set: the selection state, and zero histograms and bins
__global__ void __launch_bounds__(EN_THREADS) k_energy_init(const __grid_constant__ EnergyArgs A)
{
    const int s = blockIdx.x;
    const size_t hw = hist_words(A.n_fracs);
    for (size_t i = threadIdx.x; i < hw; i += EN_THREADS) A.hist[(size_t)s * hw + i] = 0u;
    if (A.n_radii)
        for (int i = threadIdx.x; i <= A.n_radii; i += EN_THREADS) A.bins[(size_t)s * (A.n_radii + 1) + i] = 0ull;
    if (threadIdx.x) return;
    EnergyState& S = A.state[s];
    const long long n = A.stats[s].n_kept;
    S.n = n; S.src = -1; S.src_n = 0; S.cnt = 0; S.active = 0; S.pad = 0;
    for (int f = 0; f < ORT_MAX_FRACS; f++) {
        long long k = 1;
        if (f < A.n_fracs && n > 0) {
            const double kq = ceil(__dmul_rn(A.fracs[f], (double)n));
            k = kq < 1.0 ? 1 : kq > (double)n ? n : (long long)kq;
            S.active |= 1 << f;
        }
        S.prefix[f] = 0ull; S.rank[f] = (unsigned long long)(k - 1);
    }
    S.dst = (S.active && n <= (long long)A.cap) ? 0 : -1;
}

// pass 0: d of every kept ray, its radius bin (the first radius >= d; n_radii: none) and the first digit of its key
__global__ void __launch_bounds__(EN_THREADS, 4)
k_energy_bin(const __grid_constant__ EnergyArgs A, const __grid_constant__ EnergyRadii RR)
{
    extern __shared__ double en_smem[];
    const int s = blockIdx.y, R = A.n_radii;
    const EnergyState& S = A.state[s];
    const bool sel = S.active != 0;
    if (!R && !sel) return;
    double* s_r = en_smem;
    unsigned* s_h = (unsigned*)(s_r + R);
    unsigned* s_b = s_h + EN_BUCKETS0;
    for (int i = threadIdx.x; i < R; i += EN_THREADS) s_r[i] = RR.r[i];
    for (int i = threadIdx.x; i < EN_BUCKETS0; i += EN_THREADS) s_h[i] = 0u;
    for (int i = threadIdx.x; i <= R; i += EN_THREADS) s_b[i] = 0u;
    __syncthreads();
    const long long len = A.mask ? A.stride : min(S.n, A.stride);
    unsigned long long* out = S.dst >= 0 ? A.cand[S.dst] + (size_t)s * A.cap : nullptr;
    unsigned* cnt = &A.state[s].cnt;
    for_each_ray(A, s, len, [&](unsigned long long key, double d, bool kept) {
        if (kept && R) {
            int lo = 0, hi = R;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (d <= s_r[mid]) hi = mid; else lo = mid + 1;
            }
            atomicAdd(&s_b[lo], 1u);
        }
        if (kept && sel) atomicAdd(&s_h[key >> 51], 1u);
        if (out) append(out, cnt, A.cap, key, kept);
    });
    __syncthreads();
    for (int i = threadIdx.x; i <= R; i += EN_THREADS)
        if (s_b[i]) atomicAdd(&A.bins[(size_t)s * (R + 1) + i], (unsigned long long)s_b[i]);
    if (sel) {
        unsigned* h = A.hist + (size_t)s * hist_words(A.n_fracs);
        for (int i = threadIdx.x; i < EN_BUCKETS0; i += EN_THREADS)
            if (s_h[i]) atomicAdd(&h[i], s_h[i]);
    }
}

// pass p = 1..5: per fraction, the digit histogram of the keys that carry its prefix; appends the keys that carry any
// fraction's prefix to candidate list dst when k_energy_select asked for it
__global__ void __launch_bounds__(EN_THREADS, 3) k_energy_refine(const __grid_constant__ EnergyArgs A, int p)
{
    extern __shared__ unsigned en_hist[];
    __shared__ unsigned long long s_pf[ORT_MAX_FRACS];
    const int s = blockIdx.y, Q = A.n_fracs;
    const EnergyState& S = A.state[s];
    const int active = S.active;
    if (!active) return;
    const int lo = pass_lo(p), hi = pass_hi(p);
    const unsigned long long dmask = (1ull << (hi - lo)) - 1ull;
    if (threadIdx.x < ORT_MAX_FRACS) s_pf[threadIdx.x] = S.prefix[threadIdx.x];
    for (int i = threadIdx.x; i < Q * EN_BUCKETS; i += EN_THREADS) en_hist[i] = 0u;
    __syncthreads();
    unsigned long long* out = S.dst >= 0 ? A.cand[S.dst] + (size_t)s * A.cap : nullptr;
    unsigned* cnt = &A.state[s].cnt;
    auto body = [&](unsigned long long key, double, bool kept) {
        bool any = false;
        if (kept)
            for (int f = 0; f < Q; f++)
                if (((active >> f) & 1) && (key >> hi) == s_pf[f]) {
                    atomicAdd(&en_hist[f * EN_BUCKETS + (int)((key >> lo) & dmask)], 1u);
                    any = true;
                }
        if (out) append(out, cnt, A.cap, key, any);
    };
    if (S.src >= 0) for_each_cand(A.cand[S.src] + (size_t)s * A.cap, S.src_n, body);
    else for_each_ray(A, s, A.mask ? A.stride : min(S.n, A.stride), body);
    __syncthreads();
    unsigned* h = A.hist + (size_t)s * hist_words(Q);
    for (int i = threadIdx.x; i < Q * EN_BUCKETS; i += EN_THREADS)
        if (en_hist[i]) atomicAdd(&h[i], en_hist[i]);
}

// one CTA per set after pass p: the bucket that holds each fraction's rank, the size of the next candidate list, and
// zeroed histograms for the next pass.  After pass 0 it also writes the curve, after the last pass the radii.
__global__ void __launch_bounds__(EN_THREADS) k_energy_select(const __grid_constant__ EnergyArgs A, int p)
{
    __shared__ unsigned long long s_sum[EN_THREADS];
    __shared__ unsigned long long s_pf[ORT_MAX_FRACS], s_rank[ORT_MAX_FRACS], s_cnt[ORT_MAX_FRACS];
    __shared__ int s_active;
    const int s = blockIdx.x, t = threadIdx.x, Q = A.n_fracs, R = A.n_radii;
    EnergyState& S = A.state[s];
    if (p == 0 && R && t == 0) {
        const unsigned long long* b = A.bins + (size_t)s * (R + 1);
        long long c = 0;
        for (int k = 0; k < R; k++) { c += (long long)b[k]; A.counts[(size_t)s * R + k] = c; }
    }
    if (!Q) return;
    const int lo = pass_lo(p), w = pass_hi(p) - lo, nb = 1 << w;
    const int chunk = (nb + EN_THREADS - 1) / EN_THREADS;
    const int b0 = min(t * chunk, nb), b1 = min(b0 + chunk, nb);
    const size_t hw = hist_words(Q);
    unsigned* hist = A.hist + (size_t)s * hw;
    if (t == 0) s_active = S.active;
    if (t < ORT_MAX_FRACS) { s_pf[t] = S.prefix[t]; s_rank[t] = S.rank[t]; s_cnt[t] = 0; }
    __syncthreads();
    const int active = s_active;
    for (int f = 0; f < Q; f++) {
        if (!((active >> f) & 1)) continue;
        const unsigned* h = hist + (p == 0 ? 0 : f * EN_BUCKETS);
        unsigned long long mine = 0;
        for (int b = b0; b < b1; b++) mine += h[b];
        s_sum[t] = mine;
        __syncthreads();
        for (int off = 1; off < EN_THREADS; off <<= 1) {         // inclusive scan
            const unsigned long long v = t >= off ? s_sum[t - off] : 0ull;
            __syncthreads();
            s_sum[t] += v;
            __syncthreads();
        }
        const unsigned long long r = s_rank[f], incl = s_sum[t], excl = incl - mine;
        if (r >= s_sum[EN_THREADS - 1]) {                       // fewer keys than the statistics record: no radius
            if (t == 0) atomicAnd(&s_active, ~(1 << f));
        } else if (excl <= r && r < incl) {
            unsigned long long c = excl;
            for (int b = b0; b < b1; b++) {
                if (r < c + h[b]) {
                    s_pf[f] = (s_pf[f] << w) | (unsigned long long)b;
                    s_rank[f] = r - c;
                    s_cnt[f] = h[b];
                    break;
                }
                c += h[b];
            }
        }
        __syncthreads();
    }
    for (size_t i = t; i < hw; i += EN_THREADS) hist[i] = 0u;
    if (t) return;
    const int act = s_active;
    S.active = act;
    for (int f = 0; f < ORT_MAX_FRACS; f++) { S.prefix[f] = s_pf[f]; S.rank[f] = s_rank[f]; }
    if (S.dst >= 0) { S.src = S.dst; S.src_n = min(S.cnt, A.cap); }
    unsigned long long next = 0;                                // keys that carry a picked prefix, each counted once
    for (int f = 0; f < Q; f++) {
        if (!((act >> f) & 1)) continue;
        bool seen = false;
        for (int g = 0; g < f; g++) seen |= ((act >> g) & 1) && s_pf[g] == s_pf[f];
        if (!seen) next += s_cnt[f];
    }
    if (p + 1 < EN_PASSES && act && next <= A.cap) { S.dst = S.src == 0 ? 1 : 0; S.cnt = 0; }
    else S.dst = -1;
    if (p + 1 == EN_PASSES)
        for (int f = 0; f < Q; f++)
            A.radius[(size_t)s * Q + f] = ((act >> f) & 1) ? __longlong_as_double((long long)s_pf[f]) : __longlong_as_double(0x7ff8000000000000ll);
}

}  // namespace

size_t energy_hist_words(int n_fracs)
{
    return (size_t)(n_fracs * EN_BUCKETS > EN_BUCKETS0 ? n_fracs * EN_BUCKETS : EN_BUCKETS0);
}

// Candidate-list capacity per set: the whole set up to 2^22 keys, and at most 2^26 keys (512 MB) per list over all sets
unsigned energy_cand_cap(long long stride, int n_sets)
{
    long long cap = stride < (1ll << 22) ? stride : (1ll << 22);
    const long long share = (1ll << 26) / (n_sets > 0 ? n_sets : 1);
    if (cap > share) cap = share;
    return (unsigned)(cap > 0 ? cap : 0);
}

cudaError_t launch_energy(const EnergyArgs& A, const double* radii, int sm_count, cudaStream_t st, int* launches)
{
    EnergyRadii RR;
    memset(&RR, 0, sizeof RR);
    if (A.n_radii) memcpy(RR.r, radii, sizeof(double) * (size_t)A.n_radii);
    const size_t smem0 = sizeof(double) * A.n_radii + sizeof(unsigned) * (EN_BUCKETS0 + A.n_radii + 1);
    const size_t smem1 = sizeof(unsigned) * EN_BUCKETS * (size_t)A.n_fracs;
    cudaError_t e = cudaFuncSetAttribute(k_energy_refine, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(sizeof(unsigned) * EN_BUCKETS * ORT_MAX_FRACS));
    if (e != cudaSuccess) return e;
    // CTAs per set: about 8 resident per SM over all sets, no more than the tiles of the largest set
    long long gx = ((long long)sm_count * 8) / A.n_sets;
    const long long tiles = (A.stride + EN_TILE - 1) / EN_TILE;
    if (gx > tiles) gx = tiles;
    if (gx < 1) gx = 1;
    const dim3 grid((unsigned)gx, (unsigned)A.n_sets);
    k_energy_init<<<A.n_sets, EN_THREADS, 0, st>>>(A);
    k_energy_bin<<<grid, EN_THREADS, smem0, st>>>(A, RR);
    k_energy_select<<<A.n_sets, EN_THREADS, 0, st>>>(A, 0);
    for (int p = 1; p < EN_PASSES; p++) {
        k_energy_refine<<<grid, EN_THREADS, smem1, st>>>(A, p);
        k_energy_select<<<A.n_sets, EN_THREADS, 0, st>>>(A, p);
    }
    *launches = 1 + 2 * EN_PASSES;
    return cudaGetLastError();
}
