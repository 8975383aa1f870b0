// ort_comm.cu -- the communicator behind the C ABI (include/ort_b200.h, "communicator inside the library") and the
// sharded sweeps built on it.
//
// The path shards without a data-path collective: rays are independent (src/PupilSampling.jl:123-138 has no
// cross-iteration state except the push! order), so every rank traces a contiguous block of y-rows -- or a contiguous
// range of candidate prescriptions -- and exactly one exchange follows: an all-gather of the n_fields x 112 B statistics
// records (merged in rank order by k_merge_stats, so sigma of :169-173 is bit-identical on every rank), or of the
// 32 B-per-candidate merit table.  Both run on the stream of the sweep, right behind its last kernel.
//
// NCCL is resolved with dlopen on first use: the library itself has no link-time dependency on it, loads on machines
// without it, and shares the process's libnccl.so.2 with whatever else uses NCCL there (e.g. torch.distributed).
#include <dlfcn.h>
#include <math.h>
#include <stdlib.h>

#include <mutex>

#include <nccl.h>

#include "ort_ctx.cuh"

namespace {

struct Nccl {
    void* h;
    ncclResult_t (*GetVersion)(int*);
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)(void);
    ncclResult_t (*GroupEnd)(void);
    const char* (*GetErrorString)(ncclResult_t);
    char why[384];
    bool ok;
};

Nccl g_nccl;
std::once_flag g_nccl_once;

void nccl_load()
{
    Nccl& N = g_nccl;
    memset(&N, 0, sizeof N);
    const char* env = getenv("ORT_NCCL_LIB");
    const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        if (!nm || !*nm) continue;
        N.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (N.h) break;
        snprintf(N.why, sizeof N.why, "dlopen(%s): %s", nm, dlerror());
    }
    if (!N.h) return;
#define SYM(field, name)                                                                          \
    do { *(void**)(&N.field) = dlsym(N.h, name);                                                  \
         if (!N.field) { snprintf(N.why, sizeof N.why, "dlsym(%s) failed", name); return; } } while (0)
    SYM(GetVersion, "ncclGetVersion"); SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommInitAll, "ncclCommInitAll"); SYM(CommDestroy, "ncclCommDestroy"); SYM(AllGather, "ncclAllGather");
    SYM(Broadcast, "ncclBroadcast"); SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    N.ok = true;
}

Nccl* nccl()
{
    std::call_once(g_nccl_once, nccl_load);
    return &g_nccl;
}

#define NCK(call)                                                                                  \
    do {                                                                                           \
        ncclResult_t r_ = (call);                                                                  \
        if (r_ != ncclSuccess)                                                                     \
            return fail(ctx, ORT_ENCCL, "%s:%d %s -> %s", __FILE__, __LINE__, #call, N->GetErrorString(r_)); \
    } while (0)
#define NEED_NCCL(N)                                                                               \
    Nccl* N = nccl();                                                                              \
    if (!N->ok) return fail(ctx, ORT_ENCCL, "NCCL is not available: %s", N->why[0] ? N->why : "libnccl.so.2 not found")

// Rank-order Chan merge of the gathered records, one thread per field: the same operations, in the same order and
// never contracted, as the host function ort_merge_stats -- every rank folds the same bytes the same way, so the
// merged records (hence sigma) are bit-identical everywhere.
__global__ void k_merge_stats(const ort_stats* recs, int n_shards, int n_fields, ort_stats* out)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_fields) return;
    ort_stats a;
    a.n_kept = 0; a.mean_x = a.mean_y = a.m2_x = a.m2_y = a.mean_opd = a.m2_opd = 0.0; a.r_max = -CUDART_INF;
    a.n_miss = a.n_tir = a.n_domain = a.n_clip = a.n_vig = a.n_strict = 0;
    for (int r = 0; r < n_shards; r++) {
        const ort_stats b = recs[(size_t)r * n_fields + f];
        a.n_miss += b.n_miss; a.n_tir += b.n_tir; a.n_domain += b.n_domain; a.n_clip += b.n_clip; a.n_vig += b.n_vig;
        a.n_strict += b.n_strict;
        if (b.n_kept == 0) continue;
        if (a.n_kept == 0) {
            a.n_kept = b.n_kept; a.mean_x = b.mean_x; a.mean_y = b.mean_y; a.m2_x = b.m2_x; a.m2_y = b.m2_y;
            a.r_max = b.r_max; a.mean_opd = b.mean_opd; a.m2_opd = b.m2_opd;
            continue;
        }
        const double na = (double)a.n_kept, nb = (double)b.n_kept, n = SA(na, nb), w = SD(nb, n), naw = SM(na, w);
        const double dx = SS(b.mean_x, a.mean_x), dy = SS(b.mean_y, a.mean_y), dd = SS(b.mean_opd, a.mean_opd);
        a.mean_x = SA(a.mean_x, SM(dx, w)); a.m2_x = SA(SA(a.m2_x, b.m2_x), SM(SM(dx, dx), naw));
        a.mean_y = SA(a.mean_y, SM(dy, w)); a.m2_y = SA(SA(a.m2_y, b.m2_y), SM(SM(dy, dy), naw));
        a.mean_opd = SA(a.mean_opd, SM(dd, w)); a.m2_opd = SA(SA(a.m2_opd, b.m2_opd), SM(SM(dd, dd), naw));
        a.n_kept += b.n_kept;
        if (b.r_max > a.r_max) a.r_max = b.r_max;
    }
    out[f] = a;
}

int merge_enqueue(ort_ctx* ctx, const ort_stats* d_ranks, int n_shards, int n_fields, ort_stats* d_merged, cudaStream_t st)
{
    k_merge_stats<<<1, ORT_MAX_FIELDS, 0, st>>>(d_ranks, n_shards, n_fields, d_merged);
    CK(cudaGetLastError());
    ctx->launches++;
    return ORT_OK;
}

void comm_range(long long total, int rank, int world, long long* lo, long long* hi)
{
    const long long base = total / world, rem = total % world;
    *lo = rank * base + (rank < rem ? rank : rem);
    *hi = *lo + base + (rank < rem ? 1 : 0);
}

}  // namespace

// One rank of a multi-process communicator: all-gather behind the statistics kernel, then the merge.
int ort_comm_gather_stats(ort_ctx* ctx, const ort_stats* d_local, int n_fields, ort_stats* d_merged, ort_stats* d_ranks,
                          cudaStream_t st)
{
    if (!ctx->comm) return fail(ctx, ORT_ENCCL, "gather_stats: no communicator");
    NEED_NCCL(N);
    if (!d_ranks) ENSURE(SL_GATHER, sizeof(ort_stats) * (size_t)n_fields * ctx->comm_world, d_ranks);
    NCK(N->AllGather(d_local, d_ranks, sizeof(ort_stats) * (size_t)n_fields, ncclChar, (ncclComm_t)ctx->comm, st));
    return merge_enqueue(ctx, d_ranks, ctx->comm_world, n_fields, d_merged, st);
}

extern "C" {

int ort_comm_unique_id(void* id)
{
    ort_ctx* ctx = nullptr;
    if (!id) return fail(ctx, ORT_EINVAL, "ort_comm_unique_id: id is NULL");
    NEED_NCCL(N);
    static_assert(sizeof(ncclUniqueId) == ORT_COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId u;
    NCK(N->GetUniqueId(&u));
    memcpy(id, &u, sizeof u);
    return ORT_OK;
}

int ort_comm_init_rank(ort_ctx* ctx, const void* id, int rank, int world)
{
    if (!ctx) return ORT_EINVAL;
    if (!id || world < 1 || rank < 0 || rank >= world) return fail(ctx, ORT_EINVAL, "ort_comm_init_rank: rank %d of %d", rank, world);
    if (ctx->comm) return fail(ctx, ORT_EINVAL, "ort_comm_init_rank: the context already has a communicator (ort_comm_free first)");
    NEED_NCCL(N);
    CK(cudaSetDevice(ctx->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof u);
    ncclComm_t c = nullptr;
    NCK(N->CommInitRank(&c, world, u, rank));
    ctx->comm = c; ctx->comm_rank = rank; ctx->comm_world = world;
    return ORT_OK;
}

int ort_comm_init_all(ort_ctx** ctxs, int n)
{
    ort_ctx* ctx = ctxs ? ctxs[0] : nullptr;
    if (!ctxs || n < 1 || n > ORT_MAX_GPUS) return fail(ctx, ORT_EINVAL, "ort_comm_init_all: n = %d not in [1, %d]", n, ORT_MAX_GPUS);
    int devs[ORT_MAX_GPUS];
    for (int i = 0; i < n; i++) {
        if (!ctxs[i]) return fail(ctx, ORT_EINVAL, "ort_comm_init_all: ctxs[%d] is NULL", i);
        if (ctxs[i]->comm) return fail(ctx, ORT_EINVAL, "ort_comm_init_all: ctxs[%d] already has a communicator", i);
        devs[i] = ctxs[i]->device;
        for (int j = 0; j < i; j++)
            if (devs[j] == devs[i]) return fail(ctx, ORT_EINVAL, "ort_comm_init_all: ctxs[%d] and ctxs[%d] share device %d", j, i, devs[i]);
    }
    NEED_NCCL(N);
    ncclComm_t comms[ORT_MAX_GPUS];
    NCK(N->CommInitAll(comms, n, devs));
    for (int i = 0; i < n; i++) { ctxs[i]->comm = comms[i]; ctxs[i]->comm_rank = i; ctxs[i]->comm_world = n; }
    return ORT_OK;
}

int ort_comm_info(ort_ctx* ctx, int* rank, int* world, int* nccl_version)
{
    if (!ctx) return ORT_EINVAL;
    if (rank) *rank = ctx->comm ? ctx->comm_rank : 0;
    if (world) *world = ctx->comm ? ctx->comm_world : 0;
    if (nccl_version) {
        *nccl_version = 0;
        Nccl* N = nccl();
        if (N->ok) N->GetVersion(nccl_version);
    }
    return ORT_OK;
}

int ort_comm_free(ort_ctx* ctx)
{
    if (!ctx) return ORT_EINVAL;
    if (ctx->comm) {
        Nccl* N = nccl();
        cudaSetDevice(ctx->device);
        cudaDeviceSynchronize();
        if (N->ok) N->CommDestroy((ncclComm_t)ctx->comm);
        ctx->comm = nullptr; ctx->comm_rank = 0; ctx->comm_world = 0;
    }
    return ORT_OK;
}

int ort_merge_stats_dev(ort_ctx* ctx, const ort_stats* d_recs, int n_shards, int n_fields, ort_stats* d_out, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (!d_recs || !d_out || n_shards < 1 || n_fields < 1 || n_fields > ORT_MAX_FIELDS) return fail(ctx, ORT_EINVAL, "merge_stats_dev: bad input");
    CK(cudaSetDevice(ctx->device));
    return merge_enqueue(ctx, d_recs, n_shards, n_fields, d_out, (cudaStream_t)stream);
}

int ort_comm_range(int64_t total, int rank, int world, int64_t* lo, int64_t* hi)
{
    if (total < 0 || world < 1 || rank < 0 || rank >= world || !lo || !hi) return ORT_EINVAL;
    long long a, b;
    comm_range(total, rank, world, &a, &b);
    *lo = a; *hi = b;
    return ORT_OK;
}

// ------------------------------------------------------------------------------------------
// one process, n contexts: the whole pupil grid in one call
// ------------------------------------------------------------------------------------------
// `ctx` always names the context being acted on (CK / ENSURE report into it, ENSURE allocates in it); *cur follows it so
// the entry point can forward the message of a failing device to ctxs[0]
static int grid_multi_impl(ort_ctx** ctxs, int n, const ort_field* fields, int n_fields, const double* ys, int ny,
                           const double* xs, int nx, int stop, double a_stop, const ort_opts* opts, ort_grid_out* out,
                           ort_ctx** cur)
{
    ort_ctx*& ctx = *cur;
    ctx = ctxs ? ctxs[0] : nullptr;
    if (!ctxs || !ctx || n < 1 || n > ORT_MAX_GPUS) return fail(ctx, ORT_EINVAL, "trace3d_grid_multi: n = %d not in [1, %d]", n, ORT_MAX_GPUS);
    for (int d = 0; d < n; d++) {
        if (!ctxs[d]) return fail(ctx, ORT_EINVAL, "trace3d_grid_multi: ctxs[%d] is NULL", d);
        if (n > 1 && (!ctxs[d]->comm || ctxs[d]->comm_world != n || ctxs[d]->comm_rank != d))
            return fail(ctx, ORT_ENCCL, "trace3d_grid_multi: ctxs[%d] is not rank %d of an %d-context communicator (ort_comm_init_all)", d, d, n);
    }
    ort_opts o1 = opts ? *opts : ort_opts();
    o1.gather_stats = 0;                                    // the gather is driven from here, grouped over the contexts
    int rc = ort_grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts ? &o1 : nullptr, out);
    if (rc) return rc;
    const size_t NNt = (size_t)ny * nx;                     // whole grid, per field
    struct Dev {
        long long lo, hi; unsigned NN;
        ort_grid_out full, comp;
        ort_stats *d_stats, *d_merged, *d_ranks;
    } D[ORT_MAX_GPUS];
    static thread_local ort_stats hstats[ORT_MAX_GPUS][ORT_MAX_FIELDS];
    ort_stats hmerged[ORT_MAX_FIELDS];

    // ---- phase A: every context traces its block of y-rows --------------------------------------------------
    for (int d = 0; d < n; d++) {
        ort_ctx* c = ctxs[d];
        Dev& V = D[d];
        memset(&V, 0, sizeof V);
        comm_range(ny, d, n, &V.lo, &V.hi);
        const int nyd = (int)(V.hi - V.lo);
        V.NN = (unsigned)((long long)nyd * nx);
        ctx = c;                                            // CK / ENSURE report into the context they act on
        CK(cudaSetDevice(c->device));
        if (d > 0) {                                        // the layout of ctxs[0] on every context
            const double* poly0 = ctxs[0]->presc.poly;
            c->presc = ctxs[0]->presc; c->rows = ctxs[0]->rows; c->have_layout = true; c->fast_ok_layout = ctxs[0]->fast_ok_layout;
            c->have_polyk = ctxs[0]->have_polyk; if (c->have_polyk) c->polyk = ctxs[0]->polyk;
            if (poly0) {
                const size_t nb = 2 * (size_t)(c->rows - 1) * c->presc.npoly * 8;      // coefficients and k c_k
                double* dp; ENSURE(SL_POLY, nb, dp);
                CK(cudaMemcpyPeerAsync(dp, c->device, poly0, ctxs[0]->device, nb, c->stream));
                c->presc.poly = dp;
            }
        }
        cudaStream_t st = c->stream;
        ScratchScope scratch(c, st);
        const int gx = ort_grid_dims(c, c->bps, ort_grid_waves(), &o1, n_fields, V.NN);
        double *d_ys, *d_xs;
        const size_t nys = (size_t)nyd * (o1.ys_per_field ? n_fields : 1);
        ENSURE(SL_YS, sizeof(double) * nys, d_ys);
        ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
        RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * n_fields, d_partials);
        ENSURE(SL_STATS, sizeof(ort_stats) * (size_t)n_fields, V.d_stats);
        ENSURE(SL_MERGED, sizeof(ort_stats) * (size_t)n_fields, V.d_merged);
        ENSURE(SL_GATHER, sizeof(ort_stats) * (size_t)n_fields * n, V.d_ranks);
        int* d_tiles;
        if ((rc = ort_sweep_scratch(c, out, &o1, false, V.NN, n_fields, 1, &V.full, &V.comp, &d_tiles))) return rc;
        if (o1.ys_per_field)
            for (int f = 0; f < n_fields; f++)
                CK(cudaMemcpyAsync(d_ys + (size_t)f * nyd, ys + (size_t)f * ny + V.lo, sizeof(double) * (size_t)nyd, cudaMemcpyHostToDevice, st));
        else
            CK(cudaMemcpyAsync(d_ys, ys + V.lo, sizeof(double) * (size_t)nyd, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
        rc = ort_grid_enqueue(c, fields, n_fields, d_ys, nyd, d_xs, nx, stop, a_stop, nullptr, 1, &o1, V.full,
                              o1.compact ? &V.comp : nullptr, V.d_stats, d_partials, d_tiles, gx, st);
        if (rc) return rc;
    }
    // ---- the one exchange: grouped all-gather of the records, rank-order merge on every device ----------------
    if (n > 1) {
        ctx = ctxs[0];
        NEED_NCCL(N);
        NCK(N->GroupStart());
        for (int d = 0; d < n; d++) {
            ncclResult_t r = N->AllGather(D[d].d_stats, D[d].d_ranks, sizeof(ort_stats) * (size_t)n_fields, ncclChar,
                                          (ncclComm_t)ctxs[d]->comm, ctxs[d]->stream);
            if (r != ncclSuccess) { N->GroupEnd(); return fail(ctx, ORT_ENCCL, "ncclAllGather (device %d) -> %s", ctxs[d]->device, N->GetErrorString(r)); }
        }
        NCK(N->GroupEnd());
    }
    for (int d = 0; d < n; d++) {
        ort_ctx* c = ctxs[d];
        ctx = c;
        CK(cudaSetDevice(c->device));
        if (n > 1) { rc = merge_enqueue(c, D[d].d_ranks, n, n_fields, D[d].d_merged, c->stream); if (rc) return rc; }
        CK(cudaMemcpyAsync(hstats[d], D[d].d_stats, sizeof(ort_stats) * (size_t)n_fields, cudaMemcpyDeviceToHost, c->stream));
        if (d == 0 && n > 1) CK(cudaMemcpyAsync(hmerged, D[0].d_merged, sizeof(ort_stats) * (size_t)n_fields, cudaMemcpyDeviceToHost, c->stream));
    }
    for (int d = 0; d < n; d++) { ctx = ctxs[d]; CK(cudaSetDevice(ctx->device)); CK(cudaStreamSynchronize(ctx->stream)); }
    // ---- phase C: ray-level outputs straight from every device into the caller's arrays, reference order --------
    for (int d = 0; d < n; d++) {
        ort_ctx* c = ctxs[d];
        const Dev& V = D[d];
        ctx = c;
        if (V.NN == 0) continue;
        CK(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        for (int f = 0; f < n_fields; f++) {
            const size_t src_o = (size_t)f * V.NN;
            const size_t grid_o = (size_t)f * NNt + (size_t)V.lo * nx;            // this shard's rows inside the whole grid
            if ((rc = ort_copy_out(c, out, V.full, false, grid_o, src_o, V.NN, 1, V.NN, st))) return rc;
            size_t dst_o = grid_o, cnt = V.NN;
            if (o1.compact) {                                // behind the kept rays of the preceding shards
                dst_o = (size_t)f * NNt;
                for (int e = 0; e < d; e++) dst_o += (size_t)hstats[e][f].n_kept;
                cnt = (size_t)hstats[d][f].n_kept;
            }
            if ((rc = ort_copy_out(c, out, o1.compact ? V.comp : V.full, true, dst_o, src_o, cnt, 1, V.NN, st))) return rc;
        }
    }
    for (int d = 0; d < n; d++) { ctx = ctxs[d]; CK(cudaSetDevice(ctx->device)); CK(cudaStreamSynchronize(ctx->stream)); }
    if (out->stats) memcpy(out->stats, n > 1 ? hmerged : hstats[0], sizeof(ort_stats) * (size_t)n_fields);
    if (out->stats_local)
        for (int d = 0; d < n; d++) memcpy(out->stats_local + (size_t)d * n_fields, hstats[d], sizeof(ort_stats) * (size_t)n_fields);
    return ORT_OK;
}

int ort_trace3d_grid_multi(ort_ctx** ctxs, int n, const ort_field* fields, int n_fields, const double* ys, int ny,
                           const double* xs, int nx, int stop, double a_stop, const ort_opts* opts, ort_grid_out* out)
{
    ort_ctx* cur = nullptr;
    const int rc = grid_multi_impl(ctxs, n, fields, n_fields, ys, ny, xs, nx, stop, a_stop, opts, out, &cur);
    if (rc && cur && ctxs && ctxs[0] && cur != ctxs[0]) {
        char msg[400];
        snprintf(msg, sizeof msg, "%s", cur->err);
        fail(ctxs[0], rc, "device %d: %s", cur->device, msg);
    }
    return rc;
}

// ------------------------------------------------------------------------------------------
// candidate population sharded over the ranks (BASELINE config 5)
// ------------------------------------------------------------------------------------------
// d_RtnK_mine / d_aim_mine point at THIS rank's range [lo, hi); d_out is the whole table [C][4]
static int cand_sharded_enqueue(ort_ctx* ctx, int rows, long long C, long long lo, long long hi, const double* d_RtnK_mine,
                                const double* a, double h_prime, double H, int aspheric, int ny, int nx, int arith,
                                double* d_aim_mine, double* d_out, cudaStream_t st)
{
    const int world = ctx->comm ? ctx->comm_world : 1;
    int rc = ort_aim_candidates_dev(ctx, rows, hi - lo, d_RtnK_mine, a, h_prime, H, aspheric, d_aim_mine, st);
    if (rc) return rc;
    rc = ort_trace3d_candidates_aimed_dev(ctx, rows, hi - lo, d_RtnK_mine, d_aim_mine, ny, nx, arith, d_out + 4 * lo, st);
    if (rc || world == 1) return rc;
    NEED_NCCL(N);
    if (C % world == 0) {                                    // equal segments: one in-place all-gather
        NCK(N->AllGather(d_out + 4 * lo, d_out, (size_t)(4 * (hi - lo)), ncclDouble, (ncclComm_t)ctx->comm, st));
    } else {                                                 // uneven: one grouped broadcast per owner
        NCK(N->GroupStart());
        for (int r = 0; r < world; r++) {
            long long l, h;
            comm_range(C, r, world, &l, &h);
            ncclResult_t e = N->Broadcast(d_out + 4 * l, d_out + 4 * l, (size_t)(4 * (h - l)), ncclDouble, r, (ncclComm_t)ctx->comm, st);
            if (e != ncclSuccess) { N->GroupEnd(); return fail(ctx, ORT_ENCCL, "ncclBroadcast(root %d) -> %s", r, N->GetErrorString(e)); }
        }
        NCK(N->GroupEnd());
    }
    return ORT_OK;
}

static int cand_sharded_check(ort_ctx* ctx, int rows, int64_t C, const void* RtnK, const void* a, const void* out)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS - 1) return fail(ctx, ORT_EINVAL, "candidates_sharded: rows = %d", rows);
    if (C < 0 || C >= (1LL << 31) || !RtnK || !a || !out) return fail(ctx, ORT_EINVAL, "candidates_sharded: bad input");
    return ORT_OK;
}

int ort_candidates_sharded_dev(ort_ctx* ctx, int rows, int64_t C, const double* d_RtnK, const double* a, double h_prime,
                               double H, int aspheric, int ny, int nx, int arith, double* d_aim, double* d_out, void* stream)
{
    int rc = cand_sharded_check(ctx, rows, C, d_RtnK, a, d_out);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    long long lo, hi;
    comm_range(C, ctx->comm ? ctx->comm_rank : 0, ctx->comm ? ctx->comm_world : 1, &lo, &hi);
    ScratchScope scratch(ctx, st);
    double* d_aim_mine = d_aim ? d_aim + (size_t)lo * ORT_AIM_NOUT : nullptr;
    if (!d_aim_mine) ENSURE(SL_AIM, (size_t)(hi - lo) * ORT_AIM_NOUT * 8, d_aim_mine);
    return cand_sharded_enqueue(ctx, rows, C, lo, hi, d_RtnK + (size_t)lo * 4 * rows, a, h_prime, H, aspheric, ny, nx, arith,
                                d_aim_mine, d_out, st);
}

int ort_candidates_sharded(ort_ctx* ctx, int rows, int64_t C, const double* RtnK, const double* a, double h_prime, double H,
                           int aspheric, int ny, int nx, int arith, double* aim, double* out)
{
    int rc = cand_sharded_check(ctx, rows, C, RtnK, a, out);
    if (rc) return rc;
    if (C == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    long long lo, hi;
    comm_range(C, ctx->comm ? ctx->comm_rank : 0, ctx->comm ? ctx->comm_world : 1, &lo, &hi);
    const size_t stride = (size_t)4 * rows, nmine = (size_t)(hi - lo);
    double *d_p, *d_aim, *d_tab;
    ENSURE(SL_IN0, nmine * stride * 8, d_p);
    ENSURE(SL_AIM, nmine * ORT_AIM_NOUT * 8, d_aim);
    ENSURE(SL_TABLE, (size_t)C * 32, d_tab);
    CK(cudaMemcpyAsync(d_p, RtnK + (size_t)lo * stride, nmine * stride * 8, cudaMemcpyHostToDevice, st));
    rc = cand_sharded_enqueue(ctx, rows, C, lo, hi, d_p, a, h_prime, H, aspheric, ny, nx, arith, d_aim, d_tab, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_tab, (size_t)C * 32, cudaMemcpyDeviceToHost, st));
    if (aim) CK(cudaMemcpyAsync(aim + (size_t)lo * ORT_AIM_NOUT, d_aim, nmine * ORT_AIM_NOUT * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

}  // extern "C"
