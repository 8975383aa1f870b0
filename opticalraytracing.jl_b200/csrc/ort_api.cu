// ort_api.cu -- the C ABI of libort_b200.so (include/ort_b200.h): context, prescription upload,
// host-pointer (synchronous, staged through device scratch) and device-pointer (enqueue-only)
// entry points.  No torch types, no exceptions across the boundary, no CPU fallback.
#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>

#include <new>
#include <vector>

#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <sched.h>
#include <stdlib.h>
#include <sys/syscall.h>
#include <unistd.h>
#include "ort_ctx.cuh"

thread_local char g_init_err[512] = "";

int ort_fail(ort_ctx* c, int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(c ? c->err : g_init_err, 512, fmt, ap);
    va_end(ap);
    return code;
}

// grow-only device scratch
int ort_ensure(ort_ctx* ctx, int id, size_t bytes, void** out)
{
    if (bytes == 0) bytes = 8;
    if (ctx->slot_bytes[id] < bytes) {
        // growth is rare: wait for EVERYTHING on the device (the slot may still be in use by work a *_dev call
        // enqueued on a caller-owned stream) before releasing the old block
        if (ctx->slot[id]) { cudaDeviceSynchronize(); cudaFree(ctx->slot[id]); }
        ctx->slot[id] = nullptr; ctx->slot_bytes[id] = 0;
        cudaError_t e = cudaMalloc(&ctx->slot[id], bytes);
        if (e != cudaSuccess) return fail(ctx, ORT_ENOMEM, "cudaMalloc(%zu) -> %s", bytes, cudaGetErrorString(e));
        ctx->slot_bytes[id] = bytes;
    }
    *out = ctx->slot[id];
    // ORT_POISON_SCRATCH=1 (tests): every slot is filled with 0xFF bytes -- NaNs, -1 counts -- each time an entry point
    // asks for it, on the stream the entry point works on, so that a kernel that reads scratch it did not write (or an
    // output the library forgot to write) shows up as a wrong result instead of depending on what the block held before.
    // SL_POLY is the one slot whose content outlives the call that fills it.
    static const bool poison = [] { const char* e = getenv("ORT_POISON_SCRATCH"); return e && atoi(e) != 0; }();
    if (poison && id != SL_POLY) {
        cudaError_t e = cudaMemsetAsync(ctx->slot[id], 0xFF, bytes, ctx->scratch_now);
        if (e != cudaSuccess) return fail(ctx, ORT_ECUDA, "poison memset -> %s", cudaGetErrorString(e));
    }
    return ORT_OK;
}

int ort_resolve_arith(const ort_ctx* ctx, int arith)
{
    if (arith == ORT_ARITH_FAST && !ctx->presc.fast_ok) return ORT_ARITH_STRICT;
    return arith;
}
#define resolve_arith ort_resolve_arith
#define grid_check ort_grid_check
#define grid_enqueue ort_grid_enqueue
#define grid_dims ort_grid_dims

extern "C" {

int ort_version(void) { return ORT_VERSION; }

int ort_init(ort_ctx** out, int device)
{
    ort_ctx* ctx = nullptr;
    if (!out) return fail(nullptr, ORT_EINVAL, "ort_init: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, ORT_ECUDA, "ort_init: no CUDA device (%s); libort_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= ndev) return fail(nullptr, ORT_EINVAL, "ort_init: device %d of %d", device, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, ORT_ECUDA, "cudaGetDeviceProperties -> %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, ORT_EUNSUPPORTED, "ort_init: device %d is sm_%d%d; this library is built for sm_100a only",
                    device, prop.major, prop.minor);
    ctx = new (std::nothrow) ort_ctx();
    if (!ctx) return fail(nullptr, ORT_ENOMEM, "ort_init: out of host memory");
    memset(ctx, 0, sizeof(*ctx));
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major; ctx->cc_minor = prop.minor;
    snprintf(ctx->name, sizeof ctx->name, "%.127s", prop.name);
#define CKI(call)                                                                                   \
    do { cudaError_t e2_ = (call); if (e2_ != cudaSuccess) {                                        \
             fail(nullptr, ORT_ECUDA, "ort_init: %s -> %s", #call, cudaGetErrorString(e2_));         \
             ort_free(ctx); return ORT_ECUDA; } } while (0)
    CKI(cudaSetDevice(device));
    CKI(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CKI(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    ctx->scratch_now = ctx->stream;
    CKI(cudaEventCreate(&ctx->ev_a));
    CKI(cudaEventCreate(&ctx->ev_b));
    CKI(cudaEventCreateWithFlags(&ctx->ev_scratch, cudaEventDisableTiming));
    for (int i = 0; i < ORT_MAX_FIELDS; i++) CKI(cudaEventCreateWithFlags(&ctx->ev_field[i], cudaEventDisableTiming));
    for (int i = 0; i < 64; i++) { CKI(cudaEventCreate(&ctx->prof_ev[i][0])); CKI(cudaEventCreate(&ctx->prof_ev[i][1])); }
#undef CKI
    for (int v = 0; v < 5; v++) {
        ctx->bps[ORT_ARITH_STRICT][v] = grid_blocks_per_sm(ORT_ARITH_STRICT, v);
        ctx->bps[ORT_ARITH_FAST][v] = grid_blocks_per_sm(ORT_ARITH_FAST, v);
        ctx->bps_focus[ORT_ARITH_STRICT][v] = focus_blocks_per_sm(ORT_ARITH_STRICT, v);
        ctx->bps_focus[ORT_ARITH_FAST][v] = focus_blocks_per_sm(ORT_ARITH_FAST, v);
    }
    *out = ctx;
    return ORT_OK;
}

void ort_free(ort_ctx* ctx)
{
    if (!ctx) return;
    // also the unwinding path of a failed ort_init: every handle may still be null
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    ort_comm_free(ctx);
    if (ctx->ev_scratch) cudaEventDestroy(ctx->ev_scratch);
    for (int i = 0; i < SL_COUNT; i++) if (ctx->slot[i]) cudaFree(ctx->slot[i]);
    for (int i = 0; i < ORT_MAX_FIELDS; i++) if (ctx->ev_field[i]) cudaEventDestroy(ctx->ev_field[i]);
    for (int i = 0; i < 64; i++)
        for (int j = 0; j < 2; j++) if (ctx->prof_ev[i][j]) cudaEventDestroy(ctx->prof_ev[i][j]);
    if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
    if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}

const char* ort_last_error(ort_ctx* ctx) { return ctx ? ctx->err : g_init_err; }

int ort_sync(ort_ctx* ctx)
{
    if (!ctx) return ORT_EINVAL;
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaStreamSynchronize(ctx->copy_stream));
    return ORT_OK;
}

int ort_device_info(ort_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, char* name, int name_len)
{
    if (!ctx) return ORT_EINVAL;
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", ctx->name);
    return ORT_OK;
}

// NUMA node of the context's GPU from sysfs (cudaDeviceGetPCIBusId -> /sys/bus/pci/devices/<id>/numa_node)
static int device_numa_node(ort_ctx* ctx, char* cpulist, int len)
{
    char bus[32] = "";
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, ctx->device) != cudaSuccess) return -1;
    for (char* p = bus; *p; p++) if (*p >= 'A' && *p <= 'F') *p = (char)(*p - 'A' + 'a');
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    int node = -1;
    if (f) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
    if (cpulist && len > 0) {
        cpulist[0] = 0;
        if (node >= 0) {
            snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
            f = fopen(path, "r");
            if (f) { if (!fgets(cpulist, len, f)) cpulist[0] = 0; fclose(f); }
            for (char* p = cpulist; *p; p++) if (*p == '\n') *p = 0;
        }
    }
    return node;
}

int ort_device_numa(ort_ctx* ctx, int* node, char* cpulist, int cpulist_len)
{
    if (!ctx) return ORT_EINVAL;
    const int n = device_numa_node(ctx, cpulist, cpulist_len);
    if (node) *node = n;
    return ORT_OK;
}

int ort_bind_host_thread(ort_ctx* ctx, int* bound)
{
    if (!ctx) return ORT_EINVAL;
    if (bound) *bound = 0;
    char list[1024];
    const int node = device_numa_node(ctx, list, sizeof list);
    if (node < 0 || !list[0]) return fail(ctx, ORT_EUNSUPPORTED, "ort_bind_host_thread: NUMA node of device %d unknown", ctx->device);
    int got = 0;
    cpu_set_t set; CPU_ZERO(&set);
    for (const char* p = list; *p;) {                     // "0-31,64-95"
        char* e; long a = strtol(p, &e, 10), b = a;
        if (e == p) break;
        if (*e == '-') { p = e + 1; b = strtol(p, &e, 10); }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) CPU_SET((int)c, &set);
        p = (*e == ',') ? e + 1 : e;
        if (*e != ',' ) break;
    }
    if (sched_setaffinity(0, sizeof set, &set) == 0) got |= 1;
    if (node < 64) {                                      // MPOL_PREFERRED = 1: allocate on this node when possible
        unsigned long mask = 1UL << node;
        if (syscall(SYS_set_mempolicy, 1, &mask, (unsigned long)(8 * sizeof mask)) == 0) got |= 2;
    }
    if (bound) *bound = got;
    if (!got) return fail(ctx, ORT_EUNSUPPORTED, "ort_bind_host_thread: node %d (cpus %s) is outside this process's cpuset", node, list);
    return ORT_OK;
}

void* ort_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 8, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void ort_host_free(void* p) { if (p) cudaFreeHost(p); }

int64_t ort_launch_count(ort_ctx* ctx) { return ctx ? ctx->launches : 0; }

int ort_profile_enable(ort_ctx* ctx, int on)
{
    if (!ctx) return ORT_EINVAL;
    ctx->prof_on = on ? 1 : 0;
    ctx->prof_n = 0;
    return ORT_OK;
}

int ort_profile_read(ort_ctx* ctx, double* ms_out, int max_n)
{
    if (!ctx || !ms_out || max_n < 0) return ORT_EINVAL;
    long long n = ctx->prof_n < 64 ? ctx->prof_n : 64;
    if (n > max_n) n = max_n;
    const long long first = ctx->prof_n - n;
    for (long long j = 0; j < n; j++) {
        const int slot = (int)((first + j) % 64);
        if (cudaEventSynchronize(ctx->prof_ev[slot][1]) != cudaSuccess) return ORT_ECUDA;
        float t = 0.f;
        if (cudaEventElapsedTime(&t, ctx->prof_ev[slot][0], ctx->prof_ev[slot][1]) != cudaSuccess) return ORT_ECUDA;
        ms_out[j] = (double)t;
    }
    ctx->prof_n = 0;
    return (int)n;
}

int ort_set_layout(ort_ctx* ctx, int rows, const double* R, const double* t, const double* n, const double* K)
{
    if (!ctx) return ORT_EINVAL;
    if (!R || !t || !n) return fail(ctx, ORT_EINVAL, "ort_set_layout: NULL column");
    if (rows < 2 || rows > ORT_MAX_ROWS) return fail(ctx, ORT_EINVAL, "ort_set_layout: rows = %d not in [2, %d]", rows, ORT_MAX_ROWS);
    Presc& P = ctx->presc;
    memset(&P, 0, sizeof P);
    P.nsurf = rows - 1;
    P.fast_ok = 1;
    P.t_last = t[rows - 1];
    P.n0 = n[0];
    P.nlast = n[rows - 1];
    for (int i = 0; i + 1 < rows; i++) {
        const double Ri = R[i + 1], Ki = K ? K[i + 1] : 0.0;
        derive_surface(P.s[i], Ri, Ki, t[i], n[i], n[i + 1]);
        if (Ri == 0.0 || isnan(Ri) || !isfinite(Ki) || !isfinite(t[i]) || !isfinite(n[i]) || !isfinite(n[i + 1]) ||
            n[i] == 0.0 || n[i + 1] == 0.0)
            P.fast_ok = 0;
        if (!(n[i] > 0.0) || !(n[i + 1] > 0.0)) P.has_mirror = 1;      // reflection (n2 = -n1) or anything unusual
    }
    // class of the prescription (ort_internal.cuh): 1 = refracting spheres (|R| <= 64 L) and planes; 2 = refracting conics /
    // spheres and planes with at least one conic; 0 = anything else (mirrors, dummy curved surfaces, weak spheres without conics)
    const double L = gap_scale(t, rows);
    P.simple = P.fast_ok && !P.has_mirror;
    bool conic_class = P.simple, any_conic = false;
    for (int i = 0; i + 1 < rows; i++) {
        const bool plane = (P.s[i].kcode & SURF_KIND_MASK) == SURF_PLANE;
        if (!plane && !(P.s[i].kcode & SURF_REFR)) conic_class = false;               // dummy curved surface
        if ((P.s[i].kcode & SURF_KIND_MASK) == SURF_CONIC) any_conic = true;
        if (!simple_surface(P.s[i], L)) P.simple = 0;
    }
    if (!P.simple && conic_class && any_conic) P.simple = 2;
    ctx->rows = rows;
    ctx->have_layout = true;
    ctx->fast_ok_layout = P.fast_ok;
    return ORT_OK;
}

int ort_set_polynomials(ort_ctx* ctx, int rows, int ncoef, const double* coef)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "ort_set_polynomials: call ort_set_layout first");
    Presc& P = ctx->presc;
    auto clear = [&]() {                             // no terms: every surface dispatches on its own kind again
        P.poly = nullptr; P.npoly = 0; P.fast_ok = ctx->fast_ok_layout; ctx->have_polyk = false;
        for (int i = 0; i < P.nsurf; i++) P.s[i].kcode = P.s[i].kind & 7;
    };
    if (!coef || ncoef <= 0) { clear(); return ORT_OK; }
    if (rows != ctx->rows) return fail(ctx, ORT_EINVAL, "ort_set_polynomials: rows = %d, layout has %d", rows, ctx->rows);
    if (ncoef > ORT_MAX_POLY) return fail(ctx, ORT_EINVAL, "ort_set_polynomials: ncoef = %d > %d", ncoef, ORT_MAX_POLY);
    bool any = false;
    for (int i = 0; i < rows * ncoef; i++) {
        if (isnan(coef[i])) return fail(ctx, ORT_EINVAL, "ort_set_polynomials: NaN coefficient");
        any = any || coef[i] != 0.0;
    }
    if (!any) { clear(); return ORT_OK; }            // all zero == Polynomial(zero)
    CK(cudaSetDevice(ctx->device));
    ScratchScope scratch(ctx, ctx->stream);
    const size_t ntab = (size_t)(rows - 1) * ncoef;
    double* d_c; ENSURE(SL_POLY, 2 * ntab * 8, d_c);
    // surface step i uses Layout row i + 1 (row 0 is object space); behind the coefficients, k c_k for the FAST body's dp/dy
    std::vector<double> tab(2 * ntab);
    for (size_t i = 0; i < ntab; i++) { tab[i] = coef[ncoef + i]; tab[ntab + i] = (double)(i % ncoef) * coef[ncoef + i]; }
    CK(cudaMemcpyAsync(d_c, tab.data(), 2 * ntab * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    P.poly = d_c; P.npoly = ncoef;
    ctx->have_polyk = ncoef <= ORT_POLYK_N;
    if (ctx->have_polyk) {
        memset(&ctx->polyk, 0, sizeof ctx->polyk);
        for (int i = 0; i + 1 < rows; i++)
            for (int k = 0; k < ncoef; k++) {
                ctx->polyk.r[i].c[k] = tab[(size_t)i * ncoef + k];
                ctx->polyk.r[i].d[k] = tab[ntab + (size_t)i * ncoef + k];
            }
    }
    // FAST: curved surfaces with terms take fast_step's polynomial body (kcode 7).  It has no mirror form, so prescriptions
    // with mirrors (and the degenerate ones) stay in the reference arithmetic.
    // A plane with terms keeps no sag term but does keep the tilt term (:12, :18) -- an oddity the FAST body does not restate.
    P.fast_ok = ctx->fast_ok_layout && !P.has_mirror;
    for (int i = 0; i < P.nsurf; i++) {
        bool row = false;
        for (int k = 0; k < ncoef; k++) row = row || coef[(size_t)(i + 1) * ncoef + k] != 0.0;
        const bool curved = (P.s[i].kind & SURF_KIND_MASK) != SURF_PLANE;
        if (row && !curved) P.fast_ok = 0;
        P.s[i].kcode = (row && curved) ? SURF_KCODE_POLY : (P.s[i].kind & 7);
    }
    return ORT_OK;
}

int ort_set_apertures(ort_ctx* ctx, int n, const double* a)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "ort_set_apertures: call ort_set_layout first");
    Presc& P = ctx->presc;
    if (a && (n < 0 || n > P.nsurf)) return fail(ctx, ORT_EINVAL, "ort_set_apertures: n = %d not in [0, %d]", n, P.nsurf);
    P.has_apertures = 0;
    for (int i = 0; i < P.nsurf; i++) {
        const double ai = (a && i < n && !isnan(a[i])) ? fabs(a[i]) : INFINITY;
        P.s[i].a = ai; P.s[i].a2 = ai * ai;
        if (isfinite(ai)) P.has_apertures = 1;
    }
    return ORT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// pupil-grid sweep (k_grid) and through-focus sweep (k_focus)
// ------------------------------------------------------------------------------------------
int ort_grid_check(ort_ctx* ctx, const ort_field* fields, int n_fields, const void* ys, int ny,
                      const void* xs, int nx, int stop, const ort_opts* opts, const ort_grid_out* out)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "trace3d_grid: call ort_set_layout first");
    if (!fields || n_fields < 1 || n_fields > ORT_MAX_FIELDS) return fail(ctx, ORT_EINVAL, "trace3d_grid: n_fields = %d not in [1, %d]", n_fields, ORT_MAX_FIELDS);
    if (!ys || !xs || ny < 0 || nx < 0) return fail(ctx, ORT_EINVAL, "trace3d_grid: bad grid");
    if ((long long)ny * nx >= (1LL << 31)) return fail(ctx, ORT_EINVAL, "trace3d_grid: ny*nx = %lld exceeds 2^31-1 per call", (long long)ny * nx);
    if (stop < 1 || stop > ctx->presc.nsurf) return fail(ctx, ORT_EINVAL, "trace3d_grid: stop = %d not in [1, %d]", stop, ctx->presc.nsurf);
    if (!opts || !out) return fail(ctx, ORT_EINVAL, "trace3d_grid: opts/out is NULL");
    if (opts->arith != ORT_ARITH_STRICT && opts->arith != ORT_ARITH_FAST) return fail(ctx, ORT_EINVAL, "trace3d_grid: arith = %d", opts->arith);
    for (int f = 0; f < n_fields; f++)
        if (fields[f].mode != 0 && fields[f].mode != 1) return fail(ctx, ORT_EINVAL, "trace3d_grid: field %d mode = %d", f, fields[f].mode);
    if (opts->gather_stats && !ctx->comm)
        return fail(ctx, ORT_ENCCL, "trace3d_grid: opts.gather_stats needs a communicator (ort_comm_init_rank / ort_comm_init_all)");
    return ORT_OK;
}

// The per-ray members of ort_grid_out and how a sweep stores them.  The compacted members come first, in the index order
// of CompactArgs.src / dst; mask and flags always cover the full grid.  A per-focus member of a through-focus sweep holds
// one block of NN rays per (field, focus), [n_fields][n_foci][NN].
struct OutMember {
    size_t off;                 // offsetof in ort_grid_out
    int slot, cslot;            // scratch slots of the full-grid and of the compacted array
    size_t bytes;               // per ray
    bool compacted, per_focus;
};
static const OutMember k_members[] = {
    {offsetof(ort_grid_out, ex), SL_EX, SL_CEX, 8, true, true},
    {offsetof(ort_grid_out, ey), SL_EY, SL_CEY, 8, true, true},
    {offsetof(ort_grid_out, r), SL_R, SL_CR, 8, true, false},
    {offsetof(ort_grid_out, theta), SL_TH, SL_CTH, 8, true, false},
    {offsetof(ort_grid_out, wx), SL_WX, SL_CWX, 8, true, false},
    {offsetof(ort_grid_out, wy), SL_WY, SL_CWY, 8, true, false},
    {offsetof(ort_grid_out, opd), SL_OPD, SL_COPD, 8, true, false},
    {offsetof(ort_grid_out, mask), SL_MASK, -1, 1, false, false},
    {offsetof(ort_grid_out, flags), SL_FLAGS, -1, 1, false, false},
};
static const int N_COMPACTED = 7;
static_assert(sizeof(CompactArgs::src) / sizeof(CompactArgs::src[0]) == N_COMPACTED, "one CompactArgs entry per compacted member");

static char* member(const ort_grid_out& o, const OutMember& m) { char* p; memcpy(&p, (const char*)&o + m.off, sizeof p); return p; }
static void set_member(ort_grid_out& o, const OutMember& m, void* p) { memcpy((char*)&o + m.off, &p, sizeof p); }

// the members of a grid sweep's outputs from ray i of the first field on
static ort_grid_out from_ray(const ort_grid_out& g, size_t i)
{
    ort_grid_out o = g;
    for (const OutMember& m : k_members)
        if (char* p = member(g, m)) set_member(o, m, p + i * m.bytes);
    return o;
}

// Scratch of a sweep's per-ray outputs; call it inside the entry point's ScratchScope, so that a poisoning memset is
// ordered like the work.  Host form (dev false): every member `out` wants is traced into its slot of *full -- the mask
// also when compacting -- and, when compacting, scattered into its slot of *comp.  Device form: the caller's arrays are
// the results (*full = *comp = *out); when compacting, the members that are compacted are traced into scratch, and so is
// the mask when the caller gives none, while flags are written in place.  opd is wanted only with ORT_EXT_OPD.
// *d_tiles: the tile counts of the compaction, or NULL.
int ort_sweep_scratch(ort_ctx* ctx, const ort_grid_out* out, const ort_opts* opts, bool dev, unsigned NN, int n_fields,
                      int n_foci, ort_grid_out* full, ort_grid_out* comp, int** d_tiles)
{
    *d_tiles = nullptr;
    if (dev) { *full = *out; *comp = *out; }
    else { memset(full, 0, sizeof *full); memset(comp, 0, sizeof *comp); }
    if (dev && !opts->compact) return ORT_OK;
    const size_t tot = (size_t)NN * n_fields;
    for (const OutMember& m : k_members) {
        const size_t bytes = tot * m.bytes * (m.per_focus ? n_foci : 1);
        const bool want = member(*out, m) && (m.slot != SL_OPD || (opts->ext & ORT_EXT_OPD));
        const bool mask = m.slot == SL_MASK;
        const bool traced = dev ? (m.compacted ? want : mask && !want) : want || (mask && opts->compact);
        void* p = nullptr;
        if (traced) ENSURE(m.slot, bytes, p);
        if (traced || (dev && m.compacted)) set_member(*full, m, p);
        if (!dev && opts->compact && m.compacted && want) { ENSURE(m.cslot, bytes, p); set_member(*comp, m, p); }
    }
    if (opts->compact) ENSURE(SL_TILES, sizeof(int) * compact_tile_ints(NN) * n_fields, *d_tiles);
    return ORT_OK;
}

// Device-to-host copies on `st` of one kind of member -- the compacted kind (rays) or mask and flags -- that `out` wants
// and `src` holds: n rays from ray src_o of src to ray dst_o of out, offsets of a per-field array.  A per-focus member
// copies its n_foci blocks of the field, block j from / to ray o * n_foci + j * NN.
int ort_copy_out(ort_ctx* ctx, const ort_grid_out* out, const ort_grid_out& src, bool rays, size_t dst_o, size_t src_o,
                 size_t n, int n_foci, unsigned NN, cudaStream_t st)
{
    for (const OutMember& m : k_members) {
        char *d = member(*out, m), *s = member(src, m);
        if (m.compacted != rays || !d || !s) continue;
        const size_t nb = m.per_focus ? (size_t)n_foci : 1;
        for (size_t j = 0; j < nb; j++)
            CK(cudaMemcpyAsync(d + (dst_o * nb + j * NN) * m.bytes, s + (src_o * nb + j * NN) * m.bytes, n * m.bytes,
                               cudaMemcpyDeviceToHost, st));
    }
    return ORT_OK;
}

// Enqueue on `st` the sweep of fields [0, n_fields): k_grid, or with foci k_focus at n_foci image planes; then
// k_grid_finalize over the n_fields * n_foci records and, when dst is given, the tile scan and the compaction of the
// members of `full` that dst holds.  All pointers are device pointers; a grid sweep passes foci = NULL, n_foci = 1.
int ort_grid_enqueue(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* d_ys, int ny,
                        const double* d_xs, int nx, int stop, double a_stop, const double* foci, int n_foci,
                        const ort_opts* opts, const ort_grid_out& full, const ort_grid_out* dst, ort_stats* d_stats,
                        RawPart* d_partials, int* d_tiles, int gx, cudaStream_t st)
{
    const unsigned NN = (unsigned)((long long)ny * nx);
    FocusArgs F;
    memset(&F, 0, sizeof F);
    GridArgs& A = F.G;
    A.ys = d_ys; A.xs = d_xs; A.ny = ny; A.nx = nx; A.NN = NN; A.stop = stop;
    A.ys_stride = opts->ys_per_field ? ny : 0;
    A.a_stop = a_stop; A.a_stop2 = a_stop * a_stop;
    A.wg_nu = opts->wg_nu; A.wg_lambda = opts->wg_lambda;
    A.ext = opts->ext & (ORT_EXT_OPD | ORT_EXT_VIGNETTE);
    A.opd_scale = opts->opd_scale; A.opd = (A.ext & ORT_EXT_OPD) ? full.opd : nullptr;
    A.ex = full.ex; A.ey = full.ey; A.r = full.r; A.theta = full.theta; A.wx = full.wx; A.wy = full.wy;
    A.mask = full.mask; A.flags = full.flags;
    A.partials = d_partials;
    A.tile_counts = dst ? d_tiles : nullptr;
    memcpy(A.fields, fields, sizeof(ort_field) * (size_t)n_fields);
    if (foci) {
        F.n_foci = n_foci;
        F.t_lo = F.t_hi = foci[0];
        for (int j = 0; j < n_foci; j++) {
            F.foci[j] = foci[j];
            F.t_lo = fmin(F.t_lo, foci[j]); F.t_hi = fmax(F.t_hi, foci[j]);
        }
    }
    const int arith = resolve_arith(ctx, opts->arith);
    const int nrec = n_fields * n_foci;
    const dim3 grid((unsigned)gx, (unsigned)n_fields);
    if (NN > 0) {
        ProfScope prof(ctx, st);
        CK(foci ? launch_focus(ctx->presc, F, arith, grid, st)
                : launch_grid(ctx->presc, A, arith, grid, st, ctx->have_polyk ? &ctx->polyk : nullptr));
        ctx->launches++;
    } else {
        CK(cudaMemsetAsync(d_partials, 0, sizeof(RawPart) * (size_t)gx * nrec, st));
    }
    CK(launch_grid_finalize(d_partials, gx, nrec, d_stats, st));
    ctx->launches++;
    if (dst && NN > 0) {
        CompactArgs C;
        memset(&C, 0, sizeof C);
        C.NN = NN; C.mask = full.mask; C.tile_offsets = d_tiles;
        for (int a = 0; a < N_COMPACTED; a++) {
            const OutMember& m = k_members[a];
            if (member(full, m) && member(*dst, m)) { C.src[a] = (const double*)member(full, m); C.dst[a] = (double*)member(*dst, m); }
        }
        CK(foci ? launch_compact_focus(d_tiles, C, n_fields, n_foci, st) : launch_compact(d_tiles, C, n_fields, st));
        ctx->launches += 3;
    }
    return ORT_OK;
}

// Several waves of CTAs instead of one persistent wave: the warp schedulers favour the older of the resident CTAs, so
// with one wave of equal shares the CTAs of an SM finish far apart and the SM idles at half occupancy in between
// (ncu: 3.4 of 4 warps per scheduler active on average).  With 8 waves the block scheduler refills the slot:
// 2.23 ms vs 2.34 (4, 16 waves: 2.25, 2.23; 32: 2.26 -- every CTA first traces its field's centre ray).
// ORT_GRID_WAVES overrides the grid sweep's count (tuning).
int ort_grid_waves()
{
    static const int waves = [] { const char* e = getenv("ORT_GRID_WAVES"); const int w = e ? atoi(e) : ORT_GRID_WAVES_DEFAULT; return w < 1 ? 1 : w; }();
    return waves;
}

// CTAs along x of a sweep launch: at most `waves` waves of the resident CTAs/SM in bps (ctx->bps for k_grid,
// ctx->bps_focus for k_focus).  A CTA keeps at least 16 tiles so that its prologue stays amortised; the per-CTA partial
// sums still belong to a fixed set of tiles, so the statistics stay bit-reproducible.
int ort_grid_dims(const ort_ctx* ctx, const int (&bps)[2][5], int waves, const ort_opts* opts, int n_fields, unsigned NN)
{
    const int arith = resolve_arith(ctx, opts->arith);
    const int variant = grid_variant(ctx->presc, arith, (opts->ext & 3) || ctx->presc.poly);
    const unsigned nsub = (NN + ORT_TILE - 1) / ORT_TILE;
    const unsigned rpt = (unsigned)grid_rays_per_thread(arith, variant);
    const unsigned ntiles = (nsub + rpt - 1) / rpt;
    long long slots = (long long)ctx->sm_count * bps[arith][variant] / n_fields;
    if (slots < 1) slots = 1;
    long long gx = (long long)ntiles / 16;
    if (gx < slots) gx = slots;
    if (gx > slots * waves) gx = slots * waves;
    // the kernel's per-thread flag counters are 16 bits wide (RawAcc): keep a thread below 32 000 rays whatever the grid
    const long long gmin = ((long long)nsub + 31999) / 32000;
    if (gx < gmin) gx = gmin;
    if (gx > (long long)ntiles) gx = ntiles;
    if (gx < 1) gx = 1;
    return (int)gx;
}

extern "C" {

int ort_trace3d_grid_dev(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* d_ys, int ny,
                         const double* d_xs, int nx, int stop, double a_stop, const ort_opts* opts,
                         const ort_grid_out* d_out, void* stream)
{
    int rc = grid_check(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, opts, d_out);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const int gx = grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, n_fields, NN);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * n_fields, d_partials);
    // with opts.gather_stats out->stats receives the records merged over all ranks, out->stats_local this rank's own
    const bool gather = opts->gather_stats != 0;
    ort_stats* d_stats = gather ? d_out->stats_local : d_out->stats;
    if (!d_stats) ENSURE(SL_STATS, sizeof(ort_stats) * (size_t)n_fields, d_stats);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, d_out, opts, true, NN, n_fields, 1, &full, &comp, &d_tiles))) return rc;
    rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, nullptr, 1, opts, full,
                      opts->compact ? &comp : nullptr, d_stats, d_partials, d_tiles, gx, st);
    if (rc || !gather) return rc;
    ort_stats* d_merged = d_out->stats;
    if (!d_merged) ENSURE(SL_MERGED, sizeof(ort_stats) * (size_t)n_fields, d_merged);
    return ort_comm_gather_stats(ctx, d_stats, n_fields, d_merged, nullptr, st);
}

int ort_trace3d_grid(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* ys, int ny,
                     const double* xs, int nx, int stop, double a_stop, const ort_opts* opts,
                     ort_grid_out* out)
{
    int rc = grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts, out);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream, cs = ctx->copy_stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const size_t tot = (size_t)NN * n_fields;
    // one launch per field so the D2H of field f overlaps the trace of field f+1
    const int gx = grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, 1, NN);
    double *d_ys, *d_xs;
    const size_t nys = (size_t)ny * (opts->ys_per_field ? n_fields : 1);
    ENSURE(SL_YS, sizeof(double) * nys, d_ys);
    ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * n_fields, d_partials);
    ort_stats* d_stats; ENSURE(SL_STATS, sizeof(ort_stats) * (size_t)n_fields, d_stats);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, out, opts, false, NN, n_fields, 1, &full, &comp, &d_tiles))) return rc;
    CK(cudaMemcpyAsync(d_ys, ys, sizeof(double) * nys, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
    ort_stats hstats[ORT_MAX_FIELDS];
    const ort_grid_out& src = opts->compact ? comp : full;         // of the compacted kind of member
    // Large sweeps: one launch sequence per field, so the D2H of field f overlaps the trace of field f+1.
    // Small sweeps are launch-latency bound: all fields in ONE launch sequence (fields = grid dimension y).
    const bool per_field = n_fields > 1 && tot > ((size_t)1 << 21);
    if (!per_field) {
        const int gxa = grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, n_fields, NN);     // <= gx: partials slot is large enough
        rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, nullptr, 1, opts, full,
                          opts->compact ? &comp : nullptr, d_stats, d_partials, d_tiles, gxa, st);
        if (rc) return rc;
        CK(cudaMemcpyAsync(hstats, d_stats, sizeof(ort_stats) * (size_t)n_fields, cudaMemcpyDeviceToHost, st));
        if (opts->compact) CK(cudaStreamSynchronize(st));                        // counts needed for the copy sizes
        if ((rc = ort_copy_out(ctx, out, full, false, 0, 0, tot, 1, NN, st))) return rc;
        for (int f = 0; f < n_fields; f++) {
            const size_t o = (size_t)f * NN;
            const size_t cnt = opts->compact ? (size_t)hstats[f].n_kept : (size_t)NN;
            if ((rc = ort_copy_out(ctx, out, src, true, o, o, cnt, 1, NN, st))) return rc;
        }
    }
    for (int f = 0; per_field && f < n_fields; f++) {
        const size_t o = (size_t)f * NN;
        const ort_grid_out ff = from_ray(full, o), cc = from_ray(comp, o);
        rc = grid_enqueue(ctx, fields + f, 1, d_ys + (opts->ys_per_field ? (size_t)f * ny : 0), ny, d_xs, nx, stop, a_stop,
                          nullptr, 1, opts, ff, opts->compact ? &cc : nullptr, d_stats + f, d_partials + (size_t)f * gx,
                          d_tiles ? d_tiles + (size_t)f * compact_tile_ints(NN) : nullptr, gx, st);
        if (rc) return rc;
        CK(cudaEventRecord(ctx->ev_field[f], st));
        CK(cudaStreamWaitEvent(cs, ctx->ev_field[f], 0));
        CK(cudaMemcpyAsync(&hstats[f], d_stats + f, sizeof(ort_stats), cudaMemcpyDeviceToHost, cs));
        if ((rc = ort_copy_out(ctx, out, full, false, o, o, NN, 1, NN, cs))) return rc;
        size_t cnt = NN;
        if (opts->compact) {           // copy only the kept prefix: needs this field's count
            CK(cudaStreamSynchronize(cs));
            cnt = (size_t)hstats[f].n_kept;
        }
        if ((rc = ort_copy_out(ctx, out, src, true, o, o, cnt, 1, NN, cs))) return rc;
    }
    ort_stats hmerged[ORT_MAX_FIELDS];
    if (opts->gather_stats) {               // the statistics of the whole sharded grid: all-gather + rank-order merge
        ort_stats* d_merged; ENSURE(SL_MERGED, sizeof(ort_stats) * (size_t)n_fields, d_merged);
        rc = ort_comm_gather_stats(ctx, d_stats, n_fields, d_merged, nullptr, st);
        if (rc) return rc;
        CK(cudaMemcpyAsync(hmerged, d_merged, sizeof(ort_stats) * (size_t)n_fields, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaStreamSynchronize(cs));
    if (opts->gather_stats) {
        if (out->stats) memcpy(out->stats, hmerged, sizeof(ort_stats) * (size_t)n_fields);
        if (out->stats_local) memcpy(out->stats_local, hstats, sizeof(ort_stats) * (size_t)n_fields);
    } else if (out->stats) memcpy(out->stats, hstats, sizeof(ort_stats) * (size_t)n_fields);
    return ORT_OK;
}

}  // extern "C"

static int focus_check(ort_ctx* ctx, const ort_field* fields, int n_fields, const void* ys, int ny, const void* xs, int nx,
                       int stop, const double* foci, int n_foci, const ort_opts* opts, const ort_grid_out* out)
{
    if (!ctx) return ORT_EINVAL;
    if (!opts || !out) return fail(ctx, ORT_EINVAL, "trace3d_focus: opts/out is NULL");
    if (opts->ext) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_focus: opts.ext = %d (no OPD / vignetting through focus)", opts->ext);
    if (opts->gather_stats) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_focus: opts.gather_stats is not supported");
    if (ctx->have_layout && ctx->presc.poly) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_focus: polynomial terms are set on the context");
    const int rc = grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts, out);
    if (rc) return rc;
    if (n_foci < 1 || n_foci > ORT_MAX_FOCI) return fail(ctx, ORT_EINVAL, "trace3d_focus: n_foci = %d not in [1, %d]", n_foci, ORT_MAX_FOCI);
    if (!foci) return fail(ctx, ORT_EINVAL, "trace3d_focus: foci is NULL");
    for (int j = 0; j < n_foci; j++)
        if (!isfinite(foci[j])) return fail(ctx, ORT_EINVAL, "trace3d_focus: foci[%d] is not finite", j);
    const Presc& P = ctx->presc;
    const SurfK& S = P.s[P.nsurf - 1];
    if (!isinf(S.R) || S.K != 0.0) return fail(ctx, ORT_EINVAL, "trace3d_focus: the last row of the layout is not a plane");
    if (stop > P.nsurf - 1) return fail(ctx, ORT_EINVAL, "trace3d_focus: stop = %d is the image plane (at most %d)", stop, P.nsurf - 1);
    if (out->wx || out->wy || out->opd || out->stats_local)
        return fail(ctx, ORT_EINVAL, "trace3d_focus: wx, wy, opd and stats_local must be NULL");
    return ORT_OK;
}

extern "C" {

int ort_trace3d_focus_dev(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* d_ys, int ny,
                          const double* d_xs, int nx, int stop, double a_stop, const double* foci, int n_foci,
                          const ort_opts* opts, const ort_grid_out* d_out, void* stream)
{
    int rc = focus_check(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, foci, n_foci, opts, d_out);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const int gx = grid_dims(ctx, ctx->bps_focus, ORT_GRID_WAVES_DEFAULT, opts, n_fields, NN);
    const size_t nrec = (size_t)n_fields * n_foci;
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * nrec, d_partials);
    ort_stats* d_stats = d_out->stats;
    if (!d_stats) ENSURE(SL_STATS, sizeof(ort_stats) * nrec, d_stats);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, d_out, opts, true, NN, n_fields, n_foci, &full, &comp, &d_tiles))) return rc;
    return grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, foci, n_foci, opts, full,
                        opts->compact ? &comp : nullptr, d_stats, d_partials, d_tiles, gx, st);
}

int ort_trace3d_focus(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* ys, int ny,
                      const double* xs, int nx, int stop, double a_stop, const double* foci, int n_foci,
                      const ort_opts* opts, ort_grid_out* out)
{
    int rc = focus_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, foci, n_foci, opts, out);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const size_t tot = (size_t)NN * n_fields, nrec = (size_t)n_fields * n_foci;
    const int gx = grid_dims(ctx, ctx->bps_focus, ORT_GRID_WAVES_DEFAULT, opts, n_fields, NN);
    const size_t nys = (size_t)ny * (opts->ys_per_field ? n_fields : 1);
    double *d_ys, *d_xs;
    ENSURE(SL_YS, sizeof(double) * nys, d_ys);
    ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * nrec, d_partials);
    ort_stats* d_stats; ENSURE(SL_STATS, sizeof(ort_stats) * nrec, d_stats);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, out, opts, false, NN, n_fields, n_foci, &full, &comp, &d_tiles))) return rc;
    CK(cudaMemcpyAsync(d_ys, ys, sizeof(double) * nys, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
    rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, foci, n_foci, opts, full,
                      opts->compact ? &comp : nullptr, d_stats, d_partials, d_tiles, gx, st);
    if (rc) return rc;
    std::vector<ort_stats> hstats(nrec);
    CK(cudaMemcpyAsync(hstats.data(), d_stats, sizeof(ort_stats) * nrec, cudaMemcpyDeviceToHost, st));
    if (opts->compact) CK(cudaStreamSynchronize(st));                          // counts needed for the copy sizes
    const ort_grid_out& src = opts->compact ? comp : full;
    if ((rc = ort_copy_out(ctx, out, full, false, 0, 0, tot, n_foci, NN, st))) return rc;
    for (int f = 0; f < n_fields; f++) {
        const size_t o = (size_t)f * NN;
        const size_t cnt = opts->compact ? (size_t)hstats[(size_t)f * n_foci].n_kept : (size_t)NN;
        if ((rc = ort_copy_out(ctx, out, src, true, o, o, cnt, n_foci, NN, st))) return rc;
    }
    CK(cudaStreamSynchronize(st));
    if (out->stats) memcpy(out->stats, hstats.data(), sizeof(ort_stats) * nrec);
    return ORT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// encircled / ensquared energy of the spot (kern_energy.cu)
// ------------------------------------------------------------------------------------------
static int energy_req_check(ort_ctx* ctx, const ort_energy_req* req, const void* counts, const void* radius)
{
    if (!req) return fail(ctx, ORT_EINVAL, "spot_energy: req is NULL");
    if (req->metric != ORT_ENERGY_CIRCLE && req->metric != ORT_ENERGY_SQUARE)
        return fail(ctx, ORT_EINVAL, "spot_energy: metric = %d", req->metric);
    if (req->center != ORT_CENTER_CENTROID && req->center != ORT_CENTER_PARAXIAL)
        return fail(ctx, ORT_EINVAL, "spot_energy: center = %d", req->center);
    if (req->n_radii < 0 || req->n_radii > ORT_MAX_RADII)
        return fail(ctx, ORT_EINVAL, "spot_energy: n_radii = %d not in [0, %d]", req->n_radii, ORT_MAX_RADII);
    if (req->n_fracs < 0 || req->n_fracs > ORT_MAX_FRACS)
        return fail(ctx, ORT_EINVAL, "spot_energy: n_fracs = %d not in [0, %d]", req->n_fracs, ORT_MAX_FRACS);
    if (!req->n_radii && !req->n_fracs) return fail(ctx, ORT_EINVAL, "spot_energy: neither radii nor fractions");
    if (req->n_radii && (!req->radii || !counts)) return fail(ctx, ORT_EINVAL, "spot_energy: radii or counts is NULL");
    if (req->n_fracs && (!req->fracs || !radius)) return fail(ctx, ORT_EINVAL, "spot_energy: fracs or radius is NULL");
    for (int k = 0; k < req->n_radii; k++) {
        const double r = req->radii[k];
        if (!isfinite(r) || !(r >= 0.0)) return fail(ctx, ORT_EINVAL, "spot_energy: radii[%d] = %g is not finite and >= 0", k, r);
        if (k && !(r > req->radii[k - 1])) return fail(ctx, ORT_EINVAL, "spot_energy: radii are not strictly ascending at %d", k);
    }
    for (int i = 0; i < req->n_fracs; i++) {
        const double q = req->fracs[i];
        if (!(q > 0.0 && q <= 1.0)) return fail(ctx, ORT_EINVAL, "spot_energy: fracs[%d] = %g not in (0, 1]", i, q);
    }
    return ORT_OK;
}

static int energy_sets_check(ort_ctx* ctx, const ort_spot_sets* S)
{
    if (!S) return fail(ctx, ORT_EINVAL, "spot_energy: sets is NULL");
    if (S->n_sets < 1 || S->n_sets > ORT_MAX_FIELDS * ORT_MAX_FOCI)
        return fail(ctx, ORT_EINVAL, "spot_energy: n_sets = %d not in [1, %d]", S->n_sets, ORT_MAX_FIELDS * ORT_MAX_FOCI);
    if (S->sets_per_mask < 1) return fail(ctx, ORT_EINVAL, "spot_energy: sets_per_mask = %d", S->sets_per_mask);
    if (S->stride <= 0 || S->stride >= (1LL << 31))
        return fail(ctx, ORT_EINVAL, "spot_energy: stride = %lld not in [1, 2^31)", (long long)S->stride);
    if (!S->ex || !S->ey || !S->stats) return fail(ctx, ORT_EINVAL, "spot_energy: ex, ey or stats is NULL");
    return ORT_OK;
}

// Enqueue the energy kernels over `sets` on st (inside the entry point's ScratchScope); one ProfScope around all of them
static int energy_enqueue(ort_ctx* ctx, const ort_spot_sets& S, const ort_energy_req* req, int64_t* d_counts,
                          double* d_radius, cudaStream_t st)
{
    EnergyArgs A;
    memset(&A, 0, sizeof A);
    A.n_sets = S.n_sets; A.sets_per_mask = S.sets_per_mask; A.stride = S.stride;
    A.ex = S.ex; A.ey = S.ey; A.mask = S.mask; A.stats = S.stats;
    A.metric = req->metric; A.center = req->center; A.n_radii = req->n_radii; A.n_fracs = req->n_fracs;
    for (int i = 0; i < req->n_fracs; i++) A.fracs[i] = req->fracs[i];
    A.cap = energy_cand_cap(S.stride, S.n_sets);
    const size_t ns = (size_t)S.n_sets;
    ENSURE(SL_EN_STATE, sizeof(EnergyState) * ns, A.state);
    ENSURE(SL_EN_HIST, sizeof(unsigned) * energy_hist_words(req->n_fracs) * ns, A.hist);
    ENSURE(SL_EN_BINS, sizeof(unsigned long long) * (size_t)(req->n_radii + 1) * ns, A.bins);
    ENSURE(SL_EN_CAND0, sizeof(unsigned long long) * A.cap * ns, A.cand[0]);
    ENSURE(SL_EN_CAND1, sizeof(unsigned long long) * A.cap * ns, A.cand[1]);
    A.counts = (long long*)d_counts; A.radius = d_radius;
    int n = 0;
    {
        ProfScope prof(ctx, st);
        CK(launch_energy(A, req->radii, ctx->sm_count, st, &n));
    }
    ctx->launches += n;
    return ORT_OK;
}

extern "C" {

int ort_spot_energy_dev(ort_ctx* ctx, const ort_spot_sets* sets, const ort_energy_req* req, int64_t* d_counts,
                        double* d_radius, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    int rc = energy_sets_check(ctx, sets);
    if (rc || (rc = energy_req_check(ctx, req, d_counts, d_radius))) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    ScratchScope scratch(ctx, st);
    return energy_enqueue(ctx, *sets, req, d_counts, d_radius, st);
}

int ort_trace3d_energy(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* ys, int ny, const double* xs,
                       int nx, int stop, double a_stop, const double* foci, int n_foci, const ort_opts* opts,
                       const ort_energy_req* req, ort_stats* stats, int64_t* counts, double* radius)
{
    if (!ctx) return ORT_EINVAL;
    if (!opts) return fail(ctx, ORT_EINVAL, "trace3d_energy: opts is NULL");
    if (opts->gather_stats) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_energy: opts.gather_stats is not supported");
    if (opts->compact) return fail(ctx, ORT_EINVAL, "trace3d_energy: opts.compact must be 0");
    if (n_foci < 0) return fail(ctx, ORT_EINVAL, "trace3d_energy: n_foci = %d", n_foci);
    // the members the energy reads; ort_sweep_scratch traces each one a host call wants into its scratch slot
    static double tag; static uint8_t mtag;
    ort_grid_out want;
    memset(&want, 0, sizeof want);
    want.ex = want.ey = &tag; want.mask = &mtag; want.stats = nullptr;
    int rc = n_foci ? focus_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, foci, n_foci, opts, &want)
                    : grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts, &want);
    if (rc || (rc = energy_req_check(ctx, req, counts, radius))) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    const int M = n_foci ? n_foci : 1;
    const unsigned NN = (unsigned)((long long)ny * nx);
    const size_t nrec = (size_t)n_fields * M;
    const int gx = n_foci ? grid_dims(ctx, ctx->bps_focus, ORT_GRID_WAVES_DEFAULT, opts, n_fields, NN)
                          : grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, n_fields, NN);
    const size_t nys = (size_t)ny * (opts->ys_per_field ? n_fields : 1);
    double *d_ys, *d_xs;
    ENSURE(SL_YS, sizeof(double) * nys, d_ys);
    ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * nrec, d_partials);
    ort_stats* d_stats; ENSURE(SL_STATS, sizeof(ort_stats) * nrec, d_stats);
    int64_t* d_counts; ENSURE(SL_EN_COUNTS, sizeof(int64_t) * nrec * (size_t)req->n_radii, d_counts);
    double* d_radius; ENSURE(SL_EN_RADIUS, sizeof(double) * nrec * (size_t)req->n_fracs, d_radius);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, &want, opts, false, NN, n_fields, M, &full, &comp, &d_tiles))) return rc;
    CK(cudaMemcpyAsync(d_ys, ys, sizeof(double) * nys, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
    rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, n_foci ? foci : nullptr, M, opts, full,
                      nullptr, d_stats, d_partials, nullptr, gx, st);
    if (rc) return rc;
    ort_spot_sets S;
    memset(&S, 0, sizeof S);
    S.n_sets = (int32_t)nrec; S.sets_per_mask = M; S.stride = NN;
    S.ex = full.ex; S.ey = full.ey; S.mask = full.mask; S.stats = d_stats;
    if ((rc = energy_enqueue(ctx, S, req, d_counts, d_radius, st))) return rc;
    if (stats) CK(cudaMemcpyAsync(stats, d_stats, sizeof(ort_stats) * nrec, cudaMemcpyDeviceToHost, st));
    if (req->n_radii) CK(cudaMemcpyAsync(counts, d_counts, sizeof(int64_t) * nrec * req->n_radii, cudaMemcpyDeviceToHost, st));
    if (req->n_fracs) CK(cudaMemcpyAsync(radius, d_radius, sizeof(double) * nrec * req->n_fracs, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// Zernike fit of the wavefront (kern_zernike.cu)
// ------------------------------------------------------------------------------------------
static int zernike_req_check(ort_ctx* ctx, const ort_zernike_req* req, const void* coef, const void* resid,
                             const void* status)
{
    if (!req) return fail(ctx, ORT_EINVAL, "zernike: req is NULL");
    if (req->n_max < 0 || req->n_max > ORT_ZERN_MAX_ORDER)
        return fail(ctx, ORT_EINVAL, "zernike: n_max = %d not in [0, %d]", req->n_max, ORT_ZERN_MAX_ORDER);
    if (!isfinite(req->r_norm) || req->r_norm < 0.0)
        return fail(ctx, ORT_EINVAL, "zernike: r_norm = %g is not finite and >= 0", req->r_norm);
    if (!coef || !resid || !status) return fail(ctx, ORT_EINVAL, "zernike: coef, resid or status is NULL");
    return ORT_OK;
}

// Enqueue the four fit kernels over `sets` on st (inside the entry point's ScratchScope); one ProfScope around them
static int zernike_enqueue(ort_ctx* ctx, const ort_wave_sets& S, const ort_zernike_req* req, double* d_coef,
                           double* d_resid, int32_t* d_status, cudaStream_t st)
{
    ZernArgs A;
    memset(&A, 0, sizeof A);
    A.n_sets = S.n_sets; A.n_max = req->n_max; A.stride = S.stride;
    A.opd = S.opd; A.r = S.r; A.theta = S.theta; A.mask = S.mask; A.stats = S.stats;
    A.r_norm = req->r_norm;
    CK(zern_dims(A, ctx->sm_count));
    const size_t ns = (size_t)S.n_sets;
    ENSURE(SL_ZN_GPART, sizeof(double) * zern_gram_record(A) * (size_t)A.gx * ns, A.gpart);
    ENSURE(SL_ZN_RPART, sizeof(double) * 3 * (size_t)A.gx_resid * ns, A.rpart);
    ENSURE(SL_ZN_CSYM, sizeof(double) * zern_fitted_terms(ORT_ZERN_MAX_ORDER) * ns, A.csym);
    A.coef = d_coef; A.resid = d_resid; A.status = (int*)d_status;
    int n = 0;
    {
        ProfScope prof(ctx, st);
        CK(launch_zernike(A, st, &n));
    }
    ctx->launches += n;
    return ORT_OK;
}

extern "C" {

int ort_wavefront_zernike_dev(ort_ctx* ctx, const ort_wave_sets* sets, const ort_zernike_req* req, double* d_coef,
                              double* d_resid, int32_t* d_status, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (!sets) return fail(ctx, ORT_EINVAL, "wavefront_zernike: sets is NULL");
    if (sets->n_sets < 1 || sets->n_sets > ORT_MAX_FIELDS)
        return fail(ctx, ORT_EINVAL, "wavefront_zernike: n_sets = %d not in [1, %d]", sets->n_sets, ORT_MAX_FIELDS);
    if (sets->stride <= 0 || sets->stride >= (1LL << 31))
        return fail(ctx, ORT_EINVAL, "wavefront_zernike: stride = %lld not in [1, 2^31)", (long long)sets->stride);
    if (!sets->opd || !sets->r || !sets->theta || !sets->stats)
        return fail(ctx, ORT_EINVAL, "wavefront_zernike: opd, r, theta or stats is NULL");
    int rc = zernike_req_check(ctx, req, d_coef, d_resid, d_status);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    ScratchScope scratch(ctx, st);
    return zernike_enqueue(ctx, *sets, req, d_coef, d_resid, d_status, st);
}

int ort_trace3d_zernike(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* ys, int ny, const double* xs,
                        int nx, int stop, double a_stop, const ort_opts* opts, const ort_zernike_req* req,
                        ort_stats* stats, double* coef, double* resid, int32_t* status)
{
    if (!ctx) return ORT_EINVAL;
    if (!opts) return fail(ctx, ORT_EINVAL, "trace3d_zernike: opts is NULL");
    if (opts->gather_stats) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_zernike: opts.gather_stats is not supported");
    if (opts->compact) return fail(ctx, ORT_EINVAL, "trace3d_zernike: opts.compact must be 0");
    if (!(opts->ext & ORT_EXT_OPD)) return fail(ctx, ORT_EINVAL, "trace3d_zernike: opts.ext must hold ORT_EXT_OPD");
    // the members the fit reads; ort_sweep_scratch traces each one a host call wants into its scratch slot
    static double tag; static uint8_t mtag;
    ort_grid_out want;
    memset(&want, 0, sizeof want);
    want.opd = want.r = want.theta = &tag; want.mask = &mtag;
    int rc = grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts, &want);
    if (rc || (rc = zernike_req_check(ctx, req, coef, resid, status))) return rc;
    if ((long long)ny * nx == 0) return fail(ctx, ORT_EINVAL, "trace3d_zernike: empty grid");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const size_t nf = (size_t)n_fields, J = (size_t)(req->n_max + 1) * (req->n_max + 2) / 2;
    const int gx = grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, n_fields, NN);
    const size_t nys = (size_t)ny * (opts->ys_per_field ? n_fields : 1);
    double *d_ys, *d_xs;
    ENSURE(SL_YS, sizeof(double) * nys, d_ys);
    ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * nf, d_partials);
    ort_stats* d_stats; ENSURE(SL_STATS, sizeof(ort_stats) * nf, d_stats);
    double* d_coef; ENSURE(SL_ZN_COEF, sizeof(double) * nf * J, d_coef);
    double* d_resid; ENSURE(SL_ZN_RESID, sizeof(double) * nf * 2, d_resid);
    int32_t* d_status; ENSURE(SL_ZN_STATUS, sizeof(int32_t) * nf, d_status);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, &want, opts, false, NN, n_fields, 1, &full, &comp, &d_tiles))) return rc;
    CK(cudaMemcpyAsync(d_ys, ys, sizeof(double) * nys, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
    rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, nullptr, 1, opts, full, nullptr, d_stats,
                      d_partials, nullptr, gx, st);
    if (rc) return rc;
    ort_wave_sets S;
    memset(&S, 0, sizeof S);
    S.n_sets = n_fields; S.stride = NN;
    S.opd = full.opd; S.r = full.r; S.theta = full.theta; S.mask = full.mask; S.stats = d_stats;
    if ((rc = zernike_enqueue(ctx, S, req, d_coef, d_resid, d_status, st))) return rc;
    if (stats) CK(cudaMemcpyAsync(stats, d_stats, sizeof(ort_stats) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(coef, d_coef, sizeof(double) * nf * J, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(resid, d_resid, sizeof(double) * nf * 2, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, d_status, sizeof(int32_t) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// Diffraction PSF of the wavefront (kern_psf.cu)
// ------------------------------------------------------------------------------------------
static int psf_req_check(ort_ctx* ctx, const ort_psf_req* req, const void* psf, const void* strehl, const void* peak,
                         const void* status)
{
    if (!req) return fail(ctx, ORT_EINVAL, "psf: req is NULL");
    if (req->n_u < 1 || req->n_u > ORT_PSF_MAX_SIDE || req->n_v < 1 || req->n_v > ORT_PSF_MAX_SIDE)
        return fail(ctx, ORT_EINVAL, "psf: n_u = %d, n_v = %d not in [1, %d]", req->n_u, req->n_v, ORT_PSF_MAX_SIDE);
    if (!(isfinite(req->du) && req->du > 0.0) || !(isfinite(req->dv) && req->dv > 0.0) ||
        !(isfinite(req->scale) && req->scale > 0.0))
        return fail(ctx, ORT_EINVAL, "psf: du = %g, dv = %g, scale = %g must be finite and > 0", req->du, req->dv,
                    req->scale);
    if (!psf || !strehl || !peak || !status) return fail(ctx, ORT_EINVAL, "psf: psf, strehl, peak or status is NULL");
    return ORT_OK;
}

// Enqueue the five PSF kernels over `sets` on st (inside the entry point's ScratchScope); one ProfScope around them
static int psf_enqueue(ort_ctx* ctx, const ort_wave_sets& S, const double* d_ys, int ys_per_set, int ny,
                       const double* d_xs, int nx, const ort_psf_req* req, double* d_psf, double* d_strehl,
                       int32_t* d_peak, int32_t* d_status, cudaStream_t st)
{
    PsfArgs A;
    memset(&A, 0, sizeof A);
    A.n_sets = S.n_sets; A.ny = ny; A.nx = nx; A.stride = S.stride;
    A.opd = S.opd; A.mask = S.mask; A.stats = S.stats;
    A.ys = d_ys; A.ys_stride = ys_per_set ? ny : 0; A.xs = d_xs;
    A.n_u = req->n_u; A.n_v = req->n_v; A.du = req->du; A.dv = req->dv; A.scale = req->scale;
    CK(psf_dims(A, ctx->sm_count));
    const size_t ns = (size_t)S.n_sets;
    ENSURE(SL_PSF_CTAB, sizeof(double) * (size_t)nx * A.nup, A.ctab);
    ENSURE(SL_PSF_T, sizeof(double2) * ns * A.kx * (size_t)ny * A.nup, A.T);
    ENSURE(SL_PSF_RSUM, sizeof(double) * 3 * ns * A.rt * A.kx, A.rsum);
    ENSURE(SL_PSF_E, sizeof(double2) * ns * A.ky * A.n_v * A.nuh, A.E);
    ENSURE(SL_PSF_BVAL, sizeof(double) * ns * A.fb, A.bval);
    ENSURE(SL_PSF_BIDX, sizeof(int) * ns * A.fb, A.bidx);
    A.psf = d_psf; A.strehl = d_strehl; A.peak = (int*)d_peak; A.status = (int*)d_status;
    int n = 0;
    {
        ProfScope prof(ctx, st);
        CK(launch_psf(A, st, &n));
    }
    ctx->launches += n;
    return ORT_OK;
}

extern "C" {

int ort_wavefront_psf_dev(ort_ctx* ctx, const ort_wave_sets* sets, const double* d_ys, int ys_per_set, int ny,
                          const double* d_xs, int nx, const ort_psf_req* req, double* d_psf, double* d_strehl,
                          int32_t* d_peak, int32_t* d_status, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (!sets) return fail(ctx, ORT_EINVAL, "wavefront_psf: sets is NULL");
    if (sets->n_sets < 1 || sets->n_sets > ORT_MAX_FIELDS)
        return fail(ctx, ORT_EINVAL, "wavefront_psf: n_sets = %d not in [1, %d]", sets->n_sets, ORT_MAX_FIELDS);
    if (ny < 1 || nx < 1 || sets->stride != (long long)ny * nx || sets->stride >= (1LL << 31))
        return fail(ctx, ORT_EINVAL, "wavefront_psf: stride = %lld is not ny*nx = %d*%d >= 1 (< 2^31)",
                    (long long)sets->stride, ny, nx);
    if (!sets->opd || !sets->mask || !sets->stats || !d_ys || !d_xs)
        return fail(ctx, ORT_EINVAL, "wavefront_psf: opd, mask, stats, ys or xs is NULL");
    int rc = psf_req_check(ctx, req, d_psf, d_strehl, d_peak, d_status);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    ScratchScope scratch(ctx, st);
    return psf_enqueue(ctx, *sets, d_ys, ys_per_set, ny, d_xs, nx, req, d_psf, d_strehl, d_peak, d_status, st);
}

int ort_trace3d_psf(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* ys, int ny, const double* xs, int nx,
                    int stop, double a_stop, const ort_opts* opts, const ort_psf_req* req, ort_stats* stats, double* psf,
                    double* strehl, int32_t* peak, int32_t* status)
{
    if (!ctx) return ORT_EINVAL;
    if (!opts) return fail(ctx, ORT_EINVAL, "trace3d_psf: opts is NULL");
    if (opts->gather_stats) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_psf: opts.gather_stats is not supported");
    if (opts->compact) return fail(ctx, ORT_EINVAL, "trace3d_psf: opts.compact must be 0");
    if (!(opts->ext & ORT_EXT_OPD)) return fail(ctx, ORT_EINVAL, "trace3d_psf: opts.ext must hold ORT_EXT_OPD");
    // the members the PSF reads; ort_sweep_scratch traces each one a host call wants into its scratch slot
    static double tag; static uint8_t mtag;
    ort_grid_out want;
    memset(&want, 0, sizeof want);
    want.opd = &tag; want.mask = &mtag;
    int rc = grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts, &want);
    if (rc || (rc = psf_req_check(ctx, req, psf, strehl, peak, status))) return rc;
    if (ny < 1 || nx < 1) return fail(ctx, ORT_EINVAL, "trace3d_psf: empty grid");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const size_t nf = (size_t)n_fields, npix = (size_t)req->n_u * req->n_v;
    const int gx = grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, n_fields, NN);
    const size_t nys = (size_t)ny * (opts->ys_per_field ? n_fields : 1);
    double *d_ys, *d_xs;
    ENSURE(SL_YS, sizeof(double) * nys, d_ys);
    ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * nf, d_partials);
    ort_stats* d_stats; ENSURE(SL_STATS, sizeof(ort_stats) * nf, d_stats);
    double* d_psf; ENSURE(SL_PSF_OUT, sizeof(double) * nf * npix, d_psf);
    double* d_strehl; ENSURE(SL_PSF_STREHL, sizeof(double) * nf * 2, d_strehl);
    int32_t* d_peak; ENSURE(SL_PSF_PEAK, sizeof(int32_t) * nf, d_peak);
    int32_t* d_status; ENSURE(SL_PSF_STATUS, sizeof(int32_t) * nf, d_status);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, &want, opts, false, NN, n_fields, 1, &full, &comp, &d_tiles))) return rc;
    CK(cudaMemcpyAsync(d_ys, ys, sizeof(double) * nys, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
    rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, nullptr, 1, opts, full, nullptr, d_stats,
                      d_partials, nullptr, gx, st);
    if (rc) return rc;
    ort_wave_sets S;
    memset(&S, 0, sizeof S);
    S.n_sets = n_fields; S.stride = NN;
    S.opd = full.opd; S.mask = full.mask; S.stats = d_stats;
    if ((rc = psf_enqueue(ctx, S, d_ys, opts->ys_per_field, ny, d_xs, nx, req, d_psf, d_strehl, d_peak, d_status, st)))
        return rc;
    if (stats) CK(cudaMemcpyAsync(stats, d_stats, sizeof(ort_stats) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(psf, d_psf, sizeof(double) * nf * npix, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(strehl, d_strehl, sizeof(double) * nf * 2, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(peak, d_peak, sizeof(int32_t) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, d_status, sizeof(int32_t) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// Diffraction MTF of the wavefront (kern_mtf.cu)
// ------------------------------------------------------------------------------------------
static int mtf_req_check(ort_ctx* ctx, const ort_mtf_req* req, const void* otf, const void* status)
{
    if (!req) return fail(ctx, ORT_EINVAL, "mtf: req is NULL");
    if (req->n_freq < 1 || req->n_freq > ORT_MTF_MAX_FREQS)
        return fail(ctx, ORT_EINVAL, "mtf: n_freq = %d not in [1, %d]", req->n_freq, ORT_MTF_MAX_FREQS);
    if (!req->freqs) return fail(ctx, ORT_EINVAL, "mtf: freqs is NULL");
    for (int i = 0; i < req->n_freq; i++)
        if (!(isfinite(req->freqs[i]) && req->freqs[i] >= 0.0))
            return fail(ctx, ORT_EINVAL, "mtf: freqs[%d] = %g must be finite and >= 0", i, req->freqs[i]);
    if (!(isfinite(req->scale) && req->scale > 0.0))
        return fail(ctx, ORT_EINVAL, "mtf: scale = %g must be finite and > 0", req->scale);
    if (!otf || !status) return fail(ctx, ORT_EINVAL, "mtf: otf or status is NULL");
    return ORT_OK;
}

// Enqueue the four MTF kernels over `sets` on st (inside the entry point's ScratchScope); one ProfScope around them
static int mtf_enqueue(ort_ctx* ctx, const ort_wave_sets& S, const double* d_ys, int ys_per_set, int ny,
                       const double* d_xs, int nx, const ort_mtf_req* req, double* d_otf, int32_t* d_status,
                       cudaStream_t st)
{
    MtfArgs A;
    memset(&A, 0, sizeof A);
    A.n_sets = S.n_sets; A.ny = ny; A.nx = nx; A.stride = S.stride;
    A.opd = S.opd; A.mask = S.mask; A.stats = S.stats;
    A.ys = d_ys; A.ys_stride = ys_per_set ? ny : 0; A.xs = d_xs;
    A.n_freq = req->n_freq; A.scale = req->scale;
    memcpy(A.freqs, req->freqs, sizeof(double) * (size_t)req->n_freq);
    if (ctx->mtf_occ[0][0] == 0) CK(mtf_occupancy(ctx->mtf_occ));
    CK(mtf_dims(A, ctx->sm_count, ctx->mtf_occ));
    const size_t ns = (size_t)S.n_sets;
    ENSURE(SL_MTF_P, sizeof(double2) * ns * (size_t)S.stride, A.P);
    ENSURE(SL_MTF_PT, sizeof(double2) * ns * (size_t)S.stride, A.PT);
    ENSURE(SL_MTF_BAD, sizeof(uint8_t) * ns * (size_t)A.tiles, A.bad);
    ENSURE(SL_MTF_PSAG, sizeof(double) * ns * A.rg_s * A.n_slot, A.psag);
    ENSURE(SL_MTF_PTAN, sizeof(double2) * ns * A.rg_t * A.n_slot, A.ptan);
    A.otf = d_otf; A.status = (int*)d_status;
    int n = 0;
    {
        ProfScope prof(ctx, st);
        CK(launch_mtf(A, st, &n));
    }
    ctx->launches += n;
    return ORT_OK;
}

extern "C" {

int ort_wavefront_mtf_dev(ort_ctx* ctx, const ort_wave_sets* sets, const double* d_ys, int ys_per_set, int ny,
                          const double* d_xs, int nx, const ort_mtf_req* req, double* d_otf, int32_t* d_status,
                          void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (!sets) return fail(ctx, ORT_EINVAL, "wavefront_mtf: sets is NULL");
    if (sets->n_sets < 1 || sets->n_sets > ORT_MAX_FIELDS)
        return fail(ctx, ORT_EINVAL, "wavefront_mtf: n_sets = %d not in [1, %d]", sets->n_sets, ORT_MAX_FIELDS);
    if (ny < 2 || nx < 2 || sets->stride != (long long)ny * nx || sets->stride >= (1LL << 31))
        return fail(ctx, ORT_EINVAL, "wavefront_mtf: stride = %lld is not ny*nx = %d*%d with ny, nx >= 2 (< 2^31)",
                    (long long)sets->stride, ny, nx);
    if (!sets->opd || !sets->mask || !sets->stats || !d_ys || !d_xs)
        return fail(ctx, ORT_EINVAL, "wavefront_mtf: opd, mask, stats, ys or xs is NULL");
    int rc = mtf_req_check(ctx, req, d_otf, d_status);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    ScratchScope scratch(ctx, st);
    return mtf_enqueue(ctx, *sets, d_ys, ys_per_set, ny, d_xs, nx, req, d_otf, d_status, st);
}

int ort_trace3d_mtf(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* ys, int ny, const double* xs, int nx,
                    int stop, double a_stop, const ort_opts* opts, const ort_mtf_req* req, ort_stats* stats, double* otf,
                    int32_t* status)
{
    if (!ctx) return ORT_EINVAL;
    if (!opts) return fail(ctx, ORT_EINVAL, "trace3d_mtf: opts is NULL");
    if (opts->gather_stats) return fail(ctx, ORT_EUNSUPPORTED, "trace3d_mtf: opts.gather_stats is not supported");
    if (opts->compact) return fail(ctx, ORT_EINVAL, "trace3d_mtf: opts.compact must be 0");
    if (!(opts->ext & ORT_EXT_OPD)) return fail(ctx, ORT_EINVAL, "trace3d_mtf: opts.ext must hold ORT_EXT_OPD");
    // the members the MTF reads; ort_sweep_scratch traces each one a host call wants into its scratch slot
    static double tag; static uint8_t mtag;
    ort_grid_out want;
    memset(&want, 0, sizeof want);
    want.opd = &tag; want.mask = &mtag;
    int rc = grid_check(ctx, fields, n_fields, ys, ny, xs, nx, stop, opts, &want);
    if (rc || (rc = mtf_req_check(ctx, req, otf, status))) return rc;
    if (ny < 2 || nx < 2) return fail(ctx, ORT_EINVAL, "trace3d_mtf: ny = %d, nx = %d must be >= 2", ny, nx);
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    const unsigned NN = (unsigned)((long long)ny * nx);
    const size_t nf = (size_t)n_fields, nout = 4 * (size_t)req->n_freq;
    const int gx = grid_dims(ctx, ctx->bps, ort_grid_waves(), opts, n_fields, NN);
    const size_t nys = (size_t)ny * (opts->ys_per_field ? n_fields : 1);
    double *d_ys, *d_xs;
    ENSURE(SL_YS, sizeof(double) * nys, d_ys);
    ENSURE(SL_XS, sizeof(double) * (size_t)nx, d_xs);
    RawPart* d_partials; ENSURE(SL_PARTIALS, sizeof(RawPart) * (size_t)gx * nf, d_partials);
    ort_stats* d_stats; ENSURE(SL_STATS, sizeof(ort_stats) * nf, d_stats);
    double* d_otf; ENSURE(SL_MTF_OTF, sizeof(double) * nf * nout, d_otf);
    int32_t* d_status; ENSURE(SL_MTF_STATUS, sizeof(int32_t) * nf, d_status);
    ort_grid_out full, comp; int* d_tiles;
    if ((rc = ort_sweep_scratch(ctx, &want, opts, false, NN, n_fields, 1, &full, &comp, &d_tiles))) return rc;
    CK(cudaMemcpyAsync(d_ys, ys, sizeof(double) * nys, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, sizeof(double) * (size_t)nx, cudaMemcpyHostToDevice, st));
    rc = grid_enqueue(ctx, fields, n_fields, d_ys, ny, d_xs, nx, stop, a_stop, nullptr, 1, opts, full, nullptr, d_stats,
                      d_partials, nullptr, gx, st);
    if (rc) return rc;
    ort_wave_sets S;
    memset(&S, 0, sizeof S);
    S.n_sets = n_fields; S.stride = NN;
    S.opd = full.opd; S.mask = full.mask; S.stats = d_stats;
    if ((rc = mtf_enqueue(ctx, S, d_ys, opts->ys_per_field, ny, d_xs, nx, req, d_otf, d_status, st))) return rc;
    if (stats) CK(cudaMemcpyAsync(stats, d_stats, sizeof(ort_stats) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(otf, d_otf, sizeof(double) * nf * nout, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, d_status, sizeof(int32_t) * nf, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

// ------------------------------------------------------------------------------------------
// arbitrary rays / 2-D / paraxial / transfer / candidates: host wrappers stage through scratch
// ------------------------------------------------------------------------------------------
int ort_trace3d_rays_opl(ort_ctx* ctx, int64_t N, const double* y0, const double* x0, const double* u0,
                         const double* v0, int arith, double* xv, double* yv, double* kout, uint8_t* flags,
                         double* opl)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "trace3d_rays: call ort_set_layout first");
    if (N < 0 || !y0 || !x0 || !u0 || !v0) return fail(ctx, ORT_EINVAL, "trace3d_rays: bad input");
    if (arith != ORT_ARITH_STRICT && arith != ORT_ARITH_FAST) return fail(ctx, ORT_EINVAL, "trace3d_rays: arith = %d", arith);
    if (N == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N, ns = (size_t)ctx->presc.nsurf;
    RaysArgs A; memset(&A, 0, sizeof A);
    A.N = N;
    double *d0, *d1, *d2, *d3;
    ENSURE(SL_IN0, n * 8, d0); ENSURE(SL_IN1, n * 8, d1); ENSURE(SL_IN2, n * 8, d2); ENSURE(SL_IN3, n * 8, d3);
    if (xv) ENSURE(SL_OUT0, ns * n * 8, A.xv);
    if (yv) ENSURE(SL_OUT1, ns * n * 8, A.yv);
    if (kout) ENSURE(SL_OUT2, 3 * n * 8, A.kout);
    if (flags) ENSURE(SL_OUT3, n, A.flags);
    if (opl) ENSURE(SL_OUT4, n * 8, A.opl);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d0, y0, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d1, x0, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d2, u0, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d3, v0, n * 8, cudaMemcpyHostToDevice, st));
    A.y0 = d0; A.x0 = d1; A.u0 = d2; A.v0 = d3;
    CK(launch_rays(ctx->presc, A, resolve_arith(ctx, arith), st));
    ctx->launches++;
    if (xv) CK(cudaMemcpyAsync(xv, A.xv, ns * n * 8, cudaMemcpyDeviceToHost, st));
    if (yv) CK(cudaMemcpyAsync(yv, A.yv, ns * n * 8, cudaMemcpyDeviceToHost, st));
    if (kout) CK(cudaMemcpyAsync(kout, A.kout, 3 * n * 8, cudaMemcpyDeviceToHost, st));
    if (flags) CK(cudaMemcpyAsync(flags, A.flags, n, cudaMemcpyDeviceToHost, st));
    if (opl) CK(cudaMemcpyAsync(opl, A.opl, n * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_trace3d_rays_dev(ort_ctx* ctx, int64_t N, const double* d_y0, const double* d_x0, const double* d_u0,
                         const double* d_v0, int arith, double* d_xv, double* d_yv, double* d_kout, uint8_t* d_flags,
                         double* d_opl, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "trace3d_rays: call ort_set_layout first");
    if (N < 0 || !d_y0 || !d_x0 || !d_u0 || !d_v0) return fail(ctx, ORT_EINVAL, "trace3d_rays: bad input");
    if (arith != ORT_ARITH_STRICT && arith != ORT_ARITH_FAST) return fail(ctx, ORT_EINVAL, "trace3d_rays: arith = %d", arith);
    if (N == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    RaysArgs A; memset(&A, 0, sizeof A);
    A.N = N; A.y0 = d_y0; A.x0 = d_x0; A.u0 = d_u0; A.v0 = d_v0;
    A.xv = d_xv; A.yv = d_yv; A.kout = d_kout; A.flags = d_flags; A.opl = d_opl;
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_rays(ctx->presc, A, resolve_arith(ctx, arith), (cudaStream_t)stream));
    }
    ctx->launches++;
    return ORT_OK;
}

int ort_trace3d_rays(ort_ctx* ctx, int64_t N, const double* y0, const double* x0, const double* u0,
                     const double* v0, int arith, double* xv, double* yv, double* kout, uint8_t* flags)
{
    return ort_trace3d_rays_opl(ctx, N, y0, x0, u0, v0, arith, xv, yv, kout, flags, nullptr);
}

int ort_trace2d_batch(ort_ctx* ctx, int64_t N, const double* y0, const double* U0, int aspheric,
                      double* y_out, double* U_out, double* ts_out, uint8_t* flags)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "trace2d_batch: call ort_set_layout first");
    if (N < 0 || !y0 || !U0) return fail(ctx, ORT_EINVAL, "trace2d_batch: bad input");
    if (N == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N, rows = (size_t)ctx->rows;
    Trace2dArgs A; memset(&A, 0, sizeof A);
    A.N = N; A.aspheric = aspheric ? 1 : 0;
    double *d0, *d1;
    ENSURE(SL_IN0, n * 8, d0); ENSURE(SL_IN1, n * 8, d1);
    if (y_out) ENSURE(SL_OUT0, rows * n * 8, A.y_out);
    if (U_out) ENSURE(SL_OUT1, rows * n * 8, A.U_out);
    if (ts_out) ENSURE(SL_OUT2, rows * n * 8, A.ts_out);
    if (flags) ENSURE(SL_OUT3, n, A.flags);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d0, y0, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d1, U0, n * 8, cudaMemcpyHostToDevice, st));
    A.y0 = d0; A.U0 = d1;
    CK(launch_trace2d(ctx->presc, A, st));
    ctx->launches++;
    if (y_out) CK(cudaMemcpyAsync(y_out, A.y_out, rows * n * 8, cudaMemcpyDeviceToHost, st));
    if (U_out) CK(cudaMemcpyAsync(U_out, A.U_out, rows * n * 8, cudaMemcpyDeviceToHost, st));
    if (ts_out) CK(cudaMemcpyAsync(ts_out, A.ts_out, rows * n * 8, cudaMemcpyDeviceToHost, st));
    if (flags) CK(cudaMemcpyAsync(flags, A.flags, n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_aim2d(ort_ctx* ctx, int64_t N, const double* x_start, const double* other, const double* target, int stop,
              int vary_u, int mode, double atol_or_scale, int aspheric, double* x_out, int32_t* iters)
{
    if (!ctx) return ORT_EINVAL;
    if (!ctx->have_layout) return fail(ctx, ORT_EINVAL, "aim2d: call ort_set_layout first");
    if (N < 0 || !x_start || !other || !target || !x_out) return fail(ctx, ORT_EINVAL, "aim2d: bad input");
    if (stop < 1 || stop > ctx->presc.nsurf) return fail(ctx, ORT_EINVAL, "aim2d: stop = %d not in [1, %d]", stop, ctx->presc.nsurf);
    if (mode != 0 && mode != 1) return fail(ctx, ORT_EINVAL, "aim2d: mode = %d", mode);
    if (N == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N;
    double *d0, *d1, *d2, *d3; int32_t* di = nullptr;
    ENSURE(SL_IN0, n * 8, d0); ENSURE(SL_IN1, n * 8, d1); ENSURE(SL_IN2, n * 8, d2); ENSURE(SL_OUT0, n * 8, d3);
    if (iters) ENSURE(SL_OUT1, n * 4, di);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d0, x_start, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d1, other, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d2, target, n * 8, cudaMemcpyHostToDevice, st));
    AimArgs A; memset(&A, 0, sizeof A);
    A.N = N; A.stop = stop; A.vary_u = vary_u ? 1 : 0; A.mode = mode; A.aspheric = aspheric ? 1 : 0; A.tol = atol_or_scale;
    A.x0 = d0; A.other = d1; A.target = d2; A.x_out = d3; A.iters = di;
    CK(launch_aim2d(ctx->presc, A, st));
    ctx->launches++;
    CK(cudaMemcpyAsync(x_out, d3, n * 8, cudaMemcpyDeviceToHost, st));
    if (iters) CK(cudaMemcpyAsync(iters, di, n * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

// Per-row constants of the clip classifier of k_paraxial (kern_first_order.cu): with T = the high word of a read as a
// float, S = 1 / ulp(T) (a power of two) and M = T S (an integer below 2^24, exact), z = fma(|hf|, S, -M) counts high-word
// units between |y| and a.  +Inf / NaN apertures never clip (z = -4 for every ray); apertures too small for the
// 2^-21 a > 1e-13 argument, or whose constants leave the float range, send every ray to the exact test (z = 0).
static void paraxial_clip_constants(double a, float* cs, float* ncm)
{
    *cs = 0.0f; *ncm = 0.0f;
    if (isnan(a) || a == INFINITY) { *ncm = -4.0f; return; }
    if (!(a > 2.2e-7) || !isfinite(a)) return;
    int64_t bits; memcpy(&bits, &a, 8);
    const int32_t hi = (int32_t)(bits >> 32);
    float T; memcpy(&T, &hi, 4);
    const int ef = (hi >> 23) & 0xFF;
    if (ef < 1 || ef > 253) return;                          // T (and T + 2 units) must be a normal float
    const float ulp = nextafterf(T, INFINITY) - T;
    const float S = 1.0f / ulp, M = T * S;
    if (!isfinite(S) || !isfinite(M)) return;
    *cs = S; *ncm = -M;
}

static int lens_fill(ort_ctx* ctx, LensK& L, int k, const double* tau, const double* phi, const double* a, int clip)
{
    if (k < 0 || k > ORT_MAX_LENS) return fail(ctx, ORT_EINVAL, "paraxial_batch: k = %d not in [0, %d]", k, ORT_MAX_LENS);
    if (k > 0 && (!tau || !phi)) return fail(ctx, ORT_EINVAL, "paraxial_batch: NULL tau/phi");
    memset(&L, 0, sizeof L);
    L.k = k; L.clip = (clip && a) ? 1 : 0;
    L.tau_finite = 1; L.clip_nice = 1;
    float umax = 0.0f;
    for (int i = 0; i < k; i++) {
        L.tau[i] = tau[i]; L.phi[i] = phi[i]; L.a[i] = a ? a[i] : INFINITY;
        paraxial_clip_constants(L.a[i], &L.csm[i].x, &L.csm[i].y);
        if (!isfinite(tau[i])) L.tau_finite = 0;
        // the streaming kernel's classifier: T = high word of a as a float; rows that never clip get +Inf
        L.ctf[i] = INFINITY;
        if (isnan(L.a[i]) || L.a[i] == INFINITY) continue;
        if (L.csm[i].x == 0.0f) { L.clip_nice = 0; continue; }      // needs the exact test on every ray: general kernel
        int64_t bits; memcpy(&bits, &L.a[i], 8);
        const int32_t hi = (int32_t)(bits >> 32);
        float T; memcpy(&T, &hi, 4);
        L.ctf[i] = T;
        const float ulp = nextafterf(T, INFINITY) - T;
        if (ulp > umax) umax = ulp;
    }
    L.amb_thr = 1.5f * umax;
    return ORT_OK;
}

int ort_paraxial_batch_dev(ort_ctx* ctx, int k, const double* tau, const double* phi, const double* a, int clip,
                           int arith, int64_t N, const double* d_y0, const double* d_w0, double* d_y,
                           double* d_w, int32_t* d_clip_idx, double* d_y_all, double* d_w_all, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (N < 0 || !d_y0 || !d_w0) return fail(ctx, ORT_EINVAL, "paraxial_batch: bad input");
    if (arith != ORT_ARITH_STRICT && arith != ORT_ARITH_FAST) return fail(ctx, ORT_EINVAL, "paraxial_batch: arith = %d", arith);
    LensK L;
    int rc = lens_fill(ctx, L, k, tau, phi, a, clip);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    ParaxArgs A; memset(&A, 0, sizeof A);
    A.N = N; A.y0 = d_y0; A.w0 = d_w0; A.y = d_y; A.w = d_w; A.clip_idx = d_clip_idx;
    A.y_all = d_y_all; A.w_all = d_w_all;
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_paraxial(L, A, arith, (cudaStream_t)stream));
    }
    if (N > 0) ctx->launches++;
    return ORT_OK;
}

int ort_paraxial_batch(ort_ctx* ctx, int k, const double* tau, const double* phi, const double* a, int clip,
                       int arith, int64_t N, const double* y0, const double* w0, double* y, double* w,
                       int32_t* clip_idx, double* y_all, double* w_all)
{
    if (!ctx) return ORT_EINVAL;
    if (N < 0 || !y0 || !w0) return fail(ctx, ORT_EINVAL, "paraxial_batch: bad input");
    if (N == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N, kk = (size_t)k + 1;
    double *d0, *d1, *dy = nullptr, *dw = nullptr, *dya = nullptr, *dwa = nullptr;
    int32_t* dci = nullptr;
    ENSURE(SL_IN0, n * 8, d0); ENSURE(SL_IN1, n * 8, d1);
    if (y) ENSURE(SL_OUT0, n * 8, dy);
    if (w) ENSURE(SL_OUT1, n * 8, dw);
    if (clip_idx) ENSURE(SL_OUT2, n * 4, dci);
    if (y_all) ENSURE(SL_OUT3, kk * n * 8, dya);
    if (w_all) ENSURE(SL_OUT4, kk * n * 8, dwa);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d0, y0, n * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d1, w0, n * 8, cudaMemcpyHostToDevice, st));
    int rc = ort_paraxial_batch_dev(ctx, k, tau, phi, a, clip, arith, N, d0, d1, dy, dw, dci, dya, dwa, st);
    if (rc) return rc;
    if (y) CK(cudaMemcpyAsync(y, dy, n * 8, cudaMemcpyDeviceToHost, st));
    if (w) CK(cudaMemcpyAsync(w, dw, n * 8, cudaMemcpyDeviceToHost, st));
    if (clip_idx) CK(cudaMemcpyAsync(clip_idx, dci, n * 4, cudaMemcpyDeviceToHost, st));
    if (y_all) CK(cudaMemcpyAsync(y_all, dya, kk * n * 8, cudaMemcpyDeviceToHost, st));
    if (w_all) CK(cudaMemcpyAsync(w_all, dwa, kk * n * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

// extend(M, tau, taup) = [1 taup; 0 1] * M * [1 tau; 0 1]  (src/TransferMatrix.jl:8), evaluated on the
// host with Julia's generic 2x2 matmul order (C[i,j] = A[i,1]*B[1,j] + A[i,2]*B[2,j]); volatile keeps
// the host compiler from contracting.
static void mm2_host(const double* A, const double* B, double* C)
{
    volatile double p, q;
    double c[4];
    p = A[0] * B[0]; q = A[2] * B[1]; c[0] = p + q;
    p = A[1] * B[0]; q = A[3] * B[1]; c[1] = p + q;
    p = A[0] * B[2]; q = A[2] * B[3]; c[2] = p + q;
    p = A[1] * B[2]; q = A[3] * B[3]; c[3] = p + q;
    memcpy(C, c, sizeof c);
}

int ort_transfer_batch_dev(ort_ctx* ctx, const double M[4], double tau, double taup, int reverse, int64_t N,
                           const double* d_v_in, double* d_v_out, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (!M || N < 0 || !d_v_in || !d_v_out) return fail(ctx, ORT_EINVAL, "transfer_batch: bad input");
    if (((uintptr_t)d_v_in | (uintptr_t)d_v_out) & 15) return fail(ctx, ORT_EINVAL, "transfer_batch: device pointers must be 16-byte aligned");
    CK(cudaSetDevice(ctx->device));
    TransferArgs A; memset(&A, 0, sizeof A);
    const double Lm[4] = {1.0, 0.0, taup, 1.0}, Rm[4] = {1.0, 0.0, tau, 1.0};
    double T[4];
    mm2_host(Lm, M, T);
    mm2_host(T, Rm, A.E);
    A.N = N; A.reverse = reverse ? 1 : 0;
    A.v_in = (const double2*)d_v_in; A.v_out = (double2*)d_v_out;
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_transfer(A, (cudaStream_t)stream));
    }
    if (N > 0) ctx->launches++;
    return ORT_OK;
}

int ort_transfer_batch(ort_ctx* ctx, const double M[4], double tau, double taup, int reverse, int64_t N,
                       const double* v_in, double* v_out)
{
    if (!ctx) return ORT_EINVAL;
    if (!M || N < 0 || !v_in || !v_out) return fail(ctx, ORT_EINVAL, "transfer_batch: bad input");
    if (N == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)N;
    double *d0, *d1;
    ENSURE(SL_IN0, n * 16, d0); ENSURE(SL_OUT0, n * 16, d1);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d0, v_in, n * 16, cudaMemcpyHostToDevice, st));
    int rc = ort_transfer_batch_dev(ctx, M, tau, taup, reverse, N, d0, d1, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(v_out, d1, n * 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_trace3d_candidates_dev(ort_ctx* ctx, int rows, int64_t C, const double* d_RtnK, const ort_field* field,
                               const double* d_ys, int ny, const double* d_xs, int nx, int stop, double a_stop,
                               int arith, double* d_out, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS) return fail(ctx, ORT_EINVAL, "candidates: rows = %d", rows);
    if (C < 0 || C >= (1LL << 31) || !d_RtnK || !field || !d_ys || !d_xs || !d_out) return fail(ctx, ORT_EINVAL, "candidates: bad input");
    if (field->mode != 0) return fail(ctx, ORT_EUNSUPPORTED, "candidates: only collimated fields (mode 0)");
    if (stop < 1 || stop > rows - 1) return fail(ctx, ORT_EINVAL, "candidates: stop = %d", stop);
    if ((long long)ny * nx >= (1LL << 31) || ny < 0 || nx < 0) return fail(ctx, ORT_EINVAL, "candidates: bad grid");
    if (arith != ORT_ARITH_STRICT && arith != ORT_ARITH_FAST) return fail(ctx, ORT_EINVAL, "candidates: arith = %d", arith);
    CK(cudaSetDevice(ctx->device));
    CandArgs A; memset(&A, 0, sizeof A);
    A.rows = rows; A.C = C; A.RtnK = d_RtnK; A.ys = d_ys; A.xs = d_xs; A.ny = ny; A.nx = nx;
    A.stop = stop; A.a_stop = a_stop; A.a_stop2 = a_stop * a_stop;
    A.u = field->u; A.v = field->v; A.h_prime = field->h_prime; A.out = d_out;
    ScratchScope scratch(ctx, (cudaStream_t)stream);
    if (arith == ORT_ARITH_FAST && C > 0) ENSURE(SL_CLIST, sizeof(int) * (3 + 3 * (size_t)C), A.lists);
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_candidates(A, arith, (cudaStream_t)stream, ctx->sm_count));
    }
    if (C > 0) ctx->launches += A.lists ? 4 : 1;
    return ORT_OK;
}

int ort_trace3d_candidates(ort_ctx* ctx, int rows, int64_t C, const double* RtnK, const ort_field* field,
                           const double* ys, int ny, const double* xs, int nx, int stop, double a_stop,
                           int arith, double* out)
{
    if (!ctx) return ORT_EINVAL;
    if (C < 0 || !RtnK || !ys || !xs || !out || rows < 2 || ny < 0 || nx < 0) return fail(ctx, ORT_EINVAL, "candidates: bad input");
    if (C == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t nb = (size_t)C * 4 * (size_t)rows * 8;
    double *d_p, *d_ys, *d_xs, *d_o;
    ENSURE(SL_IN0, nb, d_p); ENSURE(SL_YS, (size_t)ny * 8, d_ys); ENSURE(SL_XS, (size_t)nx * 8, d_xs);
    ENSURE(SL_OUT0, (size_t)C * 32, d_o);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d_p, RtnK, nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_ys, ys, (size_t)ny * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_xs, xs, (size_t)nx * 8, cudaMemcpyHostToDevice, st));
    int rc = ort_trace3d_candidates_dev(ctx, rows, C, d_p, field, d_ys, ny, d_xs, nx, stop, a_stop, arith, d_o, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_o, (size_t)C * 32, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_vignetting_candidates_dev(ort_ctx* ctx, int rows, int64_t C, const double* d_RtnK, const double* a_solve,
                                  const double* a_vig, double h_prime, double* d_out, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS) return fail(ctx, ORT_EINVAL, "vignetting: rows = %d", rows);
    if (C < 0 || C >= (1LL << 31) || !d_RtnK || !a_solve || !d_out) return fail(ctx, ORT_EINVAL, "vignetting: bad input");
    CK(cudaSetDevice(ctx->device));
    VigArgs A; memset(&A, 0, sizeof A);
    A.rows = rows; A.C = C; A.RtnK = d_RtnK; A.h_prime = h_prime; A.out = d_out;
    for (int i = 0; i + 1 < rows; i++) { A.a_solve[i] = a_solve[i]; A.a_vig[i] = a_vig ? a_vig[i] : a_solve[i]; }
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_vignetting(A, (cudaStream_t)stream));
    }
    if (C > 0) ctx->launches++;
    return ORT_OK;
}

int ort_vignetting_candidates(ort_ctx* ctx, int rows, int64_t C, const double* RtnK, const double* a_solve,
                              const double* a_vig, double h_prime, double* out)
{
    if (!ctx) return ORT_EINVAL;
    if (C < 0 || !RtnK || !a_solve || !out || rows < 2) return fail(ctx, ORT_EINVAL, "vignetting: bad input");
    if (C == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t nb = (size_t)C * 4 * (size_t)rows * 8, no = (size_t)C * (6 * (size_t)(rows - 1) + ORT_VIG_TAIL) * 8;
    double *d_p, *d_o;
    ENSURE(SL_IN0, nb, d_p); ENSURE(SL_OUT0, no, d_o);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d_p, RtnK, nb, cudaMemcpyHostToDevice, st));
    int rc = ort_vignetting_candidates_dev(ctx, rows, C, d_p, a_solve, a_vig, h_prime, d_o, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_o, no, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_aim_candidates_dev(ort_ctx* ctx, int rows, int64_t C, const double* d_RtnK, const double* a, double h_prime,
                           double H, int aspheric, double* d_out, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS - 1) return fail(ctx, ORT_EINVAL, "aim_candidates: rows = %d", rows);
    if (C < 0 || C >= (1LL << 31) || !d_RtnK || !a || !d_out) return fail(ctx, ORT_EINVAL, "aim_candidates: bad input");
    if (!(fabs(H) <= 1.0)) return fail(ctx, ORT_EINVAL, "aim_candidates: DomainError |H| <= 1");    // src/PupilSampling.jl:88-89
    CK(cudaSetDevice(ctx->device));
    AimCandArgs A; memset(&A, 0, sizeof A);
    A.rows = rows; A.C = C; A.RtnK = d_RtnK; A.h_prime = h_prime; A.H = H; A.aspheric = aspheric; A.out = d_out;
    for (int i = 0; i + 1 < rows; i++) A.a[i] = a[i];
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_aim_candidates(A, (cudaStream_t)stream));
        CK(launch_aim_edges(rows, C, d_RtnK, d_out, 0, (cudaStream_t)stream));
    }
    if (C > 0) ctx->launches += 2;
    return ORT_OK;
}

int ort_aim_candidates(ort_ctx* ctx, int rows, int64_t C, const double* RtnK, const double* a, double h_prime,
                       double H, int aspheric, double* out)
{
    if (!ctx) return ORT_EINVAL;
    if (C < 0 || !RtnK || !a || !out || rows < 2) return fail(ctx, ORT_EINVAL, "aim_candidates: bad input");
    if (C == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t nb = (size_t)C * 4 * (size_t)rows * 8, no = (size_t)C * ORT_AIM_NOUT * 8;
    double *d_p, *d_o;
    ENSURE(SL_IN0, nb, d_p); ENSURE(SL_OUT1, no, d_o);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d_p, RtnK, nb, cudaMemcpyHostToDevice, st));
    int rc = ort_aim_candidates_dev(ctx, rows, C, d_p, a, h_prime, H, aspheric, d_o, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_o, no, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_aim_fields(ort_ctx* ctx, int rows, const double* R, const double* t, const double* n, const double* K,
                   const double* a, double h_prime, const double* Hs, int n_fields, int aspheric, double* out)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS - 1) return fail(ctx, ORT_EINVAL, "aim_fields: rows = %d", rows);
    if (!R || !t || !n || !a || !Hs || !out) return fail(ctx, ORT_EINVAL, "aim_fields: bad input");
    if (n_fields < 1 || n_fields > ORT_MAX_FIELDS) return fail(ctx, ORT_EINVAL, "aim_fields: n_fields = %d not in [1, %d]", n_fields, ORT_MAX_FIELDS);
    for (int f = 0; f < n_fields; f++)
        if (!(fabs(Hs[f]) <= 1.0)) return fail(ctx, ORT_EINVAL, "aim_fields: DomainError |H| <= 1");       // src/PupilSampling.jl:88-89
    CK(cudaSetDevice(ctx->device));
    const size_t nb = (size_t)4 * rows * 8, no = (size_t)n_fields * ORT_AIM_NOUT * 8;
    double *d_p, *d_o;
    ENSURE(SL_IN0, nb, d_p); ENSURE(SL_OUT1, no, d_o);
    double h_p[4 * ORT_MAX_ROWS];
    for (int i = 0; i < rows; i++) { h_p[i] = R[i]; h_p[rows + i] = t[i]; h_p[2 * rows + i] = n[i]; h_p[3 * rows + i] = K ? K[i] : 0.0; }
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d_p, h_p, nb, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));                  // h_p is a stack buffer
    AimCandArgs A; memset(&A, 0, sizeof A);
    A.rows = rows; A.C = n_fields; A.RtnK = d_p; A.h_prime = h_prime; A.aspheric = aspheric; A.out = d_o;
    A.n_fields = n_fields;
    for (int f = 0; f < n_fields; f++) A.Hs[f] = Hs[f];
    for (int i = 0; i + 1 < rows; i++) A.a[i] = a[i];
    CK(launch_aim_candidates(A, st));
    CK(launch_aim_edges(rows, n_fields, d_p, d_o, 1, st));
    ctx->launches += 2;
    CK(cudaMemcpyAsync(out, d_o, no, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_trace3d_candidates_aimed_dev(ort_ctx* ctx, int rows, int64_t C, const double* d_RtnK, const double* d_aim,
                                     int ny, int nx, int arith, double* d_out, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS - 1) return fail(ctx, ORT_EINVAL, "candidates_aimed: rows = %d", rows);
    if (C < 0 || C >= (1LL << 31) || !d_RtnK || !d_aim || !d_out) return fail(ctx, ORT_EINVAL, "candidates_aimed: bad input");
    if ((long long)ny * nx >= (1LL << 31) || ny < 2 || nx < 2) return fail(ctx, ORT_EINVAL, "candidates_aimed: bad grid");
    if (arith != ORT_ARITH_STRICT && arith != ORT_ARITH_FAST) return fail(ctx, ORT_EINVAL, "candidates_aimed: arith = %d", arith);
    CK(cudaSetDevice(ctx->device));
    CandArgs A; memset(&A, 0, sizeof A);
    A.rows = rows; A.C = C; A.RtnK = d_RtnK; A.aim = d_aim; A.ny = ny; A.nx = nx; A.stop = 1;
    A.v = 0.0;                                       // V = 0 (meridional field, src/PupilSampling.jl:98)
    A.out = d_out;
    ScratchScope scratch(ctx, (cudaStream_t)stream);
    if (arith == ORT_ARITH_FAST && C > 0) ENSURE(SL_CLIST, sizeof(int) * (3 + 3 * (size_t)C), A.lists);
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_candidates(A, arith, (cudaStream_t)stream, ctx->sm_count));
    }
    if (C > 0) ctx->launches += A.lists ? 4 : 1;
    return ORT_OK;
}

int ort_trace3d_candidates_aimed(ort_ctx* ctx, int rows, int64_t C, const double* RtnK, const double* aim, int ny,
                                 int nx, int arith, double* out)
{
    if (!ctx) return ORT_EINVAL;
    if (C < 0 || !RtnK || !aim || !out || rows < 2) return fail(ctx, ORT_EINVAL, "candidates_aimed: bad input");
    if (C == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t nb = (size_t)C * 4 * (size_t)rows * 8, na = (size_t)C * ORT_AIM_NOUT * 8;
    double *d_p, *d_a, *d_o;
    ENSURE(SL_IN0, nb, d_p); ENSURE(SL_OUT1, na, d_a); ENSURE(SL_OUT0, (size_t)C * 32, d_o);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d_p, RtnK, nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_a, aim, na, cudaMemcpyHostToDevice, st));
    int rc = ort_trace3d_candidates_aimed_dev(ctx, rows, C, d_p, d_a, ny, nx, arith, d_o, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_o, (size_t)C * 32, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_seidel_candidates_dev(ort_ctx* ctx, int rows, int64_t C, const double* d_RtnK, const double* a, double h_prime,
                              double lambda, const double* dn, double* d_out, double* d_per_surface, void* stream)
{
    if (!ctx) return ORT_EINVAL;
    if (rows < 2 || rows > ORT_MAX_ROWS) return fail(ctx, ORT_EINVAL, "seidel: rows = %d", rows);
    if (C < 0 || C >= (1LL << 31) || !d_RtnK || !a || !d_out) return fail(ctx, ORT_EINVAL, "seidel: bad input");
    if (!(lambda > 0.0)) return fail(ctx, ORT_EINVAL, "seidel: lambda must be positive");
    CK(cudaSetDevice(ctx->device));
    SeidelArgs A; memset(&A, 0, sizeof A);
    A.rows = rows; A.C = C; A.RtnK = d_RtnK; A.h_prime = h_prime; A.lambda = lambda; A.out = d_out; A.per = d_per_surface;
    for (int i = 0; i + 1 < rows; i++) A.a[i] = a[i];
    for (int i = 0; i < rows; i++) A.dn[i] = dn ? dn[i] : 0.0;
    {
        ProfScope prof(ctx, (cudaStream_t)stream);
        CK(launch_seidel(A, (cudaStream_t)stream));
    }
    if (C > 0) ctx->launches++;
    return ORT_OK;
}

int ort_seidel_candidates(ort_ctx* ctx, int rows, int64_t C, const double* RtnK, const double* a, double h_prime,
                          double lambda, const double* dn, double* out, double* per_surface)
{
    if (!ctx) return ORT_EINVAL;
    if (C < 0 || !RtnK || !a || !out || rows < 2) return fail(ctx, ORT_EINVAL, "seidel: bad input");
    if (C == 0) return ORT_OK;
    CK(cudaSetDevice(ctx->device));
    const size_t nb = (size_t)C * 4 * (size_t)rows * 8, no = (size_t)C * ORT_SEIDEL_NOUT * 8;
    const size_t np_ = (size_t)C * 7 * (size_t)(rows - 1) * 8;
    double *d_p, *d_o, *d_per = nullptr;
    ENSURE(SL_IN0, nb, d_p); ENSURE(SL_OUT0, no, d_o);
    if (per_surface) ENSURE(SL_OUT1, np_, d_per);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    CK(cudaMemcpyAsync(d_p, RtnK, nb, cudaMemcpyHostToDevice, st));
    int rc = ort_seidel_candidates_dev(ctx, rows, C, d_p, a, h_prime, lambda, dn, d_o, d_per, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_o, no, cudaMemcpyDeviceToHost, st));
    if (per_surface) CK(cudaMemcpyAsync(per_surface, d_per, np_, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

// Chan merge of per-shard statistics records in the given (rank) order: the combine step after the
// all-gather of a row-sharded sweep.  Pure host arithmetic; recs is [n_shards][n_fields].
int ort_merge_stats(const ort_stats* recs, int n_shards, int n_fields, ort_stats* out)
{
    if (!recs || !out || n_shards < 1 || n_fields < 1) return ORT_EINVAL;
    for (int f = 0; f < n_fields; f++) {
        ort_stats a; memset(&a, 0, sizeof a);
        a.r_max = -INFINITY;
        for (int r = 0; r < n_shards; r++) {
            const ort_stats& b = recs[(size_t)r * n_fields + f];
            a.n_miss += b.n_miss; a.n_tir += b.n_tir; a.n_domain += b.n_domain; a.n_clip += b.n_clip; a.n_vig += b.n_vig; a.n_strict += b.n_strict;
            if (b.n_kept == 0) continue;
            if (a.n_kept == 0) {
                a.n_kept = b.n_kept; a.mean_x = b.mean_x; a.mean_y = b.mean_y; a.m2_x = b.m2_x; a.m2_y = b.m2_y;
                a.r_max = b.r_max; a.mean_opd = b.mean_opd; a.m2_opd = b.m2_opd;
                continue;
            }
            const double na = (double)a.n_kept, nb = (double)b.n_kept, n = na + nb, w = nb / n;
            const double dx = b.mean_x - a.mean_x, dy = b.mean_y - a.mean_y, dd = b.mean_opd - a.mean_opd;
            a.mean_x = a.mean_x + dx * w; a.m2_x = a.m2_x + b.m2_x + dx * dx * (na * w);
            a.mean_y = a.mean_y + dy * w; a.m2_y = a.m2_y + b.m2_y + dy * dy * (na * w);
            a.mean_opd = a.mean_opd + dd * w; a.m2_opd = a.m2_opd + b.m2_opd + dd * dd * (na * w);
            a.n_kept += b.n_kept;
            if (b.r_max > a.r_max) a.r_max = b.r_max;
        }
        out[f] = a;
    }
    return ORT_OK;
}

// sigma of the mirrored spot (src/PupilSampling.jl:140-141, 169-173) from one statistics record:
// x -> [x; -x] has mean 0 and sum of squares 2 (M2x + n mean_x^2); y -> [y; y] doubles M2y.
double ort_rms_from_stats(const ort_stats* s)
{
    if (!s || s->n_kept <= 0) return NAN;
    const double n = (double)s->n_kept;
    const double sxx = s->m2_x + n * s->mean_x * s->mean_x;
    return sqrt((2.0 * sxx + 2.0 * s->m2_y) / (2.0 * n));
}

int ort_selftest_exact_ops(ort_ctx* ctx, long long n, unsigned long long seed, long long* out8)
{
    if (!ctx || !out8 || n < 0) return ORT_EINVAL;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    unsigned long long* d; ENSURE(SL_OUT0, 8 * sizeof(unsigned long long), d);
    CK(cudaMemsetAsync(d, 0, 8 * sizeof(unsigned long long), st));
    CK(launch_selftest_exact(n, seed, d, ctx->sm_count, st));
    ctx->launches++;
    CK(cudaMemcpyAsync(out8, d, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return ORT_OK;
}

int ort_fp64_peak(ort_ctx* ctx, double* tflops, double* ms)
{
    if (!ctx || !tflops) return ORT_EINVAL;
    CK(cudaSetDevice(ctx->device));
    double* sink; ENSURE(SL_SINK, 8, sink);
    cudaStream_t st = ctx->stream;
    ScratchScope scratch(ctx, st);
    long long dfma = 0;
    CK(launch_fp64_peak(sink, ctx->sm_count, 256, st, &dfma));           // warm-up
    double best = 1e30;
    for (int rep = 0; rep < 3; rep++) {
        CK(cudaEventRecord(ctx->ev_a, st));
        CK(launch_fp64_peak(sink, ctx->sm_count, 4096, st, &dfma));
        CK(cudaEventRecord(ctx->ev_b, st));
        CK(cudaEventSynchronize(ctx->ev_b));
        float t = 0.f;
        CK(cudaEventElapsedTime(&t, ctx->ev_a, ctx->ev_b));
        if (t < best) best = t;
    }
    ctx->launches += 4;
    *tflops = 2.0 * (double)dfma / (best * 1e-3) / 1e12;
    if (ms) *ms = best;
    return ORT_OK;
}

}  // extern "C"
