// ort_ctx.cuh -- the context object behind the C ABI and the helpers shared by ort_api.cu (single-GPU entry points)
// and ort_comm.cu (communicator, sharded sweeps).  Private to the library.
#pragma once
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "kern.cuh"

enum Slot {
    SL_YS, SL_XS, SL_PARTIALS, SL_TILES, SL_STATS,
    SL_EX, SL_EY, SL_R, SL_TH, SL_WX, SL_WY, SL_OPD, SL_MASK, SL_FLAGS,     // trace outputs (full grid)
    SL_CEX, SL_CEY, SL_CR, SL_CTH, SL_CWX, SL_CWY, SL_COPD,                 // compacted outputs
    SL_IN0, SL_IN1, SL_IN2, SL_IN3, SL_OUT0, SL_OUT1, SL_OUT2, SL_OUT3, SL_OUT4, SL_SINK, SL_POLY,
    SL_GATHER, SL_MERGED, SL_AIM, SL_TABLE, SL_CLIST,                                  // communicator: gathered records, merged records, prelude records, merit table
    SL_COUNT
};

struct ort_ctx {
    int device;
    int sm_count, cc_major, cc_minor;
    char name[128];
    cudaStream_t stream;        // compute stream of the host-pointer entry points
    cudaStream_t copy_stream;   // D2H stream (overlaps the next field's trace)
    cudaEvent_t ev_a, ev_b;
    cudaEvent_t ev_field[ORT_MAX_FIELDS];
    Presc presc;
    PolyK polyk;                // polynomial terms of <= ORT_POLYK_N coefficients, as k_grid's third parameter
    bool have_polyk;
    int rows;
    bool have_layout;
    int fast_ok_layout;         // fast_ok as derived from R, t, n, K alone (polynomial terms force it to 0 while set)
    int bps[2][5];              // resident CTAs/SM of k_grid<STRICT|FAST, variant general|EXT|SIMPLE|SIMPLE x EXT|SIMPLE-conic> (grid_variant)
    int bps_focus[2][5];        // the same for k_focus (variants 0, 2, 4; 1 and 3 unused)
    void* slot[SL_COUNT];
    size_t slot_bytes[SL_COUNT];
    // The scratch slots are shared by every entry point of the context.  Work that uses them is ordered across streams
    // by one event: an entry point that enqueues on a stream other than the last one used first waits for ev_scratch.
    cudaEvent_t ev_scratch;
    cudaStream_t scratch_stream;
    bool scratch_busy;
    cudaStream_t scratch_now;   // stream of the entry point that is running (ScratchScope; NULL is the default stream), for
                                // ORT_POISON_SCRATCH; ctx->stream until the first one
    long long launches;
    int prof_on;
    long long prof_n;               // event pairs recorded since the last read
    cudaEvent_t prof_ev[64][2];
    // communicator (ort_comm.cu): NCCL, resolved with dlopen on first use
    void* comm;                     // ncclComm_t
    int comm_rank, comm_world;
    char err[512];
};

int ort_fail(ort_ctx* c, int code, const char* fmt, ...);
int ort_ensure(ort_ctx* ctx, int id, size_t bytes, void** out);
int ort_resolve_arith(const ort_ctx* ctx, int arith);

#define fail ort_fail
#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(ctx, ORT_ECUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,          \
                        cudaGetErrorString(e_));                                              \
    } while (0)
#define ENSURE(id, bytes, ptr)                                                         \
    do { void* p_; int rc_ = ort_ensure(ctx, (id), (bytes), &p_); if (rc_) return rc_; \
         (ptr) = (decltype(ptr))p_; } while (0)

// Orders the use of the context's scratch slots across streams (see ort_ctx::ev_scratch).  Constructed at the top of
// every entry point that touches a slot on stream `st`; the destructor records the event behind the enqueued work.
struct ScratchScope {
    ort_ctx* c; cudaStream_t st;
    ScratchScope(ort_ctx* c_, cudaStream_t st_) : c(c_), st(st_)
    {
        if (c->scratch_busy && c->scratch_stream != st) cudaStreamWaitEvent(st, c->ev_scratch, 0);
        c->scratch_now = st;
    }
    ~ScratchScope()
    {
        cudaEventRecord(c->ev_scratch, st);
        c->scratch_stream = st; c->scratch_busy = true;
    }
};

// bracket the dominant kernel with an event pair (measurement only)
struct ProfScope {
    ort_ctx* c; cudaStream_t st; int slot;
    ProfScope(ort_ctx* c_, cudaStream_t st_) : c(c_), st(st_), slot(-1)
    {
        if (c->prof_on) { slot = (int)(c->prof_n % 64); cudaEventRecord(c->prof_ev[slot][0], st); }
    }
    ~ProfScope()
    {
        if (slot >= 0) { cudaEventRecord(c->prof_ev[slot][1], st); c->prof_n++; }
    }
};

// shared between ort_api.cu and ort_comm.cu
int ort_grid_check(ort_ctx* ctx, const ort_field* fields, int n_fields, const void* ys, int ny, const void* xs, int nx,
                   int stop, const ort_opts* opts, const ort_grid_out* out);
int ort_grid_waves();
int ort_grid_dims(const ort_ctx* ctx, const int (&bps)[2][5], int waves, const ort_opts* opts, int n_fields, unsigned NN);
int ort_grid_enqueue(ort_ctx* ctx, const ort_field* fields, int n_fields, const double* d_ys, int ny, const double* d_xs,
                     int nx, int stop, double a_stop, const double* foci, int n_foci, const ort_opts* opts,
                     const ort_grid_out& full, const ort_grid_out* dst, ort_stats* d_stats, RawPart* d_partials, int* d_tiles,
                     int gx, cudaStream_t st);
int ort_sweep_scratch(ort_ctx* ctx, const ort_grid_out* out, const ort_opts* opts, bool dev, unsigned NN, int n_fields,
                      int n_foci, ort_grid_out* full, ort_grid_out* comp, int** d_tiles);
int ort_copy_out(ort_ctx* ctx, const ort_grid_out* out, const ort_grid_out& src, bool rays, size_t dst_o, size_t src_o,
                 size_t n, int n_foci, unsigned NN, cudaStream_t st);
// all-gather of the per-field records of this rank + rank-order merge, enqueued on st (ort_comm.cu).  d_local: [n_fields]
// on the device; d_merged: [n_fields] (may alias nothing else); d_ranks: optional [world][n_fields] receive buffer.
int ort_comm_gather_stats(ort_ctx* ctx, const ort_stats* d_local, int n_fields, ort_stats* d_merged, ort_stats* d_ranks,
                          cudaStream_t st);
