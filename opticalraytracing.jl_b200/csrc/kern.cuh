// kern.cuh -- kernel argument blocks and launch wrappers shared between the kernel TUs and ort_api.cu
#pragma once
#include "ort_internal.cuh"

// shifted raw moments of one CTA / field (all CTAs of a field share the shift (cx, cy))
struct RawPart {
    long long n;
    double s1x, s2x, s1y, s2y, rmax, cx, cy;
    double s1o, s2o, co;                    // EXTENSION: OPD moments about the shift co
    int nmiss, ntir, ndom, nclip, nvig, nstrict;
};

struct GridArgs {
    const double* ys; const double* xs;     // device: grid coordinates (:121-122)
    int ny, nx;
    int ys_stride;                          // 0: ys shared by all fields; ny: one ys row per field
    unsigned NN;                            // ny * nx  (< 2^31)
    int stop;                               // 1-based system.stop
    double a_stop, a_stop2;
    double wg_nu, wg_lambda;
    double *ex, *ey, *r, *theta, *wx, *wy;  // device outputs, [n_fields][NN]; NULL = not wanted
    double *opd;                            // EXTENSION
    int ext;                                // ORT_EXT_* bits
    double opd_scale;
    uint8_t *mask, *flags;
    RawPart* partials;                      // [n_fields][gridDim.x]
    int* tile_counts;                       // [n_fields][ntiles] or NULL (no compaction requested)
    ort_field fields[ORT_MAX_FIELDS];
};

struct FocusArgs {                          // through-focus sweep (k_focus)
    GridArgs G;                             // grid, stop, per-field outputs r / theta / mask / flags, tile counts; G.ex, G.ey
                                            // are [n_fields][n_foci][NN]; G.partials is [n_fields * n_foci][gridDim.x]
    int n_foci;
    double t_lo, t_hi;                      // smallest and largest focus
    double foci[ORT_MAX_FOCI];
};

struct CompactArgs {
    unsigned NN;
    const uint8_t* mask;
    const int* tile_offsets;
    const double* src[7];
    double* dst[7];
};

struct RaysArgs {
    long long N;
    const double *y0, *x0, *u0, *v0;
    double *xv, *yv, *kout;
    uint8_t* flags;
    double* opl;                            // EXTENSION: OPL to the last surface (NULL = not wanted)
};

struct CandArgs {
    int rows; long long C;
    const double* RtnK;
    const double *ys, *xs; int ny, nx;
    int stop; double a_stop, a_stop2, u, v, h_prime;
    const double* aim;                      // NULL, or [C][ORT_AIM_NOUT]: per-candidate grid, stop, field, focus
    double* out;
    int* lists;                             // FAST: device scratch of 3 + 3 C ints for k_cand_classify (NULL: one CTA per candidate, general kernel)
};

struct SeidelArgs {
    int rows; long long C;
    const double* RtnK;
    double h_prime, lambda;
    double a[ORT_MAX_ROWS], dn[ORT_MAX_ROWS];
    double* out; double* per;
};

struct VigArgs {
    int rows; long long C;
    const double* RtnK;
    double a_solve[ORT_MAX_ROWS], a_vig[ORT_MAX_ROWS];
    double h_prime;
    double* out;                            // [C][6 * (rows - 1) + ORT_VIG_TAIL]
};

struct AimCandArgs {
    int rows; long long C;
    const double* RtnK;
    double a[ORT_MAX_ROWS];
    double h_prime, H;
    int aspheric;
    int n_fields;                           // > 0: ONE prescription (RtnK[0]) at n_fields relative fields Hs[] (C == n_fields)
    double Hs[ORT_MAX_FIELDS];
    double* out;                            // [C][ORT_AIM_NOUT]
};

struct LensK {                              // paraxial Lens rows in the constant bank
    int k; int clip;
    double tau[ORT_MAX_LENS], phi[ORT_MAX_LENS], a[ORT_MAX_LENS];
    float2 csm[ORT_MAX_LENS];               // clip classifier of k_paraxial: z = fma(|float(hi word of y)|, csm.x, csm.y)
    float ctf[ORT_MAX_LENS];                // clip classifier of k_paraxial_final: z = |float(hi word of y)| - ctf  (+Inf: the row never clips)
    float amb_thr;                          // 1.5 x the largest ulp(ctf[row]): below it a decision was within two high-word units
    int tau_finite;                         // every tau finite (Lens(surfaces) guarantees it, src/RayTracing.jl:42)
    int clip_nice;                          // every aperture is +Inf / NaN (never clips) or > 2.2e-7 with a normal float pattern
};


struct ParaxArgs {
    long long N;
    const double *y0, *w0;
    double *y, *w; int32_t* clip_idx;
    double *y_all, *w_all;
};

struct Trace2dArgs {
    long long N; int aspheric;
    const double *y0, *U0;
    double *y_out, *U_out, *ts_out;
    uint8_t* flags;
};

struct AimArgs {
    long long N; int stop, vary_u, mode, aspheric;
    double tol;
    const double *x0, *other, *target;
    double* x_out; int32_t* iters;
};

struct TransferArgs {
    long long N; int reverse;
    double E[4];                            // extend(M, tau, taup), column-major
    const double2* v_in; double2* v_out;
};

#ifndef ORT_FAST_RPT
#define ORT_FAST_RPT 2                      // rays per thread of k_grid<FAST>
#endif
#ifndef ORT_BPS1
#define ORT_BPS1 4                          // min resident CTAs/SM requested for k_grid<FAST,1>
#endif
#ifndef ORT_BPS2
#define ORT_BPS2 3                          // ... for k_grid<FAST,2>
#endif
#ifndef ORT_BPSS
#define ORT_BPSS 4                          // ... for k_grid<STRICT,1>: 64 registers, 132 B of spills.  With xdiv / xsqrt 12.44 ms per bench step
                                            // against 12.83 at 3 (78 registers, no spills); before them 3 was the optimum (13.4)
#endif
#ifndef ORT_STRICT_XF
#define ORT_STRICT_XF true                 // k_grid<STRICT>: IEEE / and sqrt with the slow path deferred (xdiv, xsqrt)
#endif
#ifndef ORT_BPS_POLY
#define ORT_BPS_POLY 3                      // ... for the k_grid<FAST,2> instantiations with the polynomial body (2 CTAs x 128 registers: the same time)
#endif
#ifndef ORT_BPS2E
#define ORT_BPS2E 3                         // ... for k_grid<FAST,2,EXT> (80 registers, ~190 B of spills: 5-7 % faster than 2 CTAs x 126 registers)
#endif
#ifndef ORT_SIMPLE_RPT
#define ORT_SIMPLE_RPT 3                    // rays per thread of k_grid<FAST, .., SIMPLE> (3 x 2 CTAs/SM: 2.53 ms vs 2.60 at 2 x 3)
#endif
#ifndef ORT_BPSP
#define ORT_BPSP 2                          // ... and its resident CTAs/SM (128 registers, no spills)
#endif
#ifndef ORT_SC_RPT
#define ORT_SC_RPT 2                        // rays per thread of the SIMPLE-conic instantiations (Presc::simple == 2)
#endif
#ifndef ORT_BPSC
#define ORT_BPSC 3                          // ... and their resident CTAs/SM
#endif
#ifndef ORT_STRICT_RPT
#define ORT_STRICT_RPT 1                    // rays per thread of k_grid<STRICT>.  With the library intrinsics: 13.4 ms per bench step at
#endif                                      // 1 x 3 CTAs/SM, 2 x 3 (spills) 13.5, 2 x 2 15.3, 3 x 2 15.5; with xdiv / xsqrt: 1 x 4 12.44, 1 x 3 12.83,
                                            // 2 x 3 13.3, 2 x 2 14.5 (ncu: FP64 pipe 62 % busy, stall reason `wait` 3.4 per issue -- the
                                            // serial chain of correctly rounded / and sqrt, which more rays per thread do not shorten)
#ifndef ORT_SE_RPT
#define ORT_SE_RPT 2                        // rays per thread of the SIMPLE x EXT instantiations (OPD sweeps over simple prescriptions)
#endif
#ifndef ORT_BPSE
#define ORT_BPSE 3                          // ... and their resident CTAs/SM (80 registers, ~190 B of spills: 0.530 ms per 16.8 M-ray OPD field
#endif                                      //     against 0.541 at 2 x 127 registers and 0.595 at 3 rays per thread)
#ifndef ORT_GRID_WAVES_DEFAULT
#define ORT_GRID_WAVES_DEFAULT 8            // CTA waves per grid sweep (grid_dims in ort_api.cu)
#endif
int grid_variant(const Presc& P, int arith, int ext);
int grid_rays_per_thread(int arith, int variant);
int grid_blocks_per_sm(int arith, int variant);
cudaError_t launch_grid(const Presc& P, const GridArgs& A, int arith, dim3 grid, cudaStream_t st, const PolyK* Q = nullptr);
cudaError_t launch_grid_finalize(const RawPart* partials, int nparts, int n_fields, ort_stats* stats,
                                 cudaStream_t st);
// ints per field of the tile-count buffer of launch_compact / launch_compact_focus: the counts and the chunk totals
size_t compact_tile_ints(unsigned NN);
cudaError_t launch_compact(int* tile_counts, const CompactArgs& C, int n_fields, cudaStream_t st);
int focus_blocks_per_sm(int arith, int variant);
cudaError_t launch_focus(const Presc& P, const FocusArgs& F, int arith, dim3 grid, cudaStream_t st);
cudaError_t launch_compact_focus(int* tile_counts, const CompactArgs& C, int n_fields, int n_foci, cudaStream_t st);
cudaError_t launch_rays(const Presc& P, const RaysArgs& A, int arith, cudaStream_t st);
cudaError_t launch_candidates(const CandArgs& A, int arith, cudaStream_t st, int sm_count);
cudaError_t launch_trace2d(const Presc& P, const Trace2dArgs& A, cudaStream_t st);
cudaError_t launch_paraxial(const LensK& L, const ParaxArgs& A, int arith, cudaStream_t st);
cudaError_t launch_transfer(const TransferArgs& A, cudaStream_t st);
cudaError_t launch_seidel(const SeidelArgs& A, cudaStream_t st);
cudaError_t launch_aim_candidates(const AimCandArgs& A, cudaStream_t st);
cudaError_t launch_vignetting(const VigArgs& A, cudaStream_t st);
cudaError_t launch_aim_edges(int rows, long long C, const double* RtnK, double* aim, int shared_prescription, cudaStream_t st);
cudaError_t launch_aim2d(const Presc& P, const AimArgs& A, cudaStream_t st);
cudaError_t launch_selftest_exact(long long n, unsigned long long seed, unsigned long long* d_out, int sm_count, cudaStream_t st);
cudaError_t launch_fp64_peak(double* d_sink, int sm_count, long long iters, cudaStream_t st,
                             long long* dfma_per_launch);
