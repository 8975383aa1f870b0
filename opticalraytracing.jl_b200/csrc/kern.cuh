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

// Encircled energy (kern_energy.cu): per-set selection state in device scratch, written by k_energy_init and
// k_energy_select, read by the pass kernels
struct EnergyState {
    unsigned long long prefix[ORT_MAX_FRACS];   // key bits selected so far, per fraction
    unsigned long long rank[ORT_MAX_FRACS];     // 0-based rank of the wanted key among the keys with that prefix
    long long n;                                // kept rays
    unsigned src_n;                             // keys in candidate list `src`
    unsigned cnt;                               // keys appended to candidate list `dst` by the running pass
    int src, dst;                               // candidate list the next pass reads / writes: -1 = the sweep outputs / none
    int active;                                 // bit f: fraction f is selecting (n > 0)
    int pad;
};

struct EnergyArgs {
    int n_sets, sets_per_mask;
    long long stride;
    const double *ex, *ey; const uint8_t* mask; const ort_stats* stats;
    int metric, center, n_radii, n_fracs;
    EnergyState* state;                         // [n_sets]
    unsigned* hist;                             // [n_sets][energy_hist_words(n_fracs)]
    unsigned long long* bins;                   // [n_sets][n_radii + 1]
    unsigned long long* cand[2];                // [n_sets][cap] each
    unsigned cap;                               // candidate-list capacity per set
    long long* counts;                          // [n_sets][n_radii]
    double* radius;                             // [n_sets][n_fracs]
    double fracs[ORT_MAX_FRACS];
};

// Zernike fit of the wavefront (kern_zernike.cu)
struct ZernArgs {
    int n_sets, n_max;
    long long stride;
    const double *opd, *r, *theta; const uint8_t* mask; const ort_stats* stats;
    double r_norm;                              // 0: stats[s].r_max
    int js, jp, nblk, R;                        // fitted terms, Gram row (js + 1 padded to 4), 4 x 4 Gram blocks, ray groups
    int gx, gx_resid;                           // CTAs per set of k_zern_gram and of k_zern_resid
    double* gpart;                              // [n_sets][gx][zern_gram_record]: per-CTA Gram blocks, non-finite flag
    double* rpart;                              // [n_sets][gx_resid][3]: per-CTA sum of squares, min, max of the residual
    double* csym;                               // [n_sets][49]: the fitted coefficients in column order
    double* coef;                               // [n_sets][(n_max + 1)(n_max + 2) / 2]
    double* resid;                              // [n_sets][2]
    int* status;                                // [n_sets]
};

// Diffraction PSF of the wavefront (kern_psf.cu)
struct PsfArgs {
    int n_sets, ny, nx;
    long long stride;
    const double* opd; const uint8_t* mask; const ort_stats* stats;
    const double *ys, *xs;                      // ys + s * ys_stride: the iy coordinates of set s
    long long ys_stride;                        // 0 or ny
    int n_u, n_v;
    double du, dv, scale;
    int nuh, nup;                               // computed columns (xi >= 0) = ceil(n_u / 2); nuh padded to k_psf_x's tile
    int tx;                                     // k_psf_x threads along the columns: 8 or 16
    int rt, kx, kx_len;                         // k_psf_x row tiles, ix chunks, ix per chunk
    int vt, jt, ky, ky_len;                     // k_psf_y iv tiles, j tiles, iy chunks, iy per chunk
    int fb;                                     // k_psf_fold CTAs per set
    double* ctab;                               // [nx][nup]: 2 cos(2 pi s x xi)
    double2* T;                                 // [n_sets][kx][ny][nup]: stage A, one partial per ix chunk
    double* rsum;                               // [n_sets][rt][kx][3]: sum P (re, im), 1.0 if a kept opd is not finite
    double2* E;                                 // [n_sets][ky][n_v][nuh]: stage B, one partial per iy chunk
    double* bval; int* bidx;                    // [n_sets][fb]: per-CTA maximum of the PSF and its grid index
    double* psf;                                // [n_sets][n_v][n_u]
    double* strehl;                             // [n_sets][2]
    int *peak, *status;                         // [n_sets]
};

// Diffraction MTF of the wavefront (kern_mtf.cu)
struct MtfArgs {
    int n_sets, ny, nx;
    long long stride;
    const double* opd; const uint8_t* mask; const ort_stats* stats;
    const double *ys, *xs;                      // ys + s * ys_stride: the iy coordinates of set s
    long long ys_stride;                        // 0 or ny
    int n_freq;
    double scale;
    int n_slot;                                 // lag slots per azimuth, 2 n_freq + 1: k0 and k0 + 1 of each frequency, 0
    int lb, nlb;                                // lag slots per block of k_mtf_sag / k_mtf_tan, blocks
    int tiles_x, tiles;                         // k_mtf_pupil 32 x 32 tiles along x, per set
    int rg_s, rl_s;                             // k_mtf_sag row groups per set, rows per group
    int rg_t, rl_t;                             // k_mtf_tan column groups per set, columns per group
    double2* P;                                 // [n_sets][ny][nx]: mask exp(2 pi i W), column 0 doubled
    double2* PT;                                // [n_sets][nx][ny]: its transpose
    uint8_t* bad;                               // [n_sets][tiles]: 1 if a kept opd of the tile is not finite
    double* psag;                               // [n_sets][rg_s][n_slot]: sagittal lag sums per row group
    double2* ptan;                              // [n_sets][rg_t][n_slot]: tangential lag sums per column group
    double* otf;                                // [n_sets][2][n_freq][2]
    int* status;                                // [n_sets]
    double freqs[ORT_MTF_MAX_FREQS];            // cycles per image unit
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
// encircled energy: hist words per set, candidate-list capacity per set, and the launch sequence (*launches kernels,
// the same number whatever the sizes)
size_t energy_hist_words(int n_fracs);
unsigned energy_cand_cap(long long stride, int n_sets);
cudaError_t launch_energy(const EnergyArgs& A, const double* radii, int sm_count, cudaStream_t st, int* launches);
// Zernike fit: zern_dims fills js .. gx_resid from n_sets, n_max and stride; zern_gram_record is the doubles per gpart
// record; launch_zernike enqueues the four kernels
int zern_fitted_terms(int n_max);
cudaError_t zern_dims(ZernArgs& A, int sm_count);
size_t zern_gram_record(const ZernArgs& A);
cudaError_t launch_zernike(const ZernArgs& A, cudaStream_t st, int* launches);
// diffraction PSF: psf_dims fills nuh .. fb from n_sets, ny, nx, n_u and n_v (the scratch sizes follow from them);
// launch_psf enqueues the five kernels
cudaError_t psf_dims(PsfArgs& A, int sm_count);
cudaError_t launch_psf(const PsfArgs& A, cudaStream_t st, int* launches);
// diffraction MTF: mtf_occupancy sets the kernels' shared-memory limit and returns the resident CTAs/SM of the lag
// kernels [sagittal, tangential][global, staged] (once per context); mtf_dims fills n_slot .. rl_t from n_sets, ny, nx
// and n_freq (the scratch sizes follow from them); launch_mtf enqueues the four kernels
cudaError_t mtf_occupancy(int (&occ)[2][2]);
cudaError_t mtf_dims(MtfArgs& A, int sm_count, const int (&occ)[2][2]);
cudaError_t launch_mtf(const MtfArgs& A, cudaStream_t st, int* launches);
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
