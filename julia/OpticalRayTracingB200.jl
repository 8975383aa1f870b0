# OpticalRayTracingB200.jl -- drop-in GPU methods for the data-parallel hot path of
# OpticalRayTracing.jl, bound to libort_b200.so (include/ort_b200.h) with plain `ccall`.
#
#   * No CUDA.jl, no Triton, no multi-backend dispatch, no CPU fallback: if the library or a B200 is
#     missing, `ort_init` fails and the error is thrown.
#   * The public API is unchanged.  Batch variants (vectors of rays / candidates) and every method that takes the
#     backend tag `B200()` first are ADDED.  `full_trace(surfaces::Layout, system, H, k_rays, focus)` has exactly the
#     reference's signature (src/PupilSampling.jl:85), so routing existing calls through the GPU means REPLACING that
#     method: this is done at load time by `__init__` (an `@eval` into this module, which is why the module opts out of
#     precompilation -- Julia >= 1.10 rejects method overwriting while precompiling) unless ENV["ORT_B200_OVERRIDE"] = "0".
#     Without the override, call `full_trace(B200(), surfaces, system, H, ...)`.
#   * Multi-GPU: ENV["ORT_B200_GPUS"] = n (default 1) opens n contexts, joins them with ort_comm_init_all (NCCL inside
#     the library) and full_trace goes through ort_trace3d_grid_multi: y-rows block-sharded over the n GPUs, outputs in the
#     reference's order, statistics all-gathered and merged inside the library.
#   * NOT RUNNABLE in the build environment (Julia is not installed there) and therefore UNTESTED; the same C ABI is
#     driven from Python (opticalraytracing.jl_b200/_lib.py, host.py) and from plain C (examples/) in tests and benchmarks.
#
# Library path: ENV["ORT_B200_LIB"] (default "libort_b200.so" on the loader path).
__precompile__(false)
module OpticalRayTracingB200

using OpticalRayTracing
using OpticalRayTracing: Layout, Lens, System, RayBasis, SystemOrRayBasis, RealRay, RealRayError,
                         TransferMatrix, trace_chief_ray, trace_marginal_ray, trace_edge_rays,
                         spot_rays, λ
import OpticalRayTracing: full_trace, raytrace, transfer, reverse_transfer, vignetting, aberrations

const LIB = get(ENV, "ORT_B200_LIB", "libort_b200.so")

const ORT_ARITH_STRICT = Cint(0)
const ORT_ARITH_FAST = Cint(1)

"Backend tag: `full_trace(B200(), surfaces, system, H, ...)` never touches the reference's own methods."
struct B200 end
export B200

# --- POD mirrors of include/ort_b200.h -------------------------------------------------------
struct OrtField            # ort_field
    mode::Int32
    reserved::Int32
    u::Float64
    v::Float64
    ybar::Float64
    z0::Float64
    h_prime::Float64
    opd_xc::Float64        # extension (ORT_EXT_OPD): reference sphere centre / radius, reference OPL
    opd_yc::Float64
    opd_radius::Float64
    opl_ref::Float64
end

struct OrtOpts             # ort_opts
    arith::Int32
    compact::Int32
    ys_per_field::Int32
    ext::Int32             # ORT_EXT_OPD = 1, ORT_EXT_VIGNETTE = 2 (extensions; 0 = the reference's behaviour)
    wg_nu::Float64
    wg_lambda::Float64
    opd_scale::Float64
    gather_stats::Int32    # 1: this call is one rank's block of y-rows; stats = merged over the communicator
    reserved::Int32
end

struct OrtStats            # ort_stats
    n_kept::Int64
    mean_x::Float64
    mean_y::Float64
    m2_x::Float64
    m2_y::Float64
    r_max::Float64
    n_miss::Int64
    n_tir::Int64
    n_domain::Int64
    n_clip::Int64
    n_vig::Int64
    mean_opd::Float64
    m2_opd::Float64
    n_strict::Int64
end

struct OrtGridOut          # ort_grid_out
    ex::Ptr{Float64}
    ey::Ptr{Float64}
    r::Ptr{Float64}
    theta::Ptr{Float64}
    wx::Ptr{Float64}
    wy::Ptr{Float64}
    opd::Ptr{Float64}
    mask::Ptr{UInt8}
    flags::Ptr{UInt8}
    stats::Ptr{OrtStats}
    stats_local::Ptr{OrtStats}
end

# --- context ---------------------------------------------------------------------------------
const CTX = Ref{Ptr{Cvoid}}(C_NULL)

function check(rc::Cint)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:ort_last_error, LIB), Cstring, (Ptr{Cvoid},), CTX[]))
    error("libort_b200 error $rc: $msg")
end

const CTXS = Ptr{Cvoid}[]          # all contexts of this process (CTXS[1] == CTX[]); more than one with ORT_B200_GPUS

function ctx()
    if CTX[] == C_NULL
        ngpu = parse(Int, get(ENV, "ORT_B200_GPUS", "1"))
        dev0 = parse(Cint, get(ENV, "LOCAL_RANK", "0"))
        for d in 0:ngpu-1
            out = Ref{Ptr{Cvoid}}(C_NULL)
            rc = ccall((:ort_init, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint), out, dev0 + d)
            d == 0 && (CTX[] = out[])
            check(rc)
            push!(CTXS, out[])
        end
        ngpu > 1 && check(ccall((:ort_comm_init_all, LIB), Cint, (Ptr{Ptr{Cvoid}}, Cint), CTXS, ngpu))
        atexit(() -> foreach(c -> ccall((:ort_free, LIB), Cvoid, (Ptr{Cvoid},), c), CTXS))
    end
    return CTX[]
end

# Aspheric polynomial terms are Julia closures: they cannot cross the C ABI.  (A Layout whose p are genuine
# polynomials can pass their COEFFICIENTS through ort_set_polynomials -- see include/ort_b200.h -- but nothing in
# Polynomial{F} exposes them, so this shim accepts p == zero only.)
function require_conic(surfaces::Layout)
    all(p -> p.f === zero, surfaces.p) ||
        throw(ArgumentError("OpticalRayTracingB200: polynomial aspheric terms (p ≢ zero) are not supported on the GPU path"))
end

function set_layout(R::Vector{Float64}, t::Vector{Float64}, n::Vector{Float64}, K::Vector{Float64})
    check(ccall((:ort_set_layout, LIB), Cint,
                (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                ctx(), length(R), R, t, n, K))
end

# --- full_trace: src/PupilSampling.jl:85-147 -------------------------------------------------
# Lines :85-114 (prelude, ray aiming, Optim) are kept verbatim; the hot loop :115-138 and the
# reductions :139-146 become ONE ccall.
function full_trace(::B200, surfaces::Layout, system::SystemOrRayBasis, H::Float64,
                    k_rays::Int = spot_rays,
                    focus = system.marginal.z[end] - system.marginal.z[end-1];
                    arith = ORT_ARITH_FAST)
    require_conic(surfaces)
    H = abs(H)
    H ≤ 1.0 || throw(DomainError(H, "Domain: |H| ≤ 1.0"))
    stop = system.stop
    a_stop = abs(system.a[stop])
    real_chief = trace_chief_ray(surfaces, system)
    real_marginal = trace_marginal_ray(surfaces, system)
    EP_t = real_chief.z[1]
    Ū = real_chief.u[1]
    U = H * Ū
    u = tan(U)
    y_EP = abs(real_marginal.y[1])
    y1, y2 = (±(y_EP) - u * EP_t for (±) ∈ (+, -))
    y1, y2 = trace_edge_rays(surfaces, y1, y2, U, stop, a_stop)
    if typeof(system) <: System
        field = OrtField(0, 0, u, tan(0.0), 0.0, 1.0, u * system.f, 0.0, 0.0, 0.0, 0.0)
    else
        z0 = system.marginal.z[1]
        ȳ = system.chief.y[2] + system.chief.u[1] * z0
        field = OrtField(1, 0, 0.0, 0.0, ȳ, z0, system.chief.y[end], 0.0, 0.0, 0.0, 0.0)
    end
    # extend the surface matrix to the paraxial image plane (:111-114)
    R = [surfaces.R; Inf]; t = [surfaces.t; 0.0]; n = [surfaces.n; 1.0]; K = [surfaces.K; 0.0]
    t[end-1] = focus
    set_layout(R, t, n, K)
    ys = collect(range(y1, y2, k_rays))              # :121  (TwicePrecision range evaluated in Julia)
    xs = collect(range(0.0, y_EP, div(k_rays, 2)))   # :122
    N = length(ys) * length(xs)
    εx = Vector{Float64}(undef, N); εy = similar(εx); r = similar(εx); θ = similar(εx)
    stats = Ref(OrtStats(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0))
    opts = Ref(OrtOpts(arith, 1, 0, 0, 0.0, 1.0, 1.0, 0, 0))   # compact = 1: the reference's push! order
    GC.@preserve εx εy r θ stats begin
        out = Ref(OrtGridOut(pointer(εx), pointer(εy), pointer(r), pointer(θ), C_NULL, C_NULL, C_NULL,
                             C_NULL, C_NULL, Base.unsafe_convert(Ptr{OrtStats}, stats), C_NULL))
        if length(CTXS) > 1      # one call, all GPUs of this process: rows block-sharded, stats merged in the library
            check(ccall((:ort_trace3d_grid_multi, LIB), Cint,
                        (Ptr{Ptr{Cvoid}}, Cint, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64,
                         Ref{OrtOpts}, Ref{OrtGridOut}),
                        CTXS, length(CTXS), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop, opts, out))
        else
            check(ccall((:ort_trace3d_grid, LIB), Cint,
                        (Ptr{Cvoid}, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64,
                         Ref{OrtOpts}, Ref{OrtGridOut}),
                        ctx(), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop, opts, out))
        end
    end
    nk = stats[].n_kept
    resize!(εx, nk); resize!(εy, nk); resize!(r, nk); resize!(θ, nk)
    # take advantage of symmetry (:139-146)
    εy = [εy; εy]
    εx = [εx; -εx]
    ρ = min.(r / stats[].r_max, 1.0)     # r_max is the correctly rounded maximum; max(ρ) == 1 as in the reference (:142)
    ρ = [ρ; ρ]
    θ = [θ; π .- θ]
    nu = system.marginal.nu[end]
    # σ(εx, εy) (:169-173) from the kernel's mergeable moments: mirrored x has mean 0
    s = stats[]
    RMS = sqrt((2 * (s.m2_x + nk * s.mean_x^2) + 2 * s.m2_y) / (2 * nk))
    return RealRayError(εx, εy, nu, ρ, θ, H, RMS)
end

# --- through focus: full_trace at every focus of `foci` (EXTENSION, no reference method) -----------
# The prelude is full_trace's (:85-114) verbatim; the pupil grid is traced ONCE and evaluated on every image plane in one
# ccall (ort_trace3d_focus).  rms[j] == full_trace(surfaces, system, H, k_rays, foci[j]).RMS.  best_focus / best_rms: the
# vertex of the least-squares parabola of rms^2 over the foci (exact: the kept set is the same at every focus).
# Like the rest of this file it cannot be run in the repository that ships it (no Julia there); the Python host's
# through_focus is the tested form of the same calls.
function through_focus(::B200, surfaces::Layout, system::SystemOrRayBasis, H::Float64, foci::Vector{Float64};
                       k_rays::Int = spot_rays, arith = ORT_ARITH_FAST)
    require_conic(surfaces)
    H = abs(H)
    H ≤ 1.0 || throw(DomainError(H, "Domain: |H| ≤ 1.0"))
    stop = system.stop
    a_stop = abs(system.a[stop])
    real_chief = trace_chief_ray(surfaces, system)
    real_marginal = trace_marginal_ray(surfaces, system)
    EP_t = real_chief.z[1]
    Ū = real_chief.u[1]
    U = H * Ū
    u = tan(U)
    y_EP = abs(real_marginal.y[1])
    y1, y2 = (±(y_EP) - u * EP_t for (±) ∈ (+, -))
    y1, y2 = trace_edge_rays(surfaces, y1, y2, U, stop, a_stop)
    if typeof(system) <: System
        field = OrtField(0, 0, u, tan(0.0), 0.0, 1.0, u * system.f, 0.0, 0.0, 0.0, 0.0)
    else
        z0 = system.marginal.z[1]
        ȳ = system.chief.y[2] + system.chief.u[1] * z0
        field = OrtField(1, 0, 0.0, 0.0, ȳ, z0, system.chief.y[end], 0.0, 0.0, 0.0, 0.0)
    end
    # the extended surfaces of :111-114; t[end-1] is replaced by each focus inside the library
    R = [surfaces.R; Inf]; t = [surfaces.t; 0.0]; n = [surfaces.n; 1.0]; K = [surfaces.K; 0.0]
    set_layout(R, t, n, K)
    ys = collect(range(y1, y2, k_rays))              # :121
    xs = collect(range(0.0, y_EP, div(k_rays, 2)))   # :122
    M = length(foci)
    stats = [OrtStats(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0) for _ in 1:M]
    opts = Ref(OrtOpts(arith, 0, 0, 0, 0.0, 1.0, 1.0, 0, 0))
    GC.@preserve stats begin
        out = Ref(OrtGridOut(C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, pointer(stats), C_NULL))
        check(ccall((:ort_trace3d_focus, LIB), Cint,
                    (Ptr{Cvoid}, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64,
                     Ptr{Float64}, Cint, Ref{OrtOpts}, Ref{OrtGridOut}),
                    ctx(), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop, foci, M, opts, out))
    end
    rms = [s.n_kept == 0 ? NaN : sqrt((2 * (s.m2_x + s.n_kept * s.mean_x^2) + 2 * s.m2_y) / (2 * s.n_kept)) for s in stats]
    n_kept = stats[1].n_kept
    best_focus, best_rms = NaN, NaN
    if length(unique(foci)) ≥ 3 && all(isfinite, rms)
        fm = sum(foci) / M
        d = foci .- fm
        A, B, C = [d .^ 2 d ones(M)] \ (rms .^ 2)
        if A > 0
            best_focus = fm - B / (2A)
            best_rms = sqrt(max(C - B^2 / (4A), 0.0))
        end
    end
    return (rms = rms, n_kept = n_kept, best_focus = best_focus, best_rms = best_rms)
end

# --- encircled energy of the spot (EXTENSION, no reference method) --------------------------------
# full_trace's prelude (:85-114), then ONE ccall (ort_trace3d_energy) that sweeps the pupil grid full-grid on the device --
# at `focus`, or through focus at `foci` -- and computes the encircled (metric = ORT_ENERGY_CIRCLE) or ensquared
# (ORT_ENERGY_SQUARE) energy there: fraction[j, k] of the mirrored spot within radii[k] of the centre, and radius[j, i],
# the k-th smallest distance with k = clamp(ceil(fractions[i] n), 1, n).  Only these numbers cross PCIe.
# Like the rest of this file it cannot be run in the repository that ships it (no Julia there); the Python host's
# encircled_energy is the tested form of the same calls.
struct OrtEnergyReq
    metric::Int32; center::Int32; n_radii::Int32; n_fracs::Int32
    radii::Ptr{Float64}; fracs::Ptr{Float64}
end
const ORT_ENERGY_CIRCLE, ORT_ENERGY_SQUARE = Int32(0), Int32(1)
const ORT_CENTER_CENTROID, ORT_CENTER_PARAXIAL = Int32(0), Int32(1)

function encircled_energy(::B200, surfaces::Layout, system::SystemOrRayBasis, H::Float64;
                          radii::Vector{Float64} = Float64[], fractions::Vector{Float64} = [0.5, 0.8, 0.9],
                          k_rays::Int = spot_rays, focus = nothing, foci::Union{Nothing, Vector{Float64}} = nothing,
                          metric = ORT_ENERGY_CIRCLE, center = ORT_CENTER_CENTROID, arith = ORT_ARITH_FAST)
    require_conic(surfaces)
    H = abs(H)
    H ≤ 1.0 || throw(DomainError(H, "Domain: |H| ≤ 1.0"))
    focus === nothing && (focus = system.marginal.z[end] - system.marginal.z[end-1])   # :87
    stop = system.stop
    a_stop = abs(system.a[stop])
    real_chief = trace_chief_ray(surfaces, system)
    real_marginal = trace_marginal_ray(surfaces, system)
    EP_t = real_chief.z[1]
    Ū = real_chief.u[1]
    U = H * Ū
    u = tan(U)
    y_EP = abs(real_marginal.y[1])
    y1, y2 = (±(y_EP) - u * EP_t for (±) ∈ (+, -))
    y1, y2 = trace_edge_rays(surfaces, y1, y2, U, stop, a_stop)
    if typeof(system) <: System
        field = OrtField(0, 0, u, tan(0.0), 0.0, 1.0, u * system.f, 0.0, 0.0, 0.0, 0.0)
    else
        z0 = system.marginal.z[1]
        ȳ = system.chief.y[2] + system.chief.u[1] * z0
        field = OrtField(1, 0, 0.0, 0.0, ȳ, z0, system.chief.y[end], 0.0, 0.0, 0.0, 0.0)
    end
    R = [surfaces.R; Inf]; t = [surfaces.t; 0.0]; n = [surfaces.n; 1.0]; K = [surfaces.K; 0.0]
    t[end-1] = focus                                 # :114 (replaced by each of foci inside the library)
    set_layout(R, t, n, K)
    ys = collect(range(y1, y2, k_rays))              # :121
    xs = collect(range(0.0, y_EP, div(k_rays, 2)))   # :122
    M = foci === nothing ? 1 : length(foci)
    stats = [OrtStats(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0) for _ in 1:M]
    counts = zeros(Int64, length(radii), M)          # [M][R] in C order
    radius = zeros(Float64, length(fractions), M)
    opts = Ref(OrtOpts(arith, 0, 0, 0, 0.0, 1.0, 1.0, 0, 0))
    GC.@preserve stats counts radius radii fractions begin
        req = Ref(OrtEnergyReq(metric, center, length(radii), length(fractions),
                               isempty(radii) ? C_NULL : pointer(radii), isempty(fractions) ? C_NULL : pointer(fractions)))
        check(ccall((:ort_trace3d_energy, LIB), Cint,
                    (Ptr{Cvoid}, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ptr{Float64},
                     Cint, Ref{OrtOpts}, Ref{OrtEnergyReq}, Ptr{OrtStats}, Ptr{Int64}, Ptr{Float64}),
                    ctx(), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop,
                    foci === nothing ? C_NULL : foci, foci === nothing ? 0 : M, opts, req, pointer(stats),
                    isempty(radii) ? C_NULL : pointer(counts), isempty(fractions) ? C_NULL : pointer(radius)))
    end
    n_kept = stats[1].n_kept
    fraction = n_kept == 0 ? fill(NaN, M, length(radii)) : permutedims(counts) ./ n_kept
    return (foci = foci === nothing ? [Float64(focus)] : foci, fraction = fraction, radius = permutedims(radius),
            n_kept = n_kept)
end

# --- Zernike decomposition of the wavefront (EXTENSION, no reference method) ------------------------------
# The OPD sweep of the Python host's wavefront() -- full_trace's prelude, the chief ray through the centre of the stop,
# the reference sphere centred on its image point with radius image plane - paraxial exit pupil -- then ONE ccall
# (ort_trace3d_zernike) that sweeps the pupil grid with ORT_EXT_OPD on the device and fits ANSI Zernike terms n <= n_max
# to the mirrored OPD map there (coefficients in waves, ANSI order j = (n(n+2) + m)/2).  Only coef, the residual RMS /
# PV and the status cross PCIe.  norm = :stop puts the stop rim at rho = 1, :rmax the largest kept r (RealRayError.r).
# Like the rest of this file it cannot be run in the repository that ships it (no Julia there); the Python host's
# zernike is the tested form of the same calls.
struct OrtZernikeReq
    n_max::Int32; reserved::Int32; r_norm::Float64
end
const ORT_EXT_OPD, ORT_EXT_VIGNETTE = Int32(1), Int32(2)

# The OPD sweep of the Python host's wavefront() for one field point: full_trace's prelude, the chief ray through the
# centre of the stop, the reference sphere centred on its image point with radius image plane - paraxial exit pupil.
# Leaves the extended layout (image plane in the last medium) and the apertures (vignette) set.
function opd_sweep_setup(surfaces::Layout, system::System, H::Float64, k_rays::Int, focus, vignette::Bool)
    H = abs(H)
    H ≤ 1.0 || throw(DomainError(H, "Domain: |H| ≤ 1.0"))
    focus === nothing && (focus = system.marginal.z[end] - system.marginal.z[end-1])   # :87
    stop = system.stop
    a_stop = abs(system.a[stop])
    real_chief = trace_chief_ray(surfaces, system)
    real_marginal = trace_marginal_ray(surfaces, system)
    EP_t = real_chief.z[1]
    U = H * real_chief.u[1]
    u = tan(U)
    y_EP = abs(real_marginal.y[1])
    y1, y2 = trace_edge_rays(surfaces, y_EP - u * EP_t, -y_EP - u * EP_t, U, stop, a_stop)
    # chief ray: the entrance height that meets the stop at y = 0 (2-D secant solve on the bare layout)
    set_layout([surfaces.R; Inf], [surfaces.t; 0.0], [surfaces.n; 1.0], [surfaces.K; 0.0])
    y_c = Ref(-u * EP_t)
    check(ccall((:ort_aim2d, LIB), Cint, (Ptr{Cvoid}, Int64, Ref{Float64}, Ref{Float64}, Ref{Float64}, Cint, Cint, Cint,
                                          Float64, Cint, Ref{Float64}, Ptr{Int32}),
                ctx(), 1, Ref(-u * EP_t), Ref(U), Ref(0.0), stop, 0, 1, a_stop, 0, y_c, C_NULL))
    # the extended layout: image plane at `focus`, in the last medium (no refraction onto it)
    R = [surfaces.R; Inf]; t = [surfaces.t; 0.0]; n = [surfaces.n; surfaces.n[end]]; K = [surfaces.K; 0.0]
    t[end-1] = focus                                 # :114
    set_layout(R, t, n, K)
    a = vignette ? Float64.(system.a) : Float64[]
    check(ccall((:ort_set_apertures, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), ctx(), length(a),
                isempty(a) ? C_NULL : a))
    rows1 = length(R) - 1
    xv = zeros(rows1); yv = zeros(rows1); opl = zeros(1)
    check(ccall((:ort_trace3d_rays_opl, LIB), Cint,
                (Ptr{Cvoid}, Int64, Ref{Float64}, Ref{Float64}, Ref{Float64}, Ref{Float64}, Cint, Ptr{Float64},
                 Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Ptr{Float64}),
                ctx(), 1, y_c, Ref(0.0), Ref(u), Ref(0.0), ORT_ARITH_STRICT, xv, yv, C_NULL, C_NULL, opl))
    Rr = focus - system.XP.t                         # image plane - paraxial exit pupil
    opl_ref = opl[1] + surfaces.n[1] * (y_c[] * u / sqrt(u^2 + 1)) - surfaces.n[end] * Rr
    field = OrtField(0, 0, u, 0.0, 0.0, 0.0, u * system.f, 0.0, yv[end], Rr, opl_ref)
    ys = collect(range(y1, y2, k_rays))              # :121
    xs = collect(range(0.0, y_EP, div(k_rays, 2)))   # :122
    return field, ys, xs, stop, a_stop, y_EP
end

function zernike(::B200, surfaces::Layout, system::System, H::Float64; n_max::Int = 8, k_rays::Int = spot_rays,
                 focus = nothing, λ = 587.5618e-6, vignette::Bool = false, norm::Symbol = :stop, arith = ORT_ARITH_FAST)
    require_conic(surfaces)
    0 ≤ n_max ≤ 12 || throw(DomainError(n_max, "0 ≤ n_max ≤ 12"))
    norm ∈ (:stop, :rmax) || throw(ArgumentError("norm is :stop or :rmax"))
    field, ys, xs, stop, a_stop, _ = opd_sweep_setup(surfaces, system, H, k_rays, focus, vignette)
    J = (n_max + 1) * (n_max + 2) ÷ 2
    stats = [OrtStats(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0)]
    coef = zeros(J); resid = zeros(2); status = zeros(Int32, 1)
    opts = Ref(OrtOpts(arith, 0, 0, ORT_EXT_OPD | (vignette ? ORT_EXT_VIGNETTE : Int32(0)), 0.0, 1.0, -1.0 / λ, 0, 0))
    req = Ref(OrtZernikeReq(n_max, 0, norm == :stop ? a_stop : 0.0))
    check(ccall((:ort_trace3d_zernike, LIB), Cint,
                (Ptr{Cvoid}, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ref{OrtOpts},
                 Ref{OrtZernikeReq}, Ptr{OrtStats}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
                ctx(), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop, opts, req, stats, coef, resid,
                status))
    check(ccall((:ort_set_apertures, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), ctx(), 0, C_NULL))
    nm = [(nn, m) for nn in 0:n_max for m in -nn:2:nn]
    return (n = first.(nm), m = last.(nm), coef = coef, rms_resid = resid[1], pv_resid = resid[2],
            status = Int(status[1]), n_kept = stats[1].n_kept)
end

# --- Diffraction PSF and Strehl ratio of the wavefront (EXTENSION, no reference method) ---------------------------
# The OPD sweep of zernike, then ONE ccall (ort_trace3d_psf) that sweeps the pupil grid with ORT_EXT_OPD on the device
# and computes the scalar Fraunhofer PSF of the mirrored pupil there, s = 1/(λ f): pupil height h maps to the image-space
# direction sine h/f (obliquity, apodisation and pupil distortion neglected).  psf is n_u × n_v: psf[iu, iv] is pixel
# (iu, iv) of the C layout [iv][iu]; u, v are the pixel centres in mm from the chief ray's image point.
# strehl: psf at that point; peak: the maximum over the grid.  Only the pixel grid crosses PCIe.  Not runnable here (no
# Julia); the Python host's psf is the tested form of the same calls.
struct OrtPsfReq
    n_u::Int32; n_v::Int32; du::Float64; dv::Float64; scale::Float64
end

function psf(::B200, surfaces::Layout, system::System, H::Float64; n_pix = nothing, pixel = nothing,
             k_rays::Int = spot_rays, focus = nothing, λ = 587.5618e-6, vignette::Bool = false, arith = ORT_ARITH_FAST)
    require_conic(surfaces)
    n_u, n_v = n_pix === nothing ? (k_rays - 1, k_rays - 1) : n_pix isa Integer ? (n_pix, n_pix) : Tuple(n_pix)
    (1 ≤ n_u ≤ 1024 && 1 ≤ n_v ≤ 1024) || throw(DomainError(n_pix, "1 ≤ n_pix ≤ 1024"))
    s = 1.0 / (λ * system.f)
    field, ys, xs, stop, a_stop, y_EP = opd_sweep_setup(surfaces, system, H, k_rays, focus, vignette)
    du, dv = pixel === nothing ? (1 / (4 * s * y_EP), 1 / (4 * s * y_EP)) : pixel isa Real ? (pixel, pixel) : Tuple(pixel)
    dx, dy = length(xs) > 1 ? xs[2] - xs[1] : 0.0, length(ys) > 1 ? abs(ys[2] - ys[1]) : 0.0
    if !(n_u * du * s * dx ≤ 1 + 1e-9 && n_v * dv * s * dy ≤ 1 + 1e-9)
        check(ccall((:ort_set_apertures, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), ctx(), 0, C_NULL))
        throw(ArgumentError("the pixel grid exceeds the alias period of the pupil grid: raise k_rays"))
    end
    stats = [OrtStats(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0)]
    img = zeros(n_u, n_v); strehl = zeros(2); peak = zeros(Int32, 1); status = zeros(Int32, 1)
    opts = Ref(OrtOpts(arith, 0, 0, ORT_EXT_OPD | (vignette ? ORT_EXT_VIGNETTE : Int32(0)), 0.0, 1.0, -1.0 / λ, 0, 0))
    req = Ref(OrtPsfReq(n_u, n_v, du, dv, s))
    check(ccall((:ort_trace3d_psf, LIB), Cint,
                (Ptr{Cvoid}, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ref{OrtOpts},
                 Ref{OrtPsfReq}, Ptr{OrtStats}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
                ctx(), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop, opts, req, stats, img, strehl,
                peak, status))
    check(ccall((:ort_set_apertures, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), ctx(), 0, C_NULL))
    u = ((0:n_u-1) .- (n_u - 1) / 2) .* du
    v = ((0:n_v-1) .- (n_v - 1) / 2) .* dv
    return (u = collect(u), v = collect(v), psf = img, strehl = strehl[1], peak = strehl[2],
            peak_uv = peak[1] < 0 ? (NaN, NaN) : (u[peak[1] % n_u + 1], v[peak[1] ÷ n_u + 1]),
            status = Int(status[1]), n_kept = stats[1].n_kept)
end

# --- Diffraction MTF of the wavefront (EXTENSION, no reference method) -------------------------------------------------
# The OPD sweep of psf, then ONE ccall (ort_trace3d_mtf) that sweeps the pupil grid with ORT_EXT_OPD on the device and
# computes there the optical transfer function of the PSF that psf describes (s = 1/(λ f)): the normalised
# autocorrelation of the mirrored pupil exp(2πi W), sagittal (frequency along x) and tangential (along y), interpolated
# linearly between lattice lags.  freqs in cycles/mm, default 32 from 0 to 1/(λ F#) = 2 s y_EP; otf is 2 × n_freq
# (row 1 sagittal, row 2 tangential), mtf = abs.(otf), ptf = angle.(otf).  Only the OTF values cross PCIe.  Not runnable
# here (no Julia); the Python host's mtf is the tested form of the same calls.
struct OrtMtfReq
    n_freq::Int32; reserved::Int32; freqs::Ptr{Float64}; scale::Float64
end

function mtf(::B200, surfaces::Layout, system::System, H::Float64; freqs = nothing, k_rays::Int = spot_rays,
             focus = nothing, λ = 587.5618e-6, vignette::Bool = false, arith = ORT_ARITH_FAST)
    require_conic(surfaces)
    k_rays ≥ 4 || throw(DomainError(k_rays, "k_rays ≥ 4"))
    s = 1.0 / (λ * system.f)
    field, ys, xs, stop, a_stop, y_EP = opd_sweep_setup(surfaces, system, H, k_rays, focus, vignette)
    f = freqs === nothing ? collect(range(0.0, 2 * s * y_EP, length = 32)) : Vector{Float64}(freqs)
    if !(1 ≤ length(f) ≤ 1024 && all(x -> isfinite(x) && x ≥ 0, f))
        check(ccall((:ort_set_apertures, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), ctx(), 0, C_NULL))
        throw(DomainError(freqs, "1 to 1024 frequencies, finite and ≥ 0"))
    end
    stats = [OrtStats(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0)]
    otf = zeros(2, length(f), 2); status = zeros(Int32, 1)          # otf[ri, j, a] is C otf[a][j][ri] ([az][f][2])
    opts = Ref(OrtOpts(arith, 0, 0, ORT_EXT_OPD | (vignette ? ORT_EXT_VIGNETTE : Int32(0)), 0.0, 1.0, -1.0 / λ, 0, 0))
    GC.@preserve f begin
        req = Ref(OrtMtfReq(length(f), 0, pointer(f), s))
        check(ccall((:ort_trace3d_mtf, LIB), Cint,
                    (Ptr{Cvoid}, Ref{OrtField}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ref{OrtOpts},
                     Ref{OrtMtfReq}, Ptr{OrtStats}, Ptr{Float64}, Ptr{Int32}),
                    ctx(), Ref(field), 1, ys, length(ys), xs, length(xs), stop, a_stop, opts, req, stats, otf, status))
    end
    check(ccall((:ort_set_apertures, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), ctx(), 0, C_NULL))
    o = [complex(otf[1, j, a], otf[2, j, a]) for a in 1:2, j in 1:length(f)]
    nx, ny = length(xs), length(ys)
    cutoff = (2 * (nx - 1) * (xs[end] / (nx - 1)) * s, (ny - 1) * abs((ys[end] - ys[1]) / (ny - 1)) * s)
    return (freqs = f, otf = o, mtf = abs.(o), ptf = angle.(o), cutoff = cutoff, status = Int(status[1]),
            n_kept = stats[1].n_kept)
end

# --- batched 2-D meridional real rays: src/RayTracing.jl:145-173 ------------------------------
# Returns (y, U, ts), each rows × N, for N rays in one kernel launch.
function raytrace(surfaces::Layout{T}, ys::Vector{Float64}, Us::Vector{Float64}, ::Type{RealRay}) where T
    require_conic(surfaces)
    set_layout(surfaces.R, surfaces.t, surfaces.n, surfaces.K)
    rows, N = length(surfaces.R), length(ys)
    y = Matrix{Float64}(undef, N, rows); U = similar(y); ts = similar(y)   # [rows][N], ray index fastest
    flags = Vector{UInt8}(undef, N)
    aspheric = T <: OpticalRayTracing.Aspheric ? 1 : 0                     # :171-173 dispatch
    check(ccall((:ort_trace2d_batch, LIB), Cint,
                (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}),
                ctx(), N, ys, Us, aspheric, y, U, ts, flags))
    return permutedims(y), permutedims(U), permutedims(ts)
end

# --- batched paraxial y-nu: src/RayTracing.jl:127-143 ------------------------------------------
# Returns the reference's rt tables (k+1) × N for y and nu, plus the clip row per ray.
function raytrace(lens::Lens, ys::Vector{Float64}, ωs::Vector{Float64},
                  a::AbstractVector = fill(Inf, size(lens, 1)); clip = false)
    τ, ϕ = collect(lens[:,1]), collect(lens[:,2])
    k, N = length(τ), length(ys)
    yf = Vector{Float64}(undef, N); ωf = similar(yf); ci = Vector{Int32}(undef, N)
    Y = Matrix{Float64}(undef, N, k + 1); W = similar(Y)
    av = collect(Float64, a)
    check(ccall((:ort_paraxial_batch, LIB), Cint,
                (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Int64, Ptr{Float64},
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}),
                ctx(), k, τ, ϕ, av, clip ? 1 : 0, ORT_ARITH_STRICT, N, ys, ωs, yf, ωf, ci, Y, W))
    return permutedims(Y), permutedims(W), ci
end

# --- batched transfer-matrix apply: src/TransferMatrix.jl:8-17 ---------------------------------
# V is 2 × N ([y; nu] per column), exactly Julia's column-major memory.
function transfer(M::AbstractMatrix, V::Matrix{Float64}, τ, τ′)
    size(V, 1) == 2 || throw(DimensionMismatch("V must be 2 × N"))
    Mc = collect(Float64, M); out = similar(V)
    check(ccall((:ort_transfer_batch, LIB), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, Cint, Int64, Ptr{Float64}, Ptr{Float64}),
                ctx(), Mc, τ, τ′, 0, size(V, 2), V, out))
    return out
end

function reverse_transfer(M::AbstractMatrix, V::Matrix{Float64}, τ′, τ)
    size(V, 1) == 2 || throw(DimensionMismatch("V must be 2 × N"))
    Mc = collect(Float64, M); out = similar(V)
    check(ccall((:ort_transfer_batch, LIB), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, Cint, Int64, Ptr{Float64}, Ptr{Float64}),
                ctx(), Mc, τ, τ′, 1, size(V, 2), V, out))
    return out
end

# --- population methods (additive): one prescription per candidate, shared apertures -----------
# pack R, t, n, K of every candidate as [C][4][rows] (rows fastest), the layout ort_b200.h documents
function pack(candidates::Vector{<:Layout})
    rows = length(first(candidates).R)
    P = Array{Float64}(undef, rows, 4, length(candidates))
    for (c, L) in enumerate(candidates)
        P[:, 1, c] = L.R; P[:, 2, c] = L.t; P[:, 3, c] = L.n; P[:, 4, c] = L.K
    end
    return P, rows
end

# full_trace (src/PupilSampling.jl:85-147) for every candidate: per-candidate solve, ray aiming, pupil grid, spot
# statistics.  Returns (spot 4 × C = n_kept, mean_x, mean_y, RMS of the half pupil; aim 24 × C prelude records).
function full_trace(candidates::Vector{<:Layout}, a::AbstractVector, h′, H, k_rays = 64; arith = 1)
    abs(H) ≤ 1.0 || throw(DomainError(H, "Domain: |H| ≤ 1.0"))
    P, rows = pack(candidates); C = length(candidates)
    aim = Matrix{Float64}(undef, 24, C); spot = Matrix{Float64}(undef, 4, C)
    av = collect(Float64, a)
    check(ccall((:ort_aim_candidates, LIB), Cint,
                (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Cint, Ptr{Float64}),
                ctx(), rows, C, P, av, h′, H, 1, aim))
    check(ccall((:ort_trace3d_candidates_aimed, LIB), Cint,
                (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Cint, Ptr{Float64}),
                ctx(), rows, C, P, aim, k_rays, k_rays ÷ 2, arith, spot))
    return spot, aim
end

# vignetting(system, a) (src/Vignetting.jl:1-30) for every candidate; out is (6k + 12) × C, see ort_b200.h
function vignetting(candidates::Vector{<:Layout}, a::AbstractVector, h′; a_vig = a)
    P, rows = pack(candidates); C = length(candidates)
    out = Matrix{Float64}(undef, 6 * (rows - 1) + 12, C)
    check(ccall((:ort_vignetting_candidates, LIB), Cint,
                (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Float64, Ptr{Float64}),
                ctx(), rows, C, P, collect(Float64, a), collect(Float64, a_vig), h′, out))
    return out
end

# first-order solve + Seidel sums (src/SeidelAberrations.jl:6-53) for every candidate; out is 16 × C
function aberrations(candidates::Vector{<:Layout}, a::AbstractVector, h′; λ = 587.5618e-6, δn = zeros(length(first(candidates).R)))
    P, rows = pack(candidates); C = length(candidates)
    out = Matrix{Float64}(undef, 16, C)
    check(ccall((:ort_seidel_candidates, LIB), Cint,
                (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                ctx(), rows, C, P, collect(Float64, a), h′, λ, collect(Float64, δn), out, C_NULL))
    return out
end

transfer(system::System, V::Matrix{Float64}, τ, τ′) = transfer(system.M, V, τ, τ′)
reverse_transfer(system::System, V::Matrix{Float64}, τ′, τ) = reverse_transfer(system.M, V, τ′, τ)

full_trace(b::B200, system::System, H::Float64, args...; kw...) = full_trace(b, system.layout, system, H, args...; kw...)

# The drop-in proper: replace the reference's own method (same signature, src/PupilSampling.jl:85) so that existing
# user code -- full_trace(system, H), spot_diagram, ... -- runs on the GPU unchanged.  Done at load time, not at
# definition time (see the header); ENV["ORT_B200_OVERRIDE"] = "0" leaves the reference's method in place.
function __init__()
    get(ENV, "ORT_B200_OVERRIDE", "1") == "0" && return
    @eval function OpticalRayTracing.full_trace(surfaces::Layout, system::SystemOrRayBasis, H::Float64,
                                                k_rays::Int = spot_rays,
                                                focus = system.marginal.z[end] - system.marginal.z[end-1])
        full_trace(B200(), surfaces, system, H, k_rays, focus)
    end
end

end # module
