"""Host-side mirror of the reference's public API for the hot path.

Same names, argument meaning and error behaviour as Sagnac/OpticalRayTracing.jl
(src/OpticalRayTracing.jl:6-50): solve, raytrace, trace_marginal_ray, trace_chief_ray,
full_trace, transfer, reverse_transfer, flatten, wavegrad, TSA, SA, Layout, Lens, TransferMatrix.
Every ray that is traced -- single rays of the prelude included -- goes through the C ABI of
libort_b200.so (`backend`, default: a GPU Context).  There is no CPU fallback; tests may inject
another backend object to exercise the host logic without a GPU.

Julia is 1-based; the `stop` fields here keep the reference's 1-based value.
"""
import math
from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import _lib

EPS = math.sqrt(np.finfo(np.float64).eps)   # const eps = sqrt(eps())          src/RayTracing.jl:1
K_RAYS = 22                                 # const k_rays                     src/RayTracing.jl:4
SPOT_RAYS = 64                              # const spot_rays                  src/RayTracing.jl:7
LAMBDA = 587.5618e-6                        # He d-line, mm                    src/SeidelAberrations.jl:2


class RealRay:            # dispatch tag: raytrace(surfaces, y, U, RealRay)            RayTracing.jl:145
    pass


class VectorRealRay:      # dispatch tag: raytrace(surfaces, y, x, U, V, Vector{RealRay})  PupilSampling.jl:34
    pass


# ------------------------------------------------------------------------------------------------
# backend
# ------------------------------------------------------------------------------------------------
_default_backend = None


def default_backend():
    """The process-wide GPU context (device = LOCAL_RANK or 0).  Raises if no B200 is usable."""
    global _default_backend
    if _default_backend is None:
        import os
        _default_backend = _lib.Context(int(os.environ.get("LOCAL_RANK", "0")))
    return _default_backend


def set_default_backend(b):
    global _default_backend
    _default_backend = b


def _be(backend):
    return backend if backend is not None else default_backend()


# ------------------------------------------------------------------------------------------------
# collect(range(start, stop, length))  -- Julia Base, base/twiceprecision.jl (NOT under the reference tree)
# ------------------------------------------------------------------------------------------------
def _add12(x, y):
    """Base.add12: (hi, lo) with hi + lo == x + y exactly (branch on magnitude, then fast two-sum)"""
    swap = np.abs(y) > np.abs(x)
    big, little = np.where(swap, y, x), np.where(swap, x, y)
    hi = big + little
    return hi, (big - hi) + little


def _truncbits(x, nb):
    """Base.truncbits: clear the nb low bits of the significand"""
    b = np.float64(x).view(np.uint64)
    return float((b & (np.uint64(0xFFFFFFFFFFFFFFFF) << np.uint64(nb))).view(np.float64))


def jl_range(start, stop, length):
    """The Float64 values of Julia's `range(start, stop, length)` (src/PupilSampling.jl:121-122 builds the pupil grid
    with it).  Julia does not compute start + i*step in plain Float64 (numpy.linspace does): a Float64 range is a
    StepRangeLen{Float64, TwicePrecision, TwicePrecision} whose reference value and step are double-double numbers
    chosen so that BOTH end points are hit exactly, and element i is ref + (i - offset) step evaluated in
    double-double -- in effect the correctly rounded linear interpolation.  This restates Base._linspace and
    Base.unsafe_getindex (base/twiceprecision.jl, Julia 1.10/1.11) for end points that are not small rationals --
    every aimed grid -- and uses exact rational arithmetic, correctly rounded, where Julia takes its rational branch
    (end points like 0.0 and 10.0).  Julia itself is absent here, so this is pinned only against exact interpolation
    (tests/test_host_logic.py); the shim passes collect(range(...)) so in the real drop-in these are inputs."""
    n = int(length)
    a, b = float(start), float(stop)
    if n < 0:
        raise ValueError("range: negative length")
    if n == 0:
        return np.empty(0)
    if n == 1:
        if a != b:
            raise ValueError("range(start, stop, length=1): endpoints differ")
        return np.array([a])
    if a == b:
        return np.full(n, a)
    if not (math.isfinite(a) and math.isfinite(b)):
        raise ValueError("start and stop must be finite")
    if _small_rational(a) and _small_rational(b):
        from fractions import Fraction
        fa, fb = Fraction(a), Fraction(b)
        return np.array([float(fa + (fb - fa) * Fraction(i, n - 1)) for i in range(n)])
    # Base._linspace(start, stop, len)
    delta, dfac = b - a, 1
    if not math.isfinite(delta):
        delta, dfac = b / n - a / n, n
    tmin = -(a / delta) / dfac
    imin = int(np.rint(tmin * (n - 1) + 1))            # round-half-even, as Julia's round(Int, x)
    if 1 < imin < n:
        t = (imin - 1) / (n - 1)
        ref = (1 - t) * a + t * b
        step = (ref - a) / (imin - 1) if imin - 1 < n - imin else (b - ref) / (n - imin)
    elif imin <= 1:
        imin, ref, step = 1, a, (delta / (n - 1)) * dfac
    else:
        imin, ref, step = n, b, (delta / (n - 1)) * dfac
    m, k = float(np.nextafter(np.finfo(np.float64).max, 0.0)), max(imin - 1, n - imin)
    step_hi_pre = min(max(step, max(-(m + ref) / k, (-m + ref) / k)), min((m - ref) / k, (m + ref) / k))
    nb = min(27, int(math.ceil(math.log2(max(imin - 1, n - imin)))) + 1)      # nbitslen(Float64, len, imin)
    step_hi = _truncbits(step_hi_pre, nb)
    x1_hi, x1_lo = _add12(np.float64((1 - imin) * step_hi), np.float64(ref))
    x2_hi, x2_lo = _add12(np.float64((n - imin) * step_hi), np.float64(ref))
    lo_a, lo_b = (a - float(x1_hi)) - float(x1_lo), (b - float(x2_hi)) - float(x2_lo)
    step_lo = (lo_b - lo_a) / (n - 1)
    ref_lo = lo_a - (1 - imin) * step_lo
    # steprangelen_hp(..., (ref, ref_lo), (step_hi, step_lo), 0, len, imin) stores both pairs as they are: step_hi keeps
    # its nb cleared low bits, so (i - offset) * step_hi below is exact
    s_hi, s_lo = step_hi, step_lo
    # Base.unsafe_getindex(r::StepRangeLen{T, <:TwicePrecision, <:TwicePrecision}, i)
    u = np.arange(1, n + 1, dtype=np.float64) - imin
    shift_hi, shift_lo = u * s_hi, u * s_lo
    x_hi, x_lo = _add12(np.full(n, ref), shift_hi)
    return x_hi + (x_lo + (shift_lo + ref_lo))


def _small_rational(x):
    """True where Base.rat finds the exact value of x as a ratio of integers below 2^24 (continued fractions): Julia's
    range then takes its integer branch (Base.linspace with numerators / denominator)"""
    y, a, b, c, d, m = x, 1, 0, 0, 1, 16777216.0
    while abs(y) <= m:
        f = int(y)
        y -= f
        a, c = f * a + c, a
        b, d = f * b + d, b
        if max(abs(a), abs(b)) > m:
            return False
        if b != 0 and a / b == x:
            return True
        if y == 0.0:
            return False
        y = 1.0 / y
    return False


# ------------------------------------------------------------------------------------------------
# types (src/Types.jl)
# ------------------------------------------------------------------------------------------------
class Layout:
    """Layout{Spherical|Aspheric} (src/Types.jl:82-112): columns R, t, n, K.  Polynomial terms `p` are arbitrary Julia
    closures in the reference and cannot cross the C ABI; here they are accepted in COEFFICIENT form (an extension):
    p[i] = (c0, c1, c2, ...) means p_i(y) = c0 + c1 y + c2 y^2 + ... for row i (None or empty = zero); callables are
    rejected.  FAST traces them with fast_step's polynomial body (STRICT when the layout also holds a mirror)."""

    def __init__(self, M, K=None, aspheric=None, p=None):
        P = None
        if p is not None:
            rows_p = list(p)
            if any(callable(pi) for pi in rows_p):
                raise ValueError("ort_b200: aspheric polynomial terms must be given as coefficient sequences "
                                 "(closures cannot cross the C ABI)")
            coefs = [np.atleast_1d(np.asarray([] if pi is None else pi, dtype=np.float64)) for pi in rows_p]
            ncoef = max((len(c) for c in coefs), default=0)
            if ncoef > 0 and any(np.any(c != 0.0) for c in coefs):
                P = np.zeros((len(coefs), ncoef))
                for i, c in enumerate(coefs):
                    P[i, :len(c)] = c
                if aspheric is None:
                    aspheric = True
        M = np.array(M, dtype=np.float64)
        if M.ndim != 2 or M.shape[1] < 3:
            raise ValueError("Layout needs rows of [R t n] or [R t n K]")
        if K is None and M.shape[1] > 3:
            K = M[:, 3]
            if aspheric is None:
                aspheric = True
        self.R, self.t, self.n = M[:, 0].copy(), M[:, 1].copy(), M[:, 2].copy()
        self.K = np.zeros(len(self.R)) if K is None else np.array(K, dtype=np.float64)
        self.aspheric = bool(aspheric)
        if P is not None and P.shape[0] != len(self.R):
            raise ValueError("Layout: one polynomial (coefficient sequence) per row")
        self.P = P                                   # (rows, ncoef) or None

    def upload(self, be):
        """prescription (+ polynomial terms) to the backend"""
        be.set_layout(self.M3, self.K)
        if self.P is not None:
            be.set_polynomials(self.P)

    @property
    def M3(self):
        return np.column_stack([self.R, self.t, self.n])

    def __len__(self):
        return len(self.R)


def _as_layout(surfaces):
    return surfaces if isinstance(surfaces, Layout) else Layout(surfaces)


@dataclass
class Lens:
    """Lens (src/Types.jl:77-80): k x 2 [tau phi] and n."""
    M: np.ndarray
    n: np.ndarray

    @property
    def tau(self):
        return self.M[:, 0]

    @property
    def phi(self):
        return self.M[:, 1]


def make_lens(surfaces):
    """Lens(surfaces) -- src/RayTracing.jl:38-53 (O(k) host arithmetic, no rays)."""
    L = _as_layout(surfaces)
    R, t, n = L.R, L.t.copy(), L.n
    rows = len(R)
    if not math.isfinite(t[0]):
        t[0] = 0.0
    M = np.empty((rows, 2))
    M[:, 0] = t / n
    for i in range(rows - 1):
        M[i, 1] = (n[i + 1] - n[i]) / R[i + 1]
    if t[-1] == 0.0 or not math.isfinite(t[-1]):
        M = M[:-1, :].copy()
    else:
        M[-1, 1] = 0.0
    return Lens(M, n.copy())


class ParaxialRay:
    """ParaxialRay{T}(ynu, tau, n) -- src/Types.jl:29-51"""

    def __init__(self, ynu, tau, n, fundamental):
        ynu = np.array(ynu, dtype=np.float64)
        y, nu = ynu[:, 0].copy(), ynu[:, 1].copy()
        n_ext = np.append(n, n[-1])
        m = min(len(nu), len(n_ext))
        u = nu[:m] / n_ext[:m]
        mt = min(len(tau), len(n_ext) - 2)
        t = np.asarray(tau[:mt]) * n_ext[:mt]
        if fundamental:
            with np.errstate(divide="ignore", invalid="ignore"):
                t = np.append(t, -y[-2] / u[-2])
        z = np.cumsum(t)
        with np.errstate(divide="ignore", invalid="ignore"):
            z0 = (z.min() - z.max()) * 0.1 if u[0] == 0.0 else -y[1] / u[0]
        self.y, self.n, self.u, self.nu, self.ynu = y, n_ext, u, nu, ynu
        self.yu = np.column_stack([y[:m], u])
        self.z = np.concatenate([[z0], z])


@dataclass
class RealRayData:
    """RealRay{T} (src/Types.jl:53-63)"""
    y: np.ndarray
    u: np.ndarray
    yu: np.ndarray
    n: np.ndarray
    z: np.ndarray
    flags: int = 0


@dataclass
class Pupil:
    D: float
    t: float


@dataclass
class System:
    """System (src/Types.jl:119-139)"""
    f: float
    EBFD: float
    EFFD: float
    N: float
    FOV: float
    stop: int
    EP: Pupil
    XP: Pupil
    marginal: ParaxialRay
    chief: ParaxialRay
    trace: np.ndarray
    H: float
    P1: float
    P2: float
    PN: float
    M: np.ndarray
    lens: Lens
    a: np.ndarray
    layout: Layout


@dataclass
class RayBasis:
    """RayBasis (src/Types.jl:65-71)"""
    marginal: ParaxialRay
    chief: ParaxialRay
    H: float
    a: np.ndarray
    stop: int


@dataclass
class RealRayError:
    """RealRayError (src/Types.jl:184-192)"""
    x: np.ndarray
    y: np.ndarray
    nu: float
    r: np.ndarray
    t: np.ndarray
    H: float
    RMS: float
    stats: Optional[np.ndarray] = field(default=None, repr=False)


# ------------------------------------------------------------------------------------------------
# paraxial path
# ------------------------------------------------------------------------------------------------
def raytrace_paraxial(lens, y, w, a=None, clip=False, backend=None):
    """raytrace(lens::Lens, y, w, a; clip) -- src/RayTracing.jl:127-143.  Scalars -> one
    ParaxialRay{Tangential}; arrays -> (y_table, nu_table, clip_idx) with shape (k+1, N)."""
    if not isinstance(lens, Lens):
        lens = make_lens(lens)                                   # :175-178
    be = _be(backend)
    scalar = np.isscalar(y) and np.isscalar(w)
    y0, w0 = np.atleast_1d(np.asarray(y, dtype=np.float64)), np.atleast_1d(np.asarray(w, dtype=np.float64))
    y0, w0 = np.broadcast_arrays(y0, w0)
    yf, wf, ci, ya, wa = be.paraxial_batch(lens.tau, lens.phi, y0, w0, a=a, clip=clip and a is not None,
                                           arith=_lib.STRICT, table=True)
    if scalar:
        return ParaxialRay(np.column_stack([ya[:, 0], wa[:, 0]]), lens.tau, lens.n, False)
    return ya, wa, ci


def transfer_matrix(lens):
    """TransferMatrix(lens) -- src/TransferMatrix.jl:1-6: M_k * ... * M_1 (left fold); O(k) host."""
    tau, phi = lens.tau, lens.phi
    acc = None
    for i in range(len(tau) - 1, -1, -1):
        Mi = np.array([[1.0, tau[i]], [-phi[i], 1.0 - tau[i] * phi[i]]])
        acc = Mi if acc is None else _mm2(acc, Mi)
    return acc


def _mm2(A, B):
    return np.array([[A[0, 0] * B[0, 0] + A[0, 1] * B[1, 0], A[0, 0] * B[0, 1] + A[0, 1] * B[1, 1]],
                     [A[1, 0] * B[0, 0] + A[1, 1] * B[1, 0], A[1, 0] * B[0, 1] + A[1, 1] * B[1, 1]]])


def _matrix_of(M):
    return M.M if isinstance(M, System) else np.asarray(M, dtype=np.float64)


def transfer(M, v, tau, taup, backend=None):
    """transfer(M | system, v, tau, taup) -- src/TransferMatrix.jl:8-11.  v: [y, nu] or (N, 2)."""
    v = np.asarray(v, dtype=np.float64)
    out = _be(backend).transfer_batch(_matrix_of(M), tau, taup, np.atleast_2d(v))
    return out[0] if v.ndim == 1 else out


def reverse_transfer(M, v, taup, tau, backend=None):
    """reverse_transfer(M | system, v, taup, tau) -- src/TransferMatrix.jl:13-17"""
    v = np.asarray(v, dtype=np.float64)
    out = _be(backend).transfer_batch(_matrix_of(M), tau, taup, np.atleast_2d(v), reverse=True)
    return out[0] if v.ndim == 1 else out


def flatten(M):
    """flatten(M) -- cardinal points, src/TransferMatrix.jl:19-28"""
    M = _matrix_of(M)
    f = -1.0 / M[1, 0]
    EFFD = -M[1, 1] * f
    EBFD = M[0, 0] * f
    return dict(f=f, EFFD=EFFD, EBFD=EBFD, P1=EFFD + f, P2=EBFD - f)


def solve(surfaces, a, h_prime=-0.5, backend=None):
    """solve(surfaces | layout, a, h') -- src/RayTracing.jl:302-335.  The two fundamental paraxial
    rays are traced by the paraxial kernel; the rest is O(k) host algebra."""
    layout = _as_layout(surfaces)
    a = np.asarray(a, dtype=np.float64)
    lens = make_lens(layout)
    tau, phi, n = lens.tau, lens.phi, lens.n
    be = _be(backend)
    # both fundamental rays in one launch: (y, w) = (1, 0) and (0, 1)   :209, :252
    _, _, _, ya, wa = be.paraxial_batch(tau, phi, np.array([1.0, 0.0]), np.array([0.0, 1.0]),
                                        arith=_lib.STRICT, table=True)
    rt = np.column_stack([ya[:, 0], wa[:, 0]])
    rt2 = np.column_stack([ya[:, 1], wa[:, 1]])
    y, w = rt[:, 0], rt[:, 1]
    f = -1.0 / w[-1]                                             # :213
    EBFD = y[-1] * f
    sv = a / y[1:]
    stop = int(np.argmin(sv)) + 1                                # findmin :216
    s = sv[stop - 1]
    mr = rt * s
    wf = mr[-1, 1]
    yf = mr[-1, 0] if wf == 0.0 else 0.0                         # extend :202-206
    mr = np.vstack([mr, [yf, wf]])
    marginal = ParaxialRay(mr, tau, n, True)
    ys_, ynu_s = marginal.y[1:-1], marginal.ynu[1:-1, :]         # trace_chief_ray :246-263
    y_stop = ys_[stop - 1]
    ynu2 = rt2[1:, :]
    y2_stop = ynu2[stop - 1, 0]
    nub = -marginal.nu[-1] * h_prime / ys_[0]
    cr = np.empty_like(marginal.ynu)
    cr[1:-1, :] = nub * (ynu2 - ynu_s * y2_stop / y_stop)
    cr[0, :] = (0.0, nub)
    cr[-1, :] = (h_prime, cr[-2, 1])
    chief = ParaxialRay(cr, tau, n, True)
    yb, nub0, nup = chief.y[1], chief.nu[0], chief.nu[-1]        # _solve :302-323
    ym, ypb = marginal.y[0], chief.y[-2]
    dp = EBFD - f
    d = (h_prime - nup * f - yb) / nub0
    EFFD = d - f
    PN = (n[-1] - n[0]) * f
    EP = Pupil(abs(ym) * 2, -yb / nub0)
    H = nub0 * ym
    XP = Pupil(abs(2 * H / nup), -ypb / nup)
    Nn = abs(f / EP.D)
    FOV = 2 * math.degrees(math.atan(abs(chief.u[0])))
    M = transfer_matrix(lens)
    return System(f, EBFD, EFFD, Nn, FOV, stop, EP, XP, marginal, chief,
                  np.column_stack([marginal.yu, chief.yu]), H, d, dp, PN, M, lens, a, layout)


def raybasis(system, ybar, s):
    """raytrace(system::System, ybar, s) -- finite-conjugate RayBasis, src/RayTracing.jl:180-200"""
    y = system.marginal.y[0]
    EP_O = s - system.EP.t
    nu = -y / EP_O
    nub = ybar / EP_O
    al = y * nu / system.H
    be = y * nub / system.H
    mr = system.marginal.ynu + al * system.chief.ynu
    cr = be * system.chief.ynu
    H = nub * y
    mr[-1, 0] = 0.0
    cr[-1, 0] = -H / mr[-1, 1]
    tau = system.lens.tau
    return RayBasis(ParaxialRay(mr, tau, system.lens.n, True), ParaxialRay(cr, tau, system.lens.n, True),
                    H, system.a, system.stop)


# ------------------------------------------------------------------------------------------------
# real rays
# ------------------------------------------------------------------------------------------------
def _trace2d(layout, y, U, aspheric, backend):
    be = _be(backend)
    layout.upload(be)
    return be.trace2d_batch(np.atleast_1d(y), np.atleast_1d(U), aspheric=aspheric)


def _real_ray(layout, yo, Uo, ts, fl, j):
    yu = np.column_stack([yo[:, j], Uo[:, j]])
    return RealRayData(yu[:, 0].copy(), yu[:, 1].copy(), yu, layout.n.copy(), np.cumsum(ts[:, j]), int(fl[j]))


def raytrace(surfaces, *args, a=None, clip=False, backend=None):
    """The reference's `raytrace` generic, dispatched on the trailing tag like Julia dispatches on type:
       raytrace(lens | surfaces, y, w[, a]; clip)               paraxial          RayTracing.jl:127-143,175-178
       raytrace(surfaces, y, U, RealRay)                        2-D meridional    RayTracing.jl:145-173
       raytrace(surfaces, y, x, U, V, VectorRealRay)            3-D skew          PupilSampling.jl:34-65
       raytrace(system, ybar, s)                                RayBasis          RayTracing.jl:180-200
    y, U, ... may be arrays: the batch is traced in one kernel launch."""
    if isinstance(surfaces, System) and len(args) == 2:
        return raybasis(surfaces, *args)
    if args and args[-1] is RealRay:
        y, U = args[0], args[1]
        layout = _as_layout(surfaces)
        # Layout{Aspheric} method (:171-173) -> K from the layout, atan branch; else asin branch (:162)
        yo, Uo, ts, fl = _trace2d(layout, y, U, layout.aspheric, backend)
        if np.isscalar(y) and np.isscalar(U):
            return _real_ray(layout, yo, Uo, ts, fl, 0)
        return yo, Uo, ts, fl
    if args and args[-1] is VectorRealRay:
        y, x, U, V = args[:4]
        layout = _as_layout(surfaces)
        be = _be(backend)
        layout.upload(be)
        y0, x0, U0, V0 = np.broadcast_arrays(*(np.atleast_1d(np.asarray(q, dtype=np.float64)) for q in (y, x, U, V)))
        xv, yv, k, fl = be.trace3d_rays(y0, x0, np.tan(U0), np.tan(V0), arith=_lib.STRICT)   # tan: :38-39
        if all(np.isscalar(q) for q in (y, x, U, V)):
            return xv[:, 0], yv[:, 0]
        return xv, yv
    if len(args) in (2, 3):
        aa = args[2] if len(args) == 3 else a
        return raytrace_paraxial(surfaces, args[0], args[1], a=aa, clip=clip, backend=backend)
    raise TypeError("raytrace: no method matching the given arguments")


def trace_marginal_ray(surfaces, system, atol=EPS, backend=None):
    """Real marginal ray aimed at the stop edge -- src/RayTracing.jl:223-240.  Each secant step
    traces (y, y + eps) as one 2-ray batch."""
    layout = _as_layout(surfaces)
    stop = system.stop
    y = system.marginal.y[0]
    a_stop = system.a[stop - 1]
    be = _be(backend)
    if hasattr(be, "aim2d"):                       # the reference's secant loop (:229-233) in one launch
        layout.upload(be)
        out, it = be.aim2d([y], [0.0], [a_stop], stop, vary_u=False, mode=0, tol=atol, aspheric=layout.aspheric)
        if it[0] < 0:
            raise RuntimeError("trace_marginal_ray did not converge")
        y = float(out[0])
    for _ in range(100):
        yo, Uo, ts, fl = _trace2d(layout, np.array([y, y + EPS]), np.zeros(2), layout.aspheric, backend)
        d = yo[stop, 0] - a_stop
        if not abs(d) > atol:
            break
        dy = yo[stop, 1] - a_stop
        y -= d * EPS / (dy - d)
    else:
        raise RuntimeError("trace_marginal_ray did not converge")
    ray = _real_ray(layout, yo, Uo, ts, fl, 0)
    z = ray.z.copy()
    z[-1] = z[-2] - ray.y[-1] / math.tan(ray.u[-1])              # :234
    z = np.concatenate([[(z.min() - z.max()) * 0.1], z])         # :235
    yv, uv = np.append(ray.y, 0.0), np.append(ray.u, ray.u[-1])
    return RealRayData(yv, uv, np.vstack([ray.yu, [0.0, ray.u[-1]]]), ray.n, z)


def trace_chief_ray(surfaces, system, atol=EPS, backend=None):
    """Real chief ray through the stop centre, traced backwards -- src/RayTracing.jl:265-296.
    `surfaces isa Layout` (:272-277) makes the reversed system a Layout{Aspheric} whose K is
    reverse(K) -- shifted one row against rev_R -- exactly as the reference does."""
    is_layout = isinstance(surfaces, Layout)
    L = _as_layout(surfaces)
    rows = len(L)
    rev_R = -np.concatenate([[np.inf], L.R[:0:-1]])
    rev_t = L.t[::-1].copy()
    rev_n = L.n[::-1].copy()
    m = system.marginal
    rev_t[0] = m.z[-1] - m.z[-2]
    rev = Layout(np.column_stack([rev_R, rev_t, rev_n]), K=L.K[::-1].copy() if is_layout else None,
                 aspheric=is_layout, p=None if (L.P is None or not is_layout) else list(L.P[::-1]))   # reverse(p) :274
    stop = rows - system.stop
    ybp = system.chief.y[-1]
    ubp = -system.chief.u[-1]
    be = _be(backend)
    if hasattr(be, "aim2d"):                       # the reference's secant loop on U (:282-286) in one launch
        rev.upload(be)
        out, it = be.aim2d([ubp], [ybp], [0.0], stop, vary_u=True, mode=0, tol=atol, aspheric=rev.aspheric)
        if it[0] < 0:
            raise RuntimeError("trace_chief_ray did not converge")
        ubp = float(out[0])
    for _ in range(100):
        yo, Uo, ts, fl = _trace2d(rev, np.array([ybp, ybp]), np.array([ubp, ubp + EPS]), rev.aspheric, backend)
        ys = yo[stop, 0]
        if not abs(ys) > atol:
            break
        ubp -= ys * EPS / (yo[stop, 1] - ys)
    else:
        raise RuntimeError("trace_chief_ray did not converge")
    ray = _real_ray(rev, yo, Uo, ts, fl, 0)
    yb = np.concatenate([[0.0], ray.y[::-1]])
    yb[-1] = ybp
    ub = np.concatenate([-ray.u[::-1], [-ray.u[0]]])
    z = ray.z[-1] - ray.z[::-1]
    z[0] = -yb[1] / math.tan(ub[0]) + z[1]                       # EP distance from vertex :293
    z = np.append(z, z[-1] - yb[-2] / math.tan(ub[-2]))
    return RealRayData(yb, ub, np.column_stack([yb, ub]), L.n.copy(), z)


def aim_rays(surfaces, y_start, U, target, stop, scale, backend=None):
    """Entrance heights y (array) such that the meridional ray (y, U) crosses surface `stop` at height
    `target`: secant iteration, every step is one batch of the 2-D kernel over all rays being aimed."""
    layout = _as_layout(surfaces)
    y = np.array(y_start, dtype=np.float64)
    UU = np.broadcast_to(np.asarray(U, dtype=np.float64), y.shape).copy()
    tgt = np.broadcast_to(np.asarray(target, dtype=np.float64), y.shape)
    m = len(y)
    be = _be(backend)
    if hasattr(be, "aim2d"):                       # the whole secant loop runs on the device: one launch
        layout.upload(be)
        out, it = be.aim2d(y, UU, tgt, stop, vary_u=False, mode=1, tol=scale, aspheric=layout.aspheric)
        if np.any(it < 0):
            raise RuntimeError("ray aiming left the domain")
        return out
    fx_prev = None                                 # injected test backends: same iteration, one batch per step
    for _ in range(60):
        h = EPS * np.maximum(1.0, np.abs(y))
        yo, _, _, _ = _trace2d(layout, np.concatenate([y, y + h]), np.concatenate([UU, UU]), layout.aspheric, backend)
        fx = yo[stop, :m] - tgt
        fh = yo[stop, m:] - tgt
        if not np.all(np.isfinite(fx)):
            raise RuntimeError("ray aiming left the domain")
        done = np.abs(fx) <= 4e-16 * scale
        if fx_prev is not None:
            done |= (np.abs(fx) >= np.abs(fx_prev)) & (np.abs(fx_prev) <= 1e-13 * scale)
        if np.all(done):
            break
        y = np.where(done, y, y - fx * h / (fh - fx))
        fx_prev = fx
    return y


def trace_edge_rays(surfaces, y1, y2, U, stop, a_stop, backend=None):
    """src/PupilSampling.jl:67-83.  The reference minimises |y_stop -/+ a_stop| with Optim.BFGS; the
    same two roots are found here by a secant iteration (2-ray batches).  U may be an array of
    field angles: all fields are aimed together."""
    U = np.atleast_1d(np.asarray(U, dtype=np.float64))
    nf = len(U)
    y0 = np.concatenate([np.broadcast_to(y1, nf), np.broadcast_to(y2, nf)]).astype(np.float64)
    tgt = np.concatenate([np.full(nf, a_stop), np.full(nf, -a_stop)])
    y = aim_rays(surfaces, y0, np.concatenate([U, U]), tgt, stop, a_stop, backend=backend)
    return y[:nf], y[nf:]


def _full_trace_setup(surfaces, system, H, k_rays, focus, backend):
    """Host prelude of full_trace, src/PupilSampling.jl:85-122, vectorised over field points H."""
    layout = _as_layout(surfaces)
    Hs = np.abs(np.atleast_1d(np.asarray(H, dtype=np.float64)))
    if not np.all(Hs <= 1.0):
        raise ValueError("DomainError: Domain: |H| <= 1.0")                      # :89
    if focus is None:
        focus = system.marginal.z[-1] - system.marginal.z[-2]                    # :87
    stop = system.stop
    a_stop = abs(system.a[stop - 1])
    be = _be(backend)
    P_ext = None if layout.P is None else np.vstack([layout.P, np.zeros((1, layout.P.shape[1]))])   # fill_poly row of the image plane
    if isinstance(system, System) and hasattr(be, "aim_fields") and layout.P is None:
        # the whole prelude (:90-108) for all fields in one call: first-order solve, reversed real chief ray, real
        # marginal ray and both edge rays per field on the device (k_aim_candidates, one thread per field).  Used only
        # when it reproduces the System it was handed (same stop, focal length and marginal nu, bit for bit).
        rec = be.aim_fields(layout.M3, layout.K, system.a, float(system.chief.y[-1]), Hs, aspheric=layout.aspheric)
        if (np.all(rec[:, 11] == 0.0) and int(rec[0, 6]) == stop and rec[0, 10] == system.f
                and rec[0, 12] == system.marginal.nu[-1]):
            ext = np.vstack([layout.M3, [np.inf, 0.0, 1.0]])                     # :111
            Kx = np.append(layout.K, 0.0)                                        # :112
            ext[-2, 1] = focus                                                   # :114
            return dict(ext=ext, K=Kx, Hs=Hs, U=rec[:, 13].copy(), u=rec[:, 3].copy(), y1=rec[:, 0].copy(),
                        y2=rec[:, 1].copy(), y_EP=float(rec[0, 2]), EP_t=float(rec[0, 8]), h_prime=rec[:, 4].copy(),
                        stop=stop, a_stop=a_stop, focus=focus, z0=None, ybar=None, k_rays=k_rays,
                        nu=system.marginal.nu[-1], P=None)
    # full_trace is reached with surfaces::Layout (:85), so trace_chief_ray takes its Layout branch
    real_chief = trace_chief_ray(layout, system, backend=backend)
    real_marginal = trace_marginal_ray(layout, system, backend=backend)
    EP_t = real_chief.z[0]
    Ubar = real_chief.u[0]
    U = Hs * Ubar
    u = np.array([math.tan(x) for x in U])         # the C library's tan, as everywhere else here: numpy's vectorised
                                                   # tan can round differently in the last bit
    y_EP = abs(real_marginal.y[0])
    y1, y2 = y_EP - u * EP_t, -y_EP - u * EP_t                                   # :99
    y1, y2 = trace_edge_rays(layout, y1, y2, U, stop, a_stop, backend=backend)   # :100
    rb = isinstance(system, RayBasis)
    if not rb:
        h_prime = u * system.f                                                   # :103
        z0 = ybar = None
    else:
        h_prime = np.full(len(Hs), system.chief.y[-1])                           # :105-108
        z0 = system.marginal.z[0]
        ybar = system.chief.y[1] + system.chief.u[0] * z0
    ext = np.vstack([layout.M3, [np.inf, 0.0, 1.0]])                             # :111
    Kx = np.append(layout.K, 0.0)                                                # :112
    ext[-2, 1] = focus                                                           # :114
    return dict(ext=ext, K=Kx, Hs=Hs, U=U, u=u, y1=y1, y2=y2, y_EP=y_EP, EP_t=EP_t, h_prime=h_prime,
                stop=stop, a_stop=a_stop, focus=focus, z0=z0, ybar=ybar, k_rays=k_rays,
                nu=system.marginal.nu[-1], P=P_ext)


def _sweep_inputs(p, k_rays):
    """the pupil grid (xs, one ys per field) and the field records of a sweep from _full_trace_setup's prelude"""
    k2 = k_rays // 2                                                             # :116
    xs = jl_range(0.0, p["y_EP"], k2)                                            # :122
    ys = np.stack([jl_range(p["y1"][j], p["y2"][j], k_rays) for j in range(len(p["Hs"]))])      # :121
    if p["z0"] is None:
        flds = [dict(mode=0, u=float(p["u"][j]), v=math.tan(0.0), h_prime=float(p["h_prime"][j]))
                for j in range(len(p["Hs"]))]
    else:
        flds = [dict(mode=1, ybar=float(p["ybar"]), z0=float(p["z0"]), h_prime=float(p["h_prime"][j]))
                for j in range(len(p["Hs"]))]
    return xs, ys, flds


def full_trace(*args, backend=None, arith=_lib.FAST):
    """full_trace(system, H[, k_rays, focus]) / full_trace(surfaces, system, H[, k_rays, focus]) /
    full_trace(surfaces, raybasis[, k_rays, focus]) -- src/PupilSampling.jl:85-163.
    Returns RealRayError (one field) exactly as the reference lays it out: mirrored vectors
    x = [ex; -ex], y = [ey; ey], r = [r; r] / max(r), t = [theta; pi - theta], RMS = sigma(x, y)."""
    if isinstance(args[0], System):
        system, rest = args[0], args[1:]
        surfaces = system.layout
    else:
        surfaces, system, rest = args[0], args[1], args[2:]
    if isinstance(system, RayBasis):
        H, rest = 1.0, rest                                                      # :149-152
    else:
        H, rest = rest[0], rest[1:]
    k_rays = int(rest[0]) if len(rest) > 0 else SPOT_RAYS
    focus = rest[1] if len(rest) > 1 else None
    if not np.isscalar(H):
        raise TypeError("full_trace takes one field point H; use full_trace_fields for a sweep")
    return full_trace_fields(surfaces, system, [float(H)], k_rays, focus, backend=backend, arith=arith)[0]


def full_trace_fields(surfaces, system, Hs, k_rays=SPOT_RAYS, focus=None, backend=None, arith=_lib.FAST):
    """All field points of a spot-diagram sweep in ONE device call (fields are a grid dimension of the
    kernel).  Each field has its own aimed y-range (:99-100), so every field gets its own ys."""
    be = _be(backend)
    p = _full_trace_setup(surfaces, system, Hs, k_rays, focus, backend)
    be.set_layout(p["ext"], p["K"])
    if p["P"] is not None:
        be.set_polynomials(p["P"])
    xs, ys, flds = _sweep_inputs(p, k_rays)
    out = []
    for j0 in range(0, len(flds), _lib.MAX_FIELDS):
        sl = slice(j0, j0 + _lib.MAX_FIELDS)
        r = be.trace3d_grid(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], arith=arith, compact=True,
                            want=("ex", "ey", "r", "theta", "mask", "stats"))
        out += [_mirror(r, j, p["nu"], float(H)) for j, H in enumerate(p["Hs"][sl])]
    return out


@dataclass
class ThroughFocus:
    """EXTENSION (no reference type): the spot of one field point through focus.  foci are image-plane distances from
    the last lens vertex, full_trace's `focus` (src/PupilSampling.jl:85,111-114); rms[j] is the RealRayError RMS of
    full_trace(..., focus = foci[j]).  The kept set is the same at every focus, so the mirrored sigma^2 is exactly
    quadratic in the focus: best_focus / best_rms are the vertex of its least-squares parabola over all foci (NaN with
    fewer than 3 distinct foci or a parabola that does not open upwards); bracketed: min(foci) <= best_focus <= max(foci)."""
    H: float
    foci: np.ndarray
    rms: np.ndarray
    n_kept: int
    stats: np.ndarray = field(repr=False)
    best_focus: float
    best_rms: float
    bracketed: bool
    spots: Optional[list] = field(default=None, repr=False)    # per focus (x, y), mirrored as in RealRayError


def best_focus_fit(foci, rms):
    """vertex of the least-squares parabola sigma^2 = A d^2 + B d + C, d = f - mean(foci) -> (best_focus, best_rms)"""
    f = np.asarray(foci, dtype=np.float64)
    s2 = np.asarray(rms, dtype=np.float64) ** 2
    if len(np.unique(f)) < 3 or not np.all(np.isfinite(s2)):
        return float("nan"), float("nan")
    fm = float(f.mean())
    d = f - fm
    (A, B, Cc), *_ = np.linalg.lstsq(np.column_stack([d * d, d, np.ones_like(d)]), s2, rcond=None)
    if not A > 0.0:
        return float("nan"), float("nan")
    return fm - B / (2.0 * A), math.sqrt(max(Cc - B * B / (4.0 * A), 0.0))


def through_focus(surfaces, system, Hs, foci, k_rays=SPOT_RAYS, spots=False, backend=None, arith=_lib.FAST):
    """EXTENSION: full_trace's spot at every focus of `foci` for every field point of Hs, each pupil grid traced once
    (ort_trace3d_focus: one device call for all fields and foci, chunked by MAX_FIELDS) -> list of ThroughFocus.
    Equivalent to full_trace_fields(surfaces, system, Hs, k_rays, focus=f) at each f, except that a ray whose image
    position is NaN at one focus is dropped at all of them (only a ray with k3 = 0 after the last surface can be)."""
    be = _be(backend)
    layout = _as_layout(surfaces)
    if layout.P is not None:
        raise NotImplementedError("through_focus: polynomial terms are not supported (ort_trace3d_focus rejects them)")
    foci = np.atleast_1d(np.asarray(foci, dtype=np.float64))
    if foci.ndim != 1 or not 1 <= len(foci) <= _lib.MAX_FOCI:
        raise ValueError(f"through_focus: between 1 and {_lib.MAX_FOCI} foci")
    if not np.all(np.isfinite(foci)):
        raise ValueError("through_focus: foci must be finite")
    p = _full_trace_setup(layout, system, Hs, k_rays, None, backend)
    be.set_layout(p["ext"], p["K"])
    xs, ys, flds = _sweep_inputs(p, k_rays)
    want = ("ex", "ey", "stats") if spots else ("stats",)
    out = []
    for j0 in range(0, len(flds), _lib.MAX_FIELDS):
        sl = slice(j0, j0 + _lib.MAX_FIELDS)
        r = be.trace3d_focus(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], foci, arith=arith, compact=spots,
                            want=want)            # statistics only: no compaction, two launches
        for j, H in enumerate(p["Hs"][sl]):
            st = r["stats"][j].copy()
            rms = np.array([rms_from_stats(st[m]) for m in range(len(foci))])
            n = int(st[0]["n_kept"])
            bf, br = best_focus_fit(foci, rms)
            sp = None
            if spots:
                sp = [(np.concatenate([r["ex"][j][m][:n], -r["ex"][j][m][:n]]), np.concatenate([r["ey"][j][m][:n]] * 2))
                      for m in range(len(foci))]
            out.append(ThroughFocus(float(H), foci.copy(), rms, n, st, bf, br,
                                    bool(foci.min() <= bf <= foci.max()), sp))
    return out


@dataclass
class EncircledEnergy:
    """EXTENSION (no reference type): geometric encircled (metric "circle") or ensquared ("square") energy of the spot of
    one field point, the figures a spot_diagram summarises.  Row j is the image plane foci[j] (one row, full_trace's
    focus, for a grid sweep).  fraction[j][k] is the share of the mirrored spot within radii[k] of the centre (NaN when no
    ray is kept); radius[j][i] the smallest radius that holds fractions[i] of it, an exact element of the ray distances
    (NaN when no ray is kept).  Centre and distance as in include/ort_b200.h (ort_spot_energy_dev)."""
    H: float
    foci: np.ndarray
    radii: np.ndarray
    fraction: np.ndarray
    fractions: np.ndarray
    radius: np.ndarray
    n_kept: int
    stats: np.ndarray = field(repr=False)


def encircled_energy(surfaces, system, Hs, radii=None, fractions=(0.5, 0.8, 0.9), k_rays=SPOT_RAYS, focus=None, foci=None,
                     metric="circle", center="centroid", backend=None, arith=_lib.FAST):
    """EXTENSION: encircled (or ensquared) energy of full_trace's spot for every field point of Hs -> list of
    EncircledEnergy.  The pupil grid is swept on the device -- at `focus` (full_trace's, default the paraxial one), or
    with `foci` at up to MAX_FOCI image planes in one pass as through_focus does -- and the curve over `radii` and the
    energy radii of `fractions` are computed there (ort_trace3d_energy); only those numbers cross PCIe.
    center "centroid" measures from the centroid of the mirrored spot, (0, mean y); "paraxial" from (0, h')."""
    be = _be(backend)
    layout = _as_layout(surfaces)
    r = np.empty(0) if radii is None else np.atleast_1d(np.asarray(radii, dtype=np.float64))
    q = np.empty(0) if fractions is None else np.atleast_1d(np.asarray(fractions, dtype=np.float64))
    if r.ndim != 1 or len(r) > _lib.MAX_RADII or not np.all(np.isfinite(r)) or np.any(r < 0) or np.any(np.diff(r) <= 0):
        raise ValueError(f"encircled_energy: radii must be finite, >= 0 and strictly ascending, at most {_lib.MAX_RADII}")
    if q.ndim != 1 or len(q) > _lib.MAX_FRACS or not np.all((q > 0) & (q <= 1)):
        raise ValueError(f"encircled_energy: fractions must lie in (0, 1], at most {_lib.MAX_FRACS}")
    if not len(r) and not len(q):
        raise ValueError("encircled_energy: neither radii nor fractions")
    if metric not in ("circle", "square") or center not in ("centroid", "paraxial"):
        raise ValueError("encircled_energy: metric is 'circle' or 'square', center 'centroid' or 'paraxial'")
    if foci is not None:
        if focus is not None:
            raise ValueError("encircled_energy: give focus or foci, not both")
        if layout.P is not None:
            raise NotImplementedError("encircled_energy: polynomial terms are not supported through focus")
        foci = np.atleast_1d(np.asarray(foci, dtype=np.float64))
        if foci.ndim != 1 or not 1 <= len(foci) <= _lib.MAX_FOCI or not np.all(np.isfinite(foci)):
            raise ValueError(f"encircled_energy: between 1 and {_lib.MAX_FOCI} finite foci")
    p = _full_trace_setup(layout, system, Hs, k_rays, focus, backend)
    be.set_layout(p["ext"], p["K"])
    if p["P"] is not None:
        be.set_polynomials(p["P"])
    xs, ys, flds = _sweep_inputs(p, k_rays)
    fo = np.array([float(p["focus"])]) if foci is None else foci
    out = []
    for j0 in range(0, len(flds), _lib.MAX_FIELDS):
        sl = slice(j0, j0 + _lib.MAX_FIELDS)
        e = be.trace3d_energy(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], radii=r, fracs=q, foci=foci, arith=arith,
                              metric=metric, center=center)
        for j, H in enumerate(p["Hs"][sl]):
            st = e["stats"][j].reshape(-1).copy()
            cnt = e["counts"][j].reshape(len(fo), len(r))
            n = int(st[0]["n_kept"])
            frac = cnt / n if n else np.full(cnt.shape, np.nan)
            out.append(EncircledEnergy(float(H), fo.copy(), r.copy(), frac, q.copy(),
                                       e["radius"][j].reshape(len(fo), len(q)).copy(), n, st))
    return out


def _mirror(r, f, nu, H):
    """take advantage of symmetry -- src/PupilSampling.jl:139-146; RMS = sigma(:169-173) evaluated
    from the kernel's mergeable moments (mirrored x has mean exactly 0)."""
    st = r["stats"][f]
    n = int(st["n_kept"])
    ex, ey, rr, th = (r[k][f][:n] for k in ("ex", "ey", "r", "theta"))
    x2 = np.concatenate([ex, -ex])
    y2 = np.concatenate([ey, ey])
    # r_max is the correctly rounded sqrt of the largest r^2 while FAST r values carry ~1 ulp: clamp so max(rho) == 1 (:142)
    rho = np.minimum(rr / st["r_max"], 1.0) if n else rr
    rho2 = np.concatenate([rho, rho])
    t2 = np.concatenate([th, math.pi - th])
    return RealRayError(x2, y2, nu, rho2, t2, H, rms_from_stats(st), stats=r["stats"][f:f + 1].copy())


def rms_from_stats(st):
    """sigma of the mirrored spot (src/PupilSampling.jl:140-141,169-173) from (n, mean, M2):
    x -> [x; -x] has mean 0 and sum of squares 2 (M2x + n mean_x^2); y -> [y; y] doubles M2y."""
    n = float(st["n_kept"])
    if n == 0:
        return float("nan")
    sxx = float(st["m2_x"]) + n * float(st["mean_x"]) ** 2
    return math.sqrt((2.0 * sxx + 2.0 * float(st["m2_y"])) / (2.0 * n))


def merge_stats(records):
    """Chan merge of per-shard ort_stats records in the given (rank) order: the multi-GPU combine
    step after the all-gather.  records: structured array (n_shards,) -> one record."""
    out = np.zeros(1, dtype=_lib.STATS_DTYPE)[0]
    out["r_max"] = -np.inf
    for rec in records:
        for k in ("n_miss", "n_tir", "n_domain", "n_clip", "n_vig", "n_strict"):
            out[k] += rec[k]
        nb = float(rec["n_kept"])
        if nb == 0:
            continue
        na = float(out["n_kept"])
        if na == 0:
            for k in ("n_kept", "mean_x", "mean_y", "m2_x", "m2_y", "r_max", "mean_opd", "m2_opd"):
                out[k] = rec[k]
            continue
        n = na + nb
        w = nb / n
        for mk, vk in (("mean_x", "m2_x"), ("mean_y", "m2_y"), ("mean_opd", "m2_opd")):
            d = float(rec[mk]) - float(out[mk])
            out[mk] = float(out[mk]) + d * w
            out[vk] = float(out[vk]) + float(rec[vk]) + d * d * (na * w)
        out["n_kept"] += rec["n_kept"]
        out["r_max"] = max(float(out["r_max"]), float(rec["r_max"]))
    return out


@dataclass
class Wavefront:
    """EXTENSION (SURVEY.md section 8 f4; no reference counterpart): ray-traced optical path difference over the
    pupil grid of full_trace, referred to the chief ray on a reference sphere centred at the chief ray's image
    point with its centre of curvature distance = image plane - paraxial exit pupil."""
    opd: np.ndarray          # waves, kept rays in push! order, mirrored like RealRayError ([opd; opd])
    x: np.ndarray            # transverse errors of the same rays (mirrored)
    y: np.ndarray
    H: float
    rms: float               # RMS OPD about its mean, waves
    mean: float
    pv: float
    stats: np.ndarray = field(default=None, repr=False)


def wavefront(surfaces, system, Hs, k_rays=SPOT_RAYS, focus=None, lam=LAMBDA, vignette=False, backend=None,
              arith=_lib.FAST):
    """OPD map per field point (list of Wavefront).  W = (OPL_chief - OPL_ray) / lam -- the sign convention of
    the reference's Seidel wavefront W(rho, theta, H) (src/SeidelAberrations.jl:61-76), so that the rho^4 term
    of the on-axis map reproduces its W040 -- with the OPL accumulated surface by surface inside the grid
    kernel and closed on the reference sphere."""
    be = _be(backend)
    p, xs, ys, flds, ext = _wavefront_setup(surfaces, system, Hs, k_rays, focus, vignette, backend, "wavefront")
    nf = len(flds)
    out = []
    for j0 in range(0, nf, _lib.MAX_FIELDS):
        sl = slice(j0, j0 + _lib.MAX_FIELDS)
        r = be.trace3d_grid(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], arith=arith, compact=True,
                            want=("ex", "ey", "opd", "mask", "stats"), ext=ext, opd_scale=-1.0 / lam)
        for j, H in enumerate(p["Hs"][sl]):
            st = r["stats"][j]
            n = int(st["n_kept"])
            o = r["opd"][j][:n]
            ex, ey = r["ex"][j][:n], r["ey"][j][:n]
            out.append(Wavefront(np.concatenate([o, o]), np.concatenate([ex, -ex]), np.concatenate([ey, ey]), float(H),
                                 math.sqrt(st["m2_opd"] / n) if n else float("nan"), float(st["mean_opd"]),
                                 float(o.max() - o.min()) if n else float("nan"), stats=r["stats"][j:j + 1].copy()))
    be.set_apertures(None)
    return out


def _wavefront_setup(surfaces, system, Hs, k_rays, focus, vignette, backend, caller):
    """The OPD sweep of wavefront() and zernike(): full_trace's prelude, the chief ray of every field through the centre
    of the stop, the reference sphere (centred on the chief ray's image point, radius = image plane - paraxial exit
    pupil) and the field records that close the OPL on it.  Leaves the extended layout (image plane in the last medium),
    polynomial terms and apertures (vignette) set on the backend -> (p, xs, ys, field records, opts.ext bits)."""
    be = _be(backend)
    layout = _as_layout(surfaces)
    p = _full_trace_setup(layout, system, Hs, k_rays, focus, backend)
    if p["z0"] is not None:
        raise NotImplementedError(f"{caller}: RayBasis (finite object) reference wavefront not implemented")
    ext = p["ext"].copy()
    ext[-1, 2] = layout.n[-1]                     # the image plane sits in the last medium (no fake refraction)
    nf = len(p["Hs"])
    # chief ray of every field: through the centre of the stop (aiming uses the 2-D kernel on the bare layout)
    y_c = aim_rays(layout, -p["u"] * p["EP_t"], p["U"], np.zeros(nf), p["stop"], p["a_stop"], backend=backend)
    be.set_layout(ext, p["K"])
    if p["P"] is not None:
        be.set_polynomials(p["P"])
    be.set_apertures(system.a if vignette else None)
    xv, yv, k, fl, opl = be.trace3d_rays(y_c, np.zeros(nf), p["u"], np.zeros(nf), arith=_lib.STRICT, opl=True)
    n0, nl = layout.n[0], layout.n[-1]
    knorm = 1.0 / np.sqrt(p["u"] ** 2 + 1.0)                 # k = normalize([0, u, 1])
    opl0 = n0 * (y_c * (p["u"] * knorm))                     # start term of the chief ray
    Rr = p["focus"] - system.XP.t                            # image plane - paraxial exit pupil
    yc = yv[-1]
    opl_ref = opl + opl0 + nl * (-Rr)
    xs = jl_range(0.0, p["y_EP"], k_rays // 2)
    ys = np.stack([jl_range(p["y1"][j], p["y2"][j], k_rays) for j in range(nf)])
    flds = [dict(mode=0, u=float(p["u"][j]), v=0.0, h_prime=float(p["h_prime"][j]), opd_xc=0.0, opd_yc=float(yc[j]),
                 opd_radius=float(Rr), opl_ref=float(opl_ref[j])) for j in range(nf)]
    return p, xs, ys, flds, _lib.EXT_OPD | (_lib.EXT_VIGNETTE if vignette else 0)


@dataclass
class ZernikeFit:
    """EXTENSION (no reference type): Zernike decomposition of the wavefront of one field point -- the OPD map that
    wavefront() returns, in waves -- over ANSI Z80.28 / OSA terms j = (n(n+2) + m)/2, n <= n_max, each of unit RMS over
    the unit disk (include/ort_b200.h, ort_wavefront_zernike_dev).  coef[j] multiplies Z_j with index n[j], m[j];
    the fit is that of the mirrored map, so the terms antisymmetric in x (sin m theta for even m, cos m theta for odd m)
    are exactly 0.  rms_resid / pv_resid: RMS and PV of the map minus the fit.  status 0 ok, 1 fewer kept rays than
    fitted terms, 2 singular normal matrix, 3 a non-finite OPD (coef and residuals NaN for status != 0)."""
    H: float
    n_max: int
    n: np.ndarray
    m: np.ndarray
    coef: np.ndarray
    rms_resid: float
    pv_resid: float
    status: int
    n_kept: int
    stats: np.ndarray = field(repr=False)


def zernike_indices(n_max):
    """(n, m) of the ANSI single index j = 0 .. (n_max + 1)(n_max + 2)/2 - 1"""
    nm = [(n, m) for n in range(n_max + 1) for m in range(-n, n + 1, 2)]
    return np.array([a for a, _ in nm], dtype=np.int64), np.array([b for _, b in nm], dtype=np.int64)


def zernike(surfaces, system, Hs, n_max=8, k_rays=SPOT_RAYS, focus=None, lam=LAMBDA, vignette=False, norm="stop",
            backend=None, arith=_lib.FAST):
    """EXTENSION: Zernike coefficients (waves) of the wavefront of every field point of Hs -> list of ZernikeFit.  The
    OPD sweep of wavefront() runs full grid on the device and the least-squares fit is made there
    (ort_trace3d_zernike); only n_max-many coefficients per field cross PCIe.  norm "stop": rho = r / a_stop, the stop
    rim is the unit circle; "rmax": rho = r / max(r) of the field's kept rays, the reference's RealRayError.r."""
    if not (isinstance(n_max, (int, np.integer)) and 0 <= n_max <= _lib.ZERN_MAX_ORDER):
        raise ValueError(f"zernike: n_max must be an integer in [0, {_lib.ZERN_MAX_ORDER}]")
    if norm not in ("stop", "rmax"):
        raise ValueError("zernike: norm is 'stop' or 'rmax'")
    be = _be(backend)
    p, xs, ys, flds, ext = _wavefront_setup(surfaces, system, Hs, k_rays, focus, vignette, backend, "zernike")
    r_norm = p["a_stop"] if norm == "stop" else 0.0
    ni, mi = zernike_indices(int(n_max))
    out = []
    for j0 in range(0, len(flds), _lib.MAX_FIELDS):
        sl = slice(j0, j0 + _lib.MAX_FIELDS)
        z = be.trace3d_zernike(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], int(n_max), r_norm, arith=arith, ext=ext,
                               opd_scale=-1.0 / lam)
        for j, H in enumerate(p["Hs"][sl]):
            out.append(ZernikeFit(float(H), int(n_max), ni.copy(), mi.copy(), z["coef"][j].copy(), float(z["resid"][j][0]),
                                  float(z["resid"][j][1]), int(z["status"][j]), int(z["stats"][j]["n_kept"]),
                                  z["stats"][j:j + 1].copy()))
    be.set_apertures(None)
    return out


@dataclass
class PSF:
    """EXTENSION (no reference type): diffraction point-spread function of one field point -- the scalar Fraunhofer PSF of
    the mirrored pupil that wavefront() returns, pupil height h mapped to the image-space direction sine h / f
    (include/ort_b200.h, ort_wavefront_psf_dev).  u, v: pixel centres in mm from the chief ray's image point, u along x
    (sagittal), v along y; psf[iv, iu], 1 = the diffraction-limited peak of the same (possibly vignetted) pupil.
    strehl: psf at the chief ray's image point, |mean(exp(2 pi i W))|^2; peak: the maximum of psf over the grid, at
    peak_uv.  status 0 ok, 1 no kept ray, 3 a non-finite OPD (psf, strehl and peak NaN for status != 0)."""
    H: float
    u: np.ndarray
    v: np.ndarray
    psf: np.ndarray
    strehl: float
    peak: float
    peak_uv: tuple
    status: int
    n_kept: int
    stats: np.ndarray = field(repr=False)


def _pair(x, name, kind):
    t = tuple(x) if isinstance(x, (tuple, list, np.ndarray)) else (x, x)
    if len(t) != 2:
        raise ValueError(f"psf: {name} is one value or a pair (along x, along y)")
    return tuple(kind(a) for a in t)


def psf(surfaces, system, Hs, n_pix=None, pixel=None, k_rays=SPOT_RAYS, focus=None, lam=LAMBDA, vignette=False,
        backend=None, arith=_lib.FAST):
    """EXTENSION: diffraction PSF and Strehl ratio of every field point of Hs -> list of PSF.  The OPD sweep of
    wavefront() runs full grid on the device and the PSF is computed there (ort_trace3d_psf): a matrix Fourier transform
    of exp(2 pi i W) over the traced pupil grid with s = 1 / (lam f).  Only the pixel grid crosses PCIe.
    n_pix: pixels per side, an int or (n_u, n_v), default k_rays - 1 (odd: the chief ray's image point is a pixel);
    pixel: pitch in mm, a value or (du, dv), default lam F# / 2 = 1 / (4 s y_EP).  Raises ValueError when the pixel grid
    is longer than the alias period 1 / (s dx) or 1 / (s dy) of the pupil grid."""
    if not (isinstance(k_rays, (int, np.integer)) and k_rays >= 2):
        raise ValueError("psf: k_rays must be an integer >= 2")
    n_u, n_v = _pair(k_rays - 1 if n_pix is None else n_pix, "n_pix", int)
    if not (1 <= n_u <= _lib.PSF_MAX_SIDE and 1 <= n_v <= _lib.PSF_MAX_SIDE):
        raise ValueError(f"psf: n_pix must lie in [1, {_lib.PSF_MAX_SIDE}]")
    if pixel is not None:
        du, dv = _pair(pixel, "pixel", float)
        if not (math.isfinite(du) and math.isfinite(dv) and du > 0 and dv > 0):
            raise ValueError("psf: pixel must be finite and > 0")
    be = _be(backend)
    p, xs, ys, flds, ext = _wavefront_setup(surfaces, system, Hs, k_rays, focus, vignette, backend, "psf")
    try:
        scale = 1.0 / (lam * system.f)
        if not (math.isfinite(scale) and scale > 0):
            raise ValueError("psf: 1 / (lam f) must be finite and > 0")
        if pixel is None:
            du = dv = 1.0 / (4.0 * scale * p["y_EP"])
        # the grid must not wrap: n du <= 1 / (s dx), the alias period of the pupil step dx (1e-9: equality is allowed)
        dx = abs(xs[1] - xs[0]) if len(xs) > 1 else 0.0
        dy = float(np.max(np.abs(ys[:, 1] - ys[:, 0]))) if ys.shape[1] > 1 else 0.0
        if n_u * du * scale * dx > 1 + 1e-9 or n_v * dv * scale * dy > 1 + 1e-9:
            span = float(np.max(np.abs(ys[:, -1] - ys[:, 0])))
            k_fit = max(2 * (math.ceil(n_u * du * scale * p["y_EP"]) + 1), math.ceil(n_v * dv * scale * span) + 1)
            raise ValueError(f"psf: {n_u} x {n_v} pixels of {du:.4g} x {dv:.4g} mm exceed the alias period "
                             f"{1 / (scale * dx) if dx else math.inf:.4g} x {1 / (scale * dy) if dy else math.inf:.4g} mm "
                             f"of k_rays = {k_rays}; k_rays >= {k_fit + (k_fit & 1)} would fit")
        u, v = (np.arange(n_u) - (n_u - 1) / 2) * du, (np.arange(n_v) - (n_v - 1) / 2) * dv
        out = []
        for j0 in range(0, len(flds), _lib.MAX_FIELDS):
            sl = slice(j0, j0 + _lib.MAX_FIELDS)
            r = be.trace3d_psf(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], n_u, n_v, du, dv, scale, arith=arith,
                               ext=ext, opd_scale=-1.0 / lam)
            for j, H in enumerate(p["Hs"][sl]):
                pk = int(r["peak"][j])
                uv = (float(u[pk % n_u]), float(v[pk // n_u])) if pk >= 0 else (math.nan, math.nan)
                out.append(PSF(float(H), u.copy(), v.copy(), r["psf"][j].copy(), float(r["strehl"][j][0]),
                               float(r["strehl"][j][1]), uv, int(r["status"][j]), int(r["stats"][j]["n_kept"]),
                               r["stats"][j:j + 1].copy()))
    finally:
        be.set_apertures(None)
    return out


@dataclass
class MTF:
    """EXTENSION (no reference type): diffraction modulation transfer function of one field point -- the optical transfer
    function of the PSF that psf() computes (scalar Fraunhofer model of the mirrored pupil, s = 1 / (lam f)), along two
    azimuths (include/ort_b200.h, ort_wavefront_mtf_dev).  freqs in cycles/mm; otf[0] sagittal (frequency along x),
    otf[1] tangential (along y), complex, otf(0) = 1; mtf = |otf|, ptf = angle(otf) in radians.  cutoff: the diffraction
    cutoffs (sagittal, tangential) of the sampled pupil, past which otf is 0.  status 0 ok, 1 no kept ray, 3 a non-finite
    OPD, 4 the pupil grid is not a lattice (otf NaN for status != 0)."""
    H: float
    freqs: np.ndarray
    otf: np.ndarray
    mtf: np.ndarray
    ptf: np.ndarray
    cutoff: tuple
    status: int
    n_kept: int
    stats: np.ndarray = field(repr=False)


def mtf(surfaces, system, Hs, freqs=None, k_rays=SPOT_RAYS, focus=None, lam=LAMBDA, vignette=False, backend=None,
        arith=_lib.FAST):
    """EXTENSION: diffraction MTF of every field point of Hs -> list of MTF.  The OPD sweep of wavefront() runs full grid
    on the device and the OTF is computed there (ort_trace3d_mtf) as the autocorrelation of the mirrored pupil function
    exp(2 pi i W) at the lattice lags the frequencies need, interpolated linearly between them.  Only the OTF values cross
    PCIe.  freqs: cycles/mm, finite and >= 0, at most MTF_MAX_FREQS; default 32 evenly spaced from 0 to 1 / (lam F#) =
    2 s y_EP."""
    if not (isinstance(k_rays, (int, np.integer)) and k_rays >= 4):
        raise ValueError("mtf: k_rays must be an integer >= 4")
    if freqs is not None:
        freqs = np.array(freqs, dtype=np.float64).ravel()
        if not (1 <= len(freqs) <= _lib.MTF_MAX_FREQS):
            raise ValueError(f"mtf: 1 to {_lib.MTF_MAX_FREQS} frequencies")
        if not (np.all(np.isfinite(freqs)) and np.all(freqs >= 0)):
            raise ValueError("mtf: frequencies must be finite and >= 0")
    be = _be(backend)
    p, xs, ys, flds, ext = _wavefront_setup(surfaces, system, Hs, k_rays, focus, vignette, backend, "mtf")
    try:
        scale = 1.0 / (lam * system.f)
        if not (math.isfinite(scale) and scale > 0):
            raise ValueError("mtf: 1 / (lam f) must be finite and > 0")
        if freqs is None:
            freqs = np.linspace(0.0, 2.0 * scale * p["y_EP"], 32)
        # the lattice steps of the contract, by index: dx = xs[-1] / (nx - 1), dy = (ys[-1] - ys[0]) / (ny - 1)
        cut_x = 2 * (len(xs) - 1) * (xs[-1] / (len(xs) - 1)) * scale
        out = []
        for j0 in range(0, len(flds), _lib.MAX_FIELDS):
            sl = slice(j0, j0 + _lib.MAX_FIELDS)
            r = be.trace3d_mtf(flds[sl], ys[sl], xs, p["stop"], p["a_stop"], freqs, scale, arith=arith, ext=ext,
                               opd_scale=-1.0 / lam)
            for j, H in enumerate(p["Hs"][sl]):
                y = ys[j0 + j]
                cut_y = (len(y) - 1) * abs((y[-1] - y[0]) / (len(y) - 1)) * scale
                o = r["otf"][j].copy()
                out.append(MTF(float(H), freqs.copy(), o, np.abs(o), np.angle(o), (float(cut_x), float(cut_y)),
                               int(r["status"][j]), int(r["stats"][j]["n_kept"]), r["stats"][j:j + 1].copy()))
    finally:
        be.set_apertures(None)
    return out


# ------------------------------------------------------------------------------------------------
# Seidel aberrations (SURVEY.md section 8 f2): the per-candidate objective of the reference's optimize()
# ------------------------------------------------------------------------------------------------
SEIDEL_FIELDS = ("f", "EBFD", "stop", "H", "W040", "W131", "W222", "W220P", "W311", "W020", "W111", "W220", "W220M",
                 "W220T", "nu_marginal", "nu_chief")
SEIDEL_SURFACE_FIELDS = ("spherical", "coma", "astigmatism", "petzval", "distortion", "axial", "lateral")


@dataclass
class Aberration:
    """Aberration (src/Types.jl:143-167): wave coefficients + per-surface contributions"""
    W040: float
    W131: float
    W222: float
    W220: float
    W311: float
    W020: float
    W111: float
    W220P: float
    W220M: float
    W220T: float
    spherical: np.ndarray
    coma: np.ndarray
    astigmatism: np.ndarray
    sagittal: np.ndarray
    distortion: np.ndarray
    axial: np.ndarray
    lateral: np.ndarray
    petzval: np.ndarray
    medial: np.ndarray
    tangential: np.ndarray
    lam: float
    field_sign: int
    nu: float

    def __call__(self, rho, theta, H):
        """W(rho, theta, H) -- the Seidel wavefront polynomial, src/SeidelAberrations.jl:61-76"""
        H = np.abs(H)
        if np.any(H > 1.0):
            raise ValueError("DomainError: Domain: |H| <= 1.0")
        if np.any((np.asarray(rho) < 0.0) | (np.asarray(rho) > 1.0)):
            raise ValueError("DomainError: Domain: 0.0 <= rho <= 1.0")
        H = H * self.field_sign
        c = np.cos(theta)
        return (self.W040 * rho ** 4 + self.W131 * H * rho ** 3 * c + self.W222 * H ** 2 * rho ** 2 * c ** 2 +
                self.W220 * H ** 2 * rho ** 2 + self.W311 * H ** 3 * rho * c + self.W020 * rho ** 2 + self.W111 * H * rho * c)

    def ray_error(self, x, y, H):
        """transverse ray error polynomials (eps_x, eps_y), src/SeidelAberrations.jl:78-102"""
        if np.any(np.hypot(x, y) > 1.0):
            raise ValueError("DomainError: Domain: hypot(x, y) <= 1.0")
        H = np.abs(H)
        if np.any(H > 1.0):
            raise ValueError("DomainError: Domain: |H| <= 1.0")
        H = H * self.field_sign
        ey = (4 * self.W040 * (x ** 2 * y + y ** 3) + self.W131 * H * (x ** 2 + 3 * y ** 2) + 2 * self.W222 * H ** 2 * y +
              2 * self.W220 * H ** 2 * y + self.W311 * H ** 3 + 2 * self.W020 * y + self.W111 * H) * self.lam / self.nu
        ex = (4 * self.W040 * (y ** 2 * x + x ** 3) + self.W131 * H * (2 * x * y) + 0 + 2 * self.W220 * H ** 2 * x + 0 +
              2 * self.W020 * x + 0) * self.lam / self.nu
        return ex, ey


def aberrations(surfaces, system, lam=LAMBDA, dn=None, backend=None):
    """aberrations(surfaces, system, lambda, dn) -- src/SeidelAberrations.jl:6-53, evaluated by the candidate
    kernel (K7) on a batch of one.  `system` must be solve(surfaces, system.a, system.chief.y[-1])."""
    layout = _as_layout(surfaces)
    RtnK = np.stack([layout.R, layout.t, layout.n, layout.K])[None]
    out, per = _be(backend).seidel_candidates(RtnK, system.a, system.chief.y[-1], lam=lam, dn=dn, per_surface=True)
    o = dict(zip(SEIDEL_FIELDS, out[0]))
    sp, co, ast, ptz, dist, ax, lat = per[0]
    return Aberration(o["W040"], o["W131"], o["W222"], o["W220"], o["W311"], o["W020"], o["W111"], o["W220P"], o["W220M"],
                      o["W220T"], sp, co, ast, ptz + ast / 2, dist, ax, lat, ptz, ptz + ast, ptz + 1.5 * ast, lam,
                      int(np.sign(system.chief.y[-1])), float(system.marginal.nu[-1]))


def seidel_merit(backend, RtnK, a, h_prime, aberr=("W040", "W131", "W222", "W220", "W311"), weights=None, lam=LAMBDA,
                 dn=None):
    """Population evaluation of the reference's optimisation objective, sum_i w_i |W_i| (src/Optimization.jl:40-45,
    without its constraint penalty), for C candidate prescriptions in one launch.  Returns (merit (C,), table (C, 16))."""
    out = _be(backend).seidel_candidates(RtnK, a, h_prime, lam=lam, dn=dn)
    w = np.ones(len(aberr)) if weights is None else np.asarray(weights, dtype=np.float64)
    cols = [SEIDEL_FIELDS.index(k) for k in aberr]
    return np.abs(out[:, cols]) @ w, out


AIM_FIELDS = ("y1", "y2", "y_EP", "u", "h_prime", "focus", "stop", "a_stop", "EP_t", "Ubar", "f", "status", "nu", "U")


def full_trace_candidates(RtnK, a, h_prime, H, k_rays=SPOT_RAYS, aspheric=False, backend=None, arith=_lib.FAST):
    """full_trace(surfaces, system, H, k_rays) (src/PupilSampling.jl:85-147) for a POPULATION of candidate
    prescriptions RtnK[C][4][rows] sharing apertures `a` and image height h' of solve(surfaces, a, h'): every
    candidate gets its own first-order solve, aimed chief / marginal / edge rays (:90-100) and its own pupil grid
    (:121-122), then its own spot statistics -- two launches for the whole population.  This is the real-ray merit
    the reference could only evaluate one `full_trace` at a time.
    Returns (spot (C, 4) = n_kept, mean_x, mean_y, RMS of the unmirrored half pupil, aim (C, 24), see AIM_FIELDS);
    the mirrored RMS of RealRayError is sqrt(RMS^2 + mean_x^2)  (x mirrors to mean 0, :140-141)."""
    if not abs(H) <= 1.0:
        raise ValueError("DomainError: Domain: |H| <= 1.0")                      # :89
    be = _be(backend)
    aim = be.aim_candidates(RtnK, a, h_prime, H, aspheric=aspheric)
    spot = be.trace3d_candidates_aimed(RtnK, aim, int(k_rays), int(k_rays) // 2, arith=arith)
    return spot, aim


@dataclass
class Vignetting:
    """Vignetting (src/Types.jl:169-176); limit / partial / full hold 1-based surface indices like the reference"""
    M: np.ndarray
    FOV: np.ndarray
    un: bool
    limit: np.ndarray
    partial: np.ndarray
    full: np.ndarray


def _isapprox(x, y):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        return (x == y) | (np.isfinite(x) & np.isfinite(y) & (np.abs(x - y) <= EPS * np.maximum(np.abs(x), np.abs(y))))


def vignetting(system, a=None, backend=None):
    """vignetting(system::SystemOrRayBasis, a = system.a) -- src/Vignetting.jl:1-30.  For a System the table comes from
    the candidate kernel (Context.vignetting_candidates, one candidate: the same first-order solve, bit for bit);
    for a RayBasis (whose rays are not a solve() of a prescription) and for injected test backends it is O(k) host
    algebra on the two paraxial rays the object already holds, like the tail of solve()."""
    a = np.asarray(system.a if a is None else a, dtype=np.float64)
    be = _be(backend)                              # no GPU and no injected backend: raises, like every other entry
    if isinstance(system, System) and hasattr(be, "vignetting_candidates"):
        L = system.layout
        RtnK = np.stack([L.R, L.t, L.n, L.K])[None]
        r = be.vignetting_candidates(RtnK, system.a, float(system.chief.y[-1]), a_vig=a)
        code = r["code"][0]
        return Vignetting(r["M"][0], r["FOV"][0], bool(r["un"][0]), np.nonzero(code & 1)[0] + 1,
                          np.nonzero(code & 2)[0] + 1, np.nonzero(code & 4)[0] + 1)
    yb = np.abs(system.chief.y[1:-1])
    y = np.abs(system.marginal.y[1:-1])
    M = np.column_stack([a, y, y + yb, yb, yb - y])
    nanmin = lambda v: np.nan if np.any(np.isnan(v)) else float(np.min(v))       # Julia's minimum propagates NaN
    with np.errstate(invalid="ignore", divide="ignore"):
        M[M[:, 3] < y, 3] = np.nan                                               # :12
        M[M[:, 4] < y, 4] = np.nan                                               # :13
        a_unvig = (a >= M[:, 2]) | _isapprox(a, M[:, 2])                         # :14
        others = np.arange(len(a)) != system.stop - 1
        scales = (nanmin(((a - y) / yb)[others]), nanmin(a / yb), nanmin((a + y) / yb))    # :17-19
        FOV = np.empty((3, 3))
        for i, sc in enumerate(scales):
            ub = abs(system.chief.u[0] * sc)
            FOV[i] = (2 * (math.atan(ub) * (180.0 / math.pi)), ub, abs(system.chief.y[-1] * sc))
        limit = np.nonzero((a < M[:, 1]) & ~_isapprox(a, M[:, 2]))[0] + 1        # :27
        full = np.nonzero(a <= M[:, 4])[0] + 1                                   # :28
        partial = np.setdiff1d(np.nonzero(~a_unvig)[0] + 1, full)                # :29
    return Vignetting(M, FOV, bool(np.all(a_unvig)), limit, partial, full)


def wavegrad(eps, lam=LAMBDA):
    """wavegrad(eps::RealRayError, lambda) -- src/PupilSampling.jl:165-167"""
    return eps.x * eps.nu / lam, eps.y * eps.nu / lam


def TSA(surfaces, system, k_rays=K_RAYS, backend=None):
    """TSA -- transverse spherical aberration fan, src/SeidelAberrations.jl:116-135.  The k_rays-1
    meridional rays are one batch of the 2-D kernel."""
    layout = _as_layout(surfaces)
    pm = system.marginal
    rm = trace_marginal_ray(surfaces, system, backend=backend)
    rc = trace_chief_ray(surfaces, system, backend=backend)
    XP_t = rc.z[-1] - rc.z[-2]
    y_EP = jl_range(rm.y[0] / k_rays, rm.y[0], k_rays)
    y_XP, eps_ = np.empty(k_rays), np.empty(k_rays)
    BFD = pm.z[-1] - pm.z[-2]
    t = BFD - (rm.z[-2] - pm.z[-2])                              # surface_to_focus :105 with sag :93-95
    y_XP[-1] = rm.y[-2] + math.tan(rm.u[-1]) * XP_t
    eps_[-1] = rm.y[-2] + math.tan(rm.u[-2]) * t
    yo, Uo, ts, _ = _trace2d(layout, y_EP[:-1], np.zeros(k_rays - 1), layout.aspheric, backend)
    z = np.cumsum(ts, axis=0)
    tt = BFD - (z[-2] - z[-1])                                   # sag(ray::RealRay{Tangential}) :91
    y_XP[:-1] = yo[-1] + np.tan(Uo[-1]) * XP_t
    eps_[:-1] = yo[-1] + np.tan(Uo[-1]) * tt
    return y_XP, eps_


def SA(y, eps_, degree):
    """SA -- odd-polynomial least-squares fit, src/SeidelAberrations.jl:139-146"""
    if degree % 2 == 0 or degree < 3:
        raise ValueError("DomainError: Required: isodd(degree) && degree >= 3")
    yp = np.asarray(y) / np.max(y)
    A = np.column_stack([yp ** k for k in range(3, degree + 1, 2)])
    return np.linalg.lstsq(A, np.asarray(eps_), rcond=None)[0]
