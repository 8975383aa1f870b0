"""Prescriptions used by tests and benchmarks.  Rows are [R t n] (row 1 = object space), `a` the
clear semi-apertures per surface, `h` the Gaussian image height passed to solve()."""
import numpy as np

inf = np.inf

# Cooke triplet: the reference's test fixture (test/runtests.jl:19-35)
COOKE = dict(
    surfaces=np.array([
        [inf, 0.0, 1.0],
        [37.40, 5.90, 1.61272],
        [-341.48, 12.93, 1.0],
        [-42.65, 2.50, 1.64769],
        [36.40, 2.00, 1.0],
        [inf, 9.85, 1.0],          # stop
        [204.52, 5.90, 1.61272],
        [-37.05, 0.0, 1.0],
    ]),
    a=np.array([14.7, 14.7, 10.8, 10.8, 10.3, 11.6, 11.6]),
    h=21.248,
)

# Tessar: the reference's docs example (docs/setup.jl:3-21; layout from Hecht's Optics)
TESSAR = dict(
    surfaces=np.array([
        [inf, 0.0, 1.0],
        [16.28, 3.57, 1.6116],
        [-275.7, 1.89, 1.0],
        [-34.57, 0.81, 1.6053],
        [15.82, 2.345, 1.0],
        [inf, 0.905, 1.0],
        [inf, 2.17, 1.5123],
        [19.2, 3.96, 1.6116],
        [-24.0, 0.0, 1.0],
    ]),
    a=np.array([9.5, 9.5, 9.0, 9.0, 7.63, 8.5, 8.5, 8.5]),
    h=21.5,
)

# Biconvex singlet (test/runtests.jl:364-366)
SINGLET = dict(
    surfaces=np.array([[inf, 0.0, 1.0], [100.0, 10.0, 1.5168], [-100.0, 0.0, 1.0]]),
    a=np.array([20.0, 20.0]), h=17.787,
)

# The Cooke triplet as a Layout{Aspheric}, rows [R t n K]: the second element's rear surface a conic, every other curved
# surface a K = 0 sphere.  A Layout{Aspheric} traces each of those spheres with atan(tilt(y, R, K, p)) (src/Types.jl:27,
# src/RayTracing.jl:162), the fixture that tells that branch from asin(tilt(y, R)).
COOKE_ASPHERIC = dict(
    surfaces=np.column_stack([COOKE["surfaces"], [0.0, 0.0, 0.0, 0.0, -0.6, 0.0, 0.0, 0.0]]),
    a=COOKE["a"], h=COOKE["h"],
)

# Parabolic reflector, Layout{Aspheric} rows [R t n K] (test/runtests.jl:335-340)
PARABOLA = dict(
    surfaces=np.array([[inf, 0.0, 1.0, 0.0], [-100.0, 0.0, -1.0, -1.0]]),
    a=np.array([30.0]), h=21.0,
)

# Mangin-like reflective stack (test/runtests.jl:377-383)
REFLECTIVE = dict(
    surfaces=np.array([[inf, 0.0, 1.0], [-100.0, -24.0, -1.0], [50.0, -3.0, -1.5], [-50.0, 0.0, -1.0]]),
    a=np.array([15.0, 11.0, 11.0]), h=10.0,
    K=np.array([0.0, 0.0, -0.5, 0.0]),     # as a Layout{Aspheric}: a K = 0 mirror first, one conic behind it
)

# 10-glass-surface double-Gauss, f/3-class (BASELINE config 2/3; NOT in the reference -- synthetic,
# SURVEY.md section 8d): 8 curved + 2 plano interfaces + stop; f = 99.50 mm, BFD = 57.50 mm.
DOUBLE_GAUSS = dict(
    surfaces=np.array([
        [inf, 0.0, 1.0],
        [54.153, 8.747, 1.60738],
        [152.522, 0.5, 1.0],
        [35.951, 14.0, 1.62041],
        [inf, 3.777, 1.60342],
        [22.270, 14.253, 1.0],
        [inf, 12.428, 1.0],        # stop
        [-25.685, 3.777, 1.60342],
        [inf, 10.834, 1.62041],
        [-36.980, 0.5, 1.0],
        [196.417, 6.858, 1.62041],
        [-67.148, 0.0, 1.0],
    ]),
    a=np.array([29.225, 28.141, 24.296, 21.297, 14.919, 10.229, 13.188, 16.468, 18.930, 21.311, 21.646]),
    h=24.0,
)
DOUBLE_GAUSS_FIELDS = (0.0, 0.25, 0.5, 0.75, 1.0)
DOUBLE_GAUSS_GLASS_SURFACES = 10      # headline intersections per ray (conservative; loop steps = 12)


def zoom20(seed=1234):
    """40-row paraxial Lens for BASELINE config 4: 20 thin-ish elements (SURVEY.md section 8d)."""
    rng = np.random.default_rng(seed)
    rows = [[inf, 0.0, 1.0]]
    sign = 1.0
    for _ in range(20):
        n_glass = rng.uniform(1.48, 1.85)
        rows.append([sign * rng.uniform(30.0, 300.0), rng.uniform(2.0, 8.0), n_glass])
        rows.append([-sign * rng.uniform(30.0, 300.0), rng.uniform(0.5, 20.0), 1.0])
        sign = -sign
    rows[-1][1] = 0.0
    return np.array(rows)


def perturbed_triplets(C, seed=7):
    """BASELINE config 5: C Cooke-triplet variants, radii * (1 + U(-0.02, 0.02)), thicknesses *
    (1 + U(-0.01, 0.01)).  Returns RtnK (C, 4, rows) for the EXTENDED surfaces given by the caller."""
    rng = np.random.default_rng(seed)
    S = COOKE["surfaces"]
    rows = S.shape[0]
    out = np.empty((C, 4, rows))
    dR = 1.0 + rng.uniform(-0.02, 0.02, size=(C, rows))
    dt = 1.0 + rng.uniform(-0.01, 0.01, size=(C, rows))
    out[:, 0, :] = np.where(np.isfinite(S[:, 0]), S[:, 0] * dR, S[:, 0])
    out[:, 1, :] = S[:, 1] * dt
    out[:, 2, :] = S[:, 2]
    out[:, 3, :] = 0.0
    return out


def reversed_chief_layout(surfaces, bfd, K=None):
    """The reversed system trace_chief_ray traces for a Layout (src/RayTracing.jl:267-277): rev_R = -[Inf; R[end:-1:2]],
    rev_t = t[end:-1:1] with rev_t[1] = BFD, rev_n = n[end:-1:1] and K = reverse(K) -- one row off against rev_R, as
    the reference builds it.  Returns ([R t n] rows, K); the reversed system is always a Layout{Aspheric}."""
    S = np.asarray(surfaces, dtype=np.float64)
    rev_t = S[::-1, 1].copy()
    rev_t[0] = bfd
    rev = np.column_stack([-np.concatenate([[inf], S[:0:-1, 0]]), rev_t, S[::-1, 2]])
    Kr = (np.zeros(S.shape[0]) if K is None else np.asarray(K, dtype=np.float64))[::-1].copy()
    return rev, Kr
