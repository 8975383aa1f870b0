"""ctypes binding of libort_b200.so (include/ort_b200.h).

There is NO CPU fallback: if the shared library is missing, or no sm_100 GPU is usable, every
compute entry point raises.  Nothing in this package imports oracle/.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ORT_B200_LIB", os.path.join(_HERE, "lib", "libort_b200.so"))

ORT_OK, ORT_EINVAL, ORT_ECUDA, ORT_ENCCL, ORT_EUNSUPPORTED, ORT_ENOMEM = 0, -1, -2, -3, -4, -5
MAX_ROWS, MAX_FIELDS, MAX_LENS, MAX_GPUS, MAX_FOCI = 64, 32, 128, 16, 64
COMM_ID_BYTES = 128
FLAG_MISS, FLAG_TIR, FLAG_DOMAIN, FLAG_CLIP, FLAG_VIGN = 1, 2, 4, 8, 16
EXT_OPD, EXT_VIGNETTE = 1, 2
STRICT, FAST = 0, 1
AIM_NOUT = 24
VIG_TAIL = 12
MAX_RADII, MAX_FRACS = 1024, 8
ENERGY_CIRCLE, ENERGY_SQUARE = 0, 1
CENTER_CENTROID, CENTER_PARAXIAL = 0, 1
ZERN_MAX_ORDER = 12
PSF_MAX_SIDE = 1024
MTF_MAX_FREQS = 1024

# every symbol include/ort_b200.h declares (tests check the .so exports exactly these)
SYMBOLS = [
    "ort_version", "ort_init", "ort_free", "ort_last_error", "ort_sync", "ort_device_info",
    "ort_host_alloc", "ort_host_free", "ort_device_numa", "ort_bind_host_thread", "ort_launch_count", "ort_profile_enable", "ort_profile_read",
    "ort_set_layout", "ort_set_apertures", "ort_set_polynomials",
    "ort_trace3d_grid", "ort_trace3d_grid_dev", "ort_trace3d_focus", "ort_trace3d_focus_dev",
    "ort_spot_energy_dev", "ort_trace3d_energy", "ort_wavefront_zernike_dev", "ort_trace3d_zernike",
    "ort_wavefront_psf_dev", "ort_trace3d_psf", "ort_wavefront_mtf_dev", "ort_trace3d_mtf",
    "ort_trace3d_rays", "ort_trace3d_rays_opl", "ort_trace3d_rays_dev", "ort_trace2d_batch", "ort_aim2d",
    "ort_paraxial_batch", "ort_paraxial_batch_dev", "ort_transfer_batch", "ort_transfer_batch_dev",
    "ort_trace3d_candidates", "ort_trace3d_candidates_dev", "ort_aim_candidates", "ort_aim_candidates_dev", "ort_aim_fields",
    "ort_trace3d_candidates_aimed", "ort_trace3d_candidates_aimed_dev", "ort_vignetting_candidates",
    "ort_vignetting_candidates_dev", "ort_seidel_candidates",
    "ort_seidel_candidates_dev", "ort_merge_stats", "ort_merge_stats_dev", "ort_rms_from_stats", "ort_fp64_peak", "ort_selftest_exact_ops",
    "ort_comm_unique_id", "ort_comm_init_rank", "ort_comm_init_all", "ort_comm_info", "ort_comm_free", "ort_comm_range",
    "ort_trace3d_grid_multi", "ort_candidates_sharded", "ort_candidates_sharded_dev",
]

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_i32p = C.POINTER(C.c_int32)


class OrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libort_b200 error {code}: {msg}")
        self.code = code


class Field(C.Structure):
    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("u", C.c_double), ("v", C.c_double),
                ("ybar", C.c_double), ("z0", C.c_double), ("h_prime", C.c_double),
                ("opd_xc", C.c_double), ("opd_yc", C.c_double), ("opd_radius", C.c_double), ("opl_ref", C.c_double)]


class Opts(C.Structure):
    _fields_ = [("arith", C.c_int32), ("compact", C.c_int32), ("ys_per_field", C.c_int32),
                ("ext", C.c_int32), ("wg_nu", C.c_double), ("wg_lambda", C.c_double), ("opd_scale", C.c_double),
                ("gather_stats", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("n_kept", C.c_int64), ("mean_x", C.c_double), ("mean_y", C.c_double),
                ("m2_x", C.c_double), ("m2_y", C.c_double), ("r_max", C.c_double),
                ("n_miss", C.c_int64), ("n_tir", C.c_int64), ("n_domain", C.c_int64),
                ("n_clip", C.c_int64), ("n_vig", C.c_int64), ("mean_opd", C.c_double), ("m2_opd", C.c_double),
                ("n_strict", C.c_int64)]


STATS_DTYPE = np.dtype([("n_kept", "<i8"), ("mean_x", "<f8"), ("mean_y", "<f8"), ("m2_x", "<f8"),
                        ("m2_y", "<f8"), ("r_max", "<f8"), ("n_miss", "<i8"), ("n_tir", "<i8"),
                        ("n_domain", "<i8"), ("n_clip", "<i8"), ("n_vig", "<i8"), ("mean_opd", "<f8"),
                        ("m2_opd", "<f8"), ("n_strict", "<i8")])
STATS_BYTES = STATS_DTYPE.itemsize
assert STATS_BYTES == C.sizeof(Stats) == 112


class GridOut(C.Structure):
    _fields_ = [("ex", C.c_void_p), ("ey", C.c_void_p), ("r", C.c_void_p), ("theta", C.c_void_p),
                ("wx", C.c_void_p), ("wy", C.c_void_p), ("opd", C.c_void_p), ("mask", C.c_void_p),
                ("flags", C.c_void_p), ("stats", C.c_void_p), ("stats_local", C.c_void_p)]


GRID_OUT_NAMES = tuple(name for name, _ in GridOut._fields_)


class EnergyReq(C.Structure):
    _fields_ = [("metric", C.c_int32), ("center", C.c_int32), ("n_radii", C.c_int32), ("n_fracs", C.c_int32),
                ("radii", C.c_void_p), ("fracs", C.c_void_p)]


class SpotSets(C.Structure):
    _fields_ = [("n_sets", C.c_int32), ("sets_per_mask", C.c_int32), ("stride", C.c_int64), ("ex", C.c_void_p),
                ("ey", C.c_void_p), ("mask", C.c_void_p), ("stats", C.c_void_p)]


SPOT_SETS_NAMES = tuple(name for name, _ in SpotSets._fields_)


class ZernikeReq(C.Structure):
    _fields_ = [("n_max", C.c_int32), ("reserved", C.c_int32), ("r_norm", C.c_double)]


class WaveSets(C.Structure):
    _fields_ = [("n_sets", C.c_int32), ("reserved", C.c_int32), ("stride", C.c_int64), ("opd", C.c_void_p),
                ("r", C.c_void_p), ("theta", C.c_void_p), ("mask", C.c_void_p), ("stats", C.c_void_p)]


WAVE_SETS_NAMES = tuple(name for name, _ in WaveSets._fields_)


class PsfReq(C.Structure):
    _fields_ = [("n_u", C.c_int32), ("n_v", C.c_int32), ("du", C.c_double), ("dv", C.c_double), ("scale", C.c_double)]


class MtfReq(C.Structure):
    _fields_ = [("n_freq", C.c_int32), ("reserved", C.c_int32), ("freqs", C.POINTER(C.c_double)),
                ("scale", C.c_double)]


def mtf_req(freqs, scale):
    """-> (MtfReq, the float64 array it points into: keep it alive while the request is used)"""
    f = np.ascontiguousarray(np.asarray(freqs, dtype=np.float64).ravel())
    return MtfReq(len(f), 0, f.ctypes.data_as(C.POINTER(C.c_double)), float(scale)), f


def zernike_terms(n_max):
    """J = (n_max + 1)(n_max + 2) / 2 coefficients per set, in ANSI order"""
    return (int(n_max) + 1) * (int(n_max) + 2) // 2
RAY_OUT_NAMES = GRID_OUT_NAMES[:9]          # the per-ray members: every one but the statistics records


_lib = None


def load():
    """Load libort_b200.so (no GPU needed to load; compute calls need one)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OrtError(ORT_ECUDA, f"{LIB_PATH} not found: build it with `python -c 'import "
                       "__graft_entry__ as g; g.build()'` (make -C opticalraytracing.jl_b200/csrc). "
                       "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.ort_version.restype = C.c_int
    L.ort_init.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.ort_free.argtypes = [C.c_void_p]
    L.ort_free.restype = None
    L.ort_last_error.argtypes = [C.c_void_p]
    L.ort_last_error.restype = C.c_char_p
    L.ort_sync.argtypes = [C.c_void_p]
    L.ort_device_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_int), C.c_char_p, C.c_int]
    L.ort_device_numa.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_char_p, C.c_int]
    L.ort_bind_host_thread.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    L.ort_host_alloc.argtypes = [C.c_size_t]
    L.ort_host_alloc.restype = C.c_void_p
    L.ort_host_free.argtypes = [C.c_void_p]
    L.ort_host_free.restype = None
    L.ort_launch_count.argtypes = [C.c_void_p]
    L.ort_launch_count.restype = C.c_int64
    L.ort_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.ort_profile_read.argtypes = [C.c_void_p, _dp, C.c_int]
    L.ort_set_layout.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp]
    L.ort_set_apertures.argtypes = [C.c_void_p, C.c_int, _dp]
    grid_args = [C.c_void_p, C.POINTER(Field), C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                 C.c_int, C.c_double, C.POINTER(Opts), C.POINTER(GridOut)]
    L.ort_trace3d_grid.argtypes = grid_args
    L.ort_trace3d_grid_dev.argtypes = grid_args + [C.c_void_p]
    L.ort_trace3d_focus.argtypes = grid_args[:9] + [_dp, C.c_int] + grid_args[9:]
    L.ort_trace3d_focus_dev.argtypes = grid_args[:9] + [_dp, C.c_int] + grid_args[9:] + [C.c_void_p]
    L.ort_spot_energy_dev.argtypes = [C.c_void_p, C.POINTER(SpotSets), C.POINTER(EnergyReq), C.c_void_p, C.c_void_p,
                                      C.c_void_p]
    L.ort_trace3d_energy.argtypes = grid_args[:9] + [_dp, C.c_int, C.POINTER(Opts), C.POINTER(EnergyReq), C.c_void_p,
                                                     C.c_void_p, C.c_void_p]
    L.ort_wavefront_zernike_dev.argtypes = [C.c_void_p, C.POINTER(WaveSets), C.POINTER(ZernikeReq), C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    L.ort_trace3d_zernike.argtypes = grid_args[:9] + [C.POINTER(Opts), C.POINTER(ZernikeReq), C.c_void_p, C.c_void_p,
                                                      C.c_void_p, C.c_void_p]
    L.ort_wavefront_psf_dev.argtypes = [C.c_void_p, C.POINTER(WaveSets), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                        C.c_int, C.POINTER(PsfReq)] + [C.c_void_p] * 5
    L.ort_trace3d_psf.argtypes = grid_args[:9] + [C.POINTER(Opts), C.POINTER(PsfReq)] + [C.c_void_p] * 5
    L.ort_wavefront_mtf_dev.argtypes = [C.c_void_p, C.POINTER(WaveSets), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                        C.c_int, C.POINTER(MtfReq)] + [C.c_void_p] * 3
    L.ort_trace3d_mtf.argtypes = grid_args[:9] + [C.POINTER(Opts), C.POINTER(MtfReq)] + [C.c_void_p] * 3
    L.ort_trace3d_rays.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, _dp, C.c_int, _dp, _dp, _dp, _u8p]
    L.ort_trace3d_rays_opl.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, _dp, C.c_int, _dp, _dp, _dp, _u8p, _dp]
    L.ort_trace3d_rays_dev.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 6
    L.ort_trace2d_batch.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, C.c_int, _dp, _dp, _dp, _u8p]
    L.ort_aim2d.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, _dp, _i32p]
    L.ort_paraxial_batch.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, C.c_int, C.c_int, C.c_int64,
                                     _dp, _dp, _dp, _dp, _i32p, _dp, _dp]
    L.ort_paraxial_batch_dev.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, C.c_int, C.c_int, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
    L.ort_transfer_batch.argtypes = [C.c_void_p, _dp, C.c_double, C.c_double, C.c_int, C.c_int64, _dp, _dp]
    L.ort_transfer_batch_dev.argtypes = [C.c_void_p, _dp, C.c_double, C.c_double, C.c_int, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
    L.ort_trace3d_candidates.argtypes = [C.c_void_p, C.c_int, C.c_int64, _dp, C.POINTER(Field), _dp,
                                         C.c_int, _dp, C.c_int, C.c_int, C.c_double, C.c_int, _dp]
    L.ort_trace3d_candidates_dev.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.POINTER(Field),
                                             C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                             C.c_double, C.c_int, C.c_void_p, C.c_void_p]
    L.ort_seidel_candidates.argtypes = [C.c_void_p, C.c_int, C.c_int64, _dp, _dp, C.c_double, C.c_double, _dp, _dp, _dp]
    L.ort_seidel_candidates_dev.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, _dp, C.c_double, C.c_double, _dp,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    L.ort_vignetting_candidates.argtypes = [C.c_void_p, C.c_int, C.c_int64, _dp, _dp, _dp, C.c_double, _dp]
    L.ort_vignetting_candidates_dev.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, _dp, _dp, C.c_double, C.c_void_p,
                                                C.c_void_p]
    L.ort_aim_candidates.argtypes = [C.c_void_p, C.c_int, C.c_int64, _dp, _dp, C.c_double, C.c_double, C.c_int, _dp]
    L.ort_set_polynomials.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp]
    L.ort_aim_fields.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp, C.c_double, _dp, C.c_int, C.c_int, _dp]
    L.ort_aim_candidates_dev.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, _dp, C.c_double, C.c_double, C.c_int,
                                         C.c_void_p, C.c_void_p]
    L.ort_trace3d_candidates_aimed.argtypes = [C.c_void_p, C.c_int, C.c_int64, _dp, _dp, C.c_int, C.c_int, C.c_int, _dp]
    L.ort_trace3d_candidates_aimed_dev.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                   C.c_int, C.c_void_p, C.c_void_p]
    L.ort_merge_stats.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.ort_merge_stats_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.ort_rms_from_stats.argtypes = [C.c_void_p]
    L.ort_rms_from_stats.restype = C.c_double
    L.ort_fp64_peak.argtypes = [C.c_void_p, _dp, _dp]
    L.ort_selftest_exact_ops.argtypes = [C.c_void_p, C.c_longlong, C.c_ulonglong, C.POINTER(C.c_longlong)]
    L.ort_comm_unique_id.argtypes = [C.c_void_p]
    L.ort_comm_init_rank.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.ort_comm_init_all.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.ort_comm_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.ort_comm_free.argtypes = [C.c_void_p]
    L.ort_comm_range.argtypes = [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.ort_trace3d_grid_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int] + grid_args[1:]
    L.ort_candidates_sharded.argtypes = [C.c_void_p, C.c_int, C.c_int64, _dp, _dp, C.c_double, C.c_double, C.c_int, C.c_int,
                                         C.c_int, C.c_int, _dp, _dp]
    L.ort_candidates_sharded_dev.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, _dp, C.c_double, C.c_double, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = L
    return L


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _vp(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class PinnedArray:
    """numpy view over cudaHostAlloc memory (ort_host_alloc).  Keep the object alive while used."""

    def __init__(self, shape, dtype=np.float64):
        L = load()
        self.dtype = np.dtype(dtype)
        self.shape = tuple(np.atleast_1d(shape).tolist()) if not isinstance(shape, tuple) else shape
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = L.ort_host_alloc(max(self.nbytes, 8))
        if not self.ptr:
            raise OrtError(ORT_ENOMEM, f"ort_host_alloc({self.nbytes}) failed")
        buf = (C.c_uint8 * max(self.nbytes, 8)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            load().ort_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def merge_stats_c(records):
    """ort_merge_stats: records (n_shards, n_fields) structured array -> (n_fields,)"""
    rec = np.ascontiguousarray(records, dtype=STATS_DTYPE)
    ns, nf = rec.shape
    out = np.zeros(nf, dtype=STATS_DTYPE)
    rc = load().ort_merge_stats(rec.ctypes.data, ns, nf, out.ctypes.data)
    if rc != ORT_OK:
        raise OrtError(rc, "ort_merge_stats")
    return out


def rms_from_stats_c(rec):
    r = np.ascontiguousarray(np.atleast_1d(rec), dtype=STATS_DTYPE)
    return float(load().ort_rms_from_stats(r.ctypes.data))


def comm_unique_id():
    """128 opaque bytes identifying a new communicator (ncclGetUniqueId); ship them to every rank"""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    rc = load().ort_comm_unique_id(buf)
    if rc != ORT_OK:
        raise OrtError(rc, load().ort_last_error(None).decode())
    return bytes(buf)


def comm_range(total, rank, world):
    lo, hi = C.c_int64(), C.c_int64()
    rc = load().ort_comm_range(int(total), int(rank), int(world), C.byref(lo), C.byref(hi))
    if rc != ORT_OK:
        raise OrtError(rc, "ort_comm_range")
    return lo.value, hi.value


def comm_init_all(contexts):
    """one process, several GPUs: a communicator over `contexts` (one per device), rank = position in the list"""
    arr = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
    rc = load().ort_comm_init_all(arr, len(contexts))
    if rc != ORT_OK:
        raise OrtError(rc, load().ort_last_error(contexts[0].h if contexts else None).decode())


def trace3d_grid_multi(contexts, fields, ys, xs, stop, a_stop, arith=FAST, compact=False,
                       want=("ex", "ey", "mask", "stats"), wavegrad=None, out=None, ext=0, opd_scale=1.0):
    """ort_trace3d_grid_multi: the WHOLE grid (ys, xs) over the contexts of this process, y-rows block-sharded; outputs as
    Context.trace3d_grid in the reference's order, 'stats' merged by the library, 'stats_local' (n, n_fields)."""
    L = load()
    farr, nf = make_fields(fields)
    ys, xs = _d(ys), _d(xs)
    per_field = ys.ndim == 2
    if per_field and ys.shape[0] != nf:
        raise ValueError("ys must be (ny,) or (n_fields, ny)")
    ny, nx = ys.shape[-1], len(xs)
    if "opd" in want:
        ext |= EXT_OPD
    stats = np.zeros(nf, dtype=STATS_DTYPE)
    local = np.zeros((len(contexts), nf), dtype=STATS_DTYPE)
    res, go = _host_out(want, out, nf, ny * nx, stats, local)
    op = _opts(arith, compact, per_field, ext, wavegrad, opd_scale)
    arr = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
    rc = L.ort_trace3d_grid_multi(arr, len(contexts), farr, nf, _vp(ys), ny, _vp(xs), nx, int(stop), float(a_stop),
                                  C.byref(op), C.byref(go))
    if rc != ORT_OK:
        raise OrtError(rc, L.ort_last_error(contexts[0].h).decode())
    res["stats"], res["stats_local"] = stats, local
    return res


def _host_out(want, out, nf, NN, stats, local=None, foci=None):
    """The result dict of a host-pointer sweep and the GridOut over it: the arrays of `out`, and new ones for the other
    per-ray members named in `want`, (n_fields, ny*nx) each.  foci = M: a through-focus sweep, whose ex, ey are
    (n_fields, M, ny*nx) and which has no wx, wy, opd."""
    res = dict(out) if out else {}
    for name in RAY_OUT_NAMES:
        if name not in want or name in res or (foci is not None and name in ("wx", "wy", "opd")):
            continue
        shape = (nf, foci, NN) if foci is not None and name in ("ex", "ey") else (nf, NN)
        res[name] = np.zeros(shape, dtype=np.uint8) if name in ("mask", "flags") else np.empty(shape, dtype=np.float64)
    go = GridOut(*[(res[k].ctypes.data if res.get(k) is not None else None) for k in RAY_OUT_NAMES],
                 stats.ctypes.data, None if local is None else local.ctypes.data)
    return res, go


def _opts(arith, compact, ys_per_field, ext=0, wavegrad=None, opd_scale=1.0, gather=False):
    nu, lam = wavegrad if wavegrad else (0.0, 1.0)
    return Opts(int(arith), int(bool(compact)), int(bool(ys_per_field)), int(ext), float(nu), float(lam), float(opd_scale),
                int(bool(gather)), 0)


_METRICS = {"circle": ENERGY_CIRCLE, "square": ENERGY_SQUARE}
_CENTERS = {"centroid": CENTER_CENTROID, "paraxial": CENTER_PARAXIAL}


def _energy_req(radii, fracs, metric, center):
    """EnergyReq over float64 copies of radii and fracs (returned too: they must outlive the call).  metric / center are
    the names ("circle" / "square", "centroid" / "paraxial") or the ORT_* codes; the library validates the values."""
    r = _d(np.atleast_1d(np.asarray(radii, dtype=np.float64)) if radii is not None else np.empty(0))
    q = _d(np.atleast_1d(np.asarray(fracs, dtype=np.float64)) if fracs is not None else np.empty(0))
    m = _METRICS[metric] if isinstance(metric, str) else int(metric)
    c = _CENTERS[center] if isinstance(center, str) else int(center)
    req = EnergyReq(m, c, len(r), len(q), r.ctypes.data if len(r) else None, q.ctypes.data if len(q) else None)
    return req, r, q


def make_fields(fields):
    """fields: iterable of dicts / Field -> (ctypes array, n)"""
    fl = list(fields)
    arr = (Field * len(fl))()
    for i, f in enumerate(fl):
        if isinstance(f, Field):
            arr[i] = f
        else:
            arr[i] = Field(int(f.get("mode", 0)), 0, float(f.get("u", 0.0)), float(f.get("v", 0.0)),
                           float(f.get("ybar", 0.0)), float(f.get("z0", 1.0)), float(f.get("h_prime", 0.0)),
                           float(f.get("opd_xc", 0.0)), float(f.get("opd_yc", 0.0)), float(f.get("opd_radius", 0.0)),
                           float(f.get("opl_ref", 0.0)))
    return arr, len(fl)


class Context:
    """One ort_ctx (one GPU).  Thin, typed wrapper over the C ABI; numpy arrays in and out."""

    def __init__(self, device=0):
        self.L = load()
        h = C.c_void_p()
        rc = self.L.ort_init(C.byref(h), int(device))
        if rc != ORT_OK:
            raise OrtError(rc, self.L.ort_last_error(None).decode())
        self.h = h
        self.device = int(device)
        self.rows = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.ort_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != ORT_OK:
            raise OrtError(rc, self.L.ort_last_error(self.h).decode())

    # ---- context -------------------------------------------------------------------------
    def device_info(self):
        sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
        name = C.create_string_buffer(128)
        self._ck(self.L.ort_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi), name, 128))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "name": name.value.decode()}

    def sync(self):
        self._ck(self.L.ort_sync(self.h))

    def device_numa(self):
        """(NUMA node of this context's GPU or -1, that node's CPU list)"""
        node, buf = C.c_int(-1), C.create_string_buffer(1024)
        self._ck(self.L.ort_device_numa(self.h, C.byref(node), buf, 1024))
        return node.value, buf.value.decode()

    def bind_host_thread(self):
        """pin the calling thread (and its future allocations) next to this context's GPU; -> 0 if not possible, else
        bit 0 = CPU affinity set, bit 1 = memory policy set"""
        got = C.c_int(0)
        rc = self.L.ort_bind_host_thread(self.h, C.byref(got))
        return got.value if rc == ORT_OK else 0

    def launch_count(self):
        return int(self.L.ort_launch_count(self.h))

    def profile_enable(self, on=True):
        self._ck(self.L.ort_profile_enable(self.h, int(bool(on))))

    def profile_read(self):
        """kernel durations (ms) of the dominant kernel of the calls since the last read (<= 64)"""
        buf = np.empty(64)
        n = self.L.ort_profile_read(self.h, _p(buf), 64)
        if n < 0:
            self._ck(n)
        return buf[:n].copy()

    def fp64_peak(self):
        t, ms = C.c_double(), C.c_double()
        self._ck(self.L.ort_fp64_peak(self.h, C.byref(t), C.byref(ms)))
        return t.value, ms.value

    def selftest_exact_ops(self, n=1 << 26, seed=1):
        """xdiv / xsqrt of the STRICT kernels against __ddiv_rn / __dsqrt_rn on >= n operand pairs (ort_selftest_exact_ops)
        -> dict(div_tested, div_flagged, div_mismatch, sqrt_tested, sqrt_flagged, sqrt_mismatch, div_flagged_moderate,
        sqrt_flagged_moderate)"""
        out = (C.c_longlong * 8)()
        self._ck(self.L.ort_selftest_exact_ops(self.h, int(n), int(seed), out))
        keys = ("div_tested", "div_flagged", "div_mismatch", "sqrt_tested", "sqrt_flagged", "sqrt_mismatch",
                "div_flagged_moderate", "sqrt_flagged_moderate")
        return dict(zip(keys, [int(v) for v in out]))

    def set_layout(self, surfaces, K=None):
        """surfaces: rows x 3 [R t n] (or rows x 4 with K); row 1 = object space."""
        S = np.asarray(surfaces, dtype=np.float64)
        if K is None and S.shape[1] > 3:
            K = S[:, 3]
        R, t, n = _d(S[:, 0]), _d(S[:, 1]), _d(S[:, 2])
        Kc = None if K is None else _d(K)
        self._ck(self.L.ort_set_layout(self.h, len(R), _p(R), _p(t), _p(n), _p(Kc)))
        self.rows = len(R)

    def set_apertures(self, a):
        """EXTENSION: clear semi-apertures of the surfaces of the current layout (None = unlimited)."""
        if a is None:
            self._ck(self.L.ort_set_apertures(self.h, 0, None))
        else:
            a = _d(a)
            self._ck(self.L.ort_set_apertures(self.h, len(a), _p(a)))

    # ---- communicator (NCCL inside the library) --------------------------------------------
    def comm_init_rank(self, comm_id, rank, world):
        """join a one-process-per-GPU communicator; comm_id = the 128 bytes of comm_unique_id() made on rank 0"""
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(bytes(comm_id))
        self._ck(self.L.ort_comm_init_rank(self.h, buf, int(rank), int(world)))

    def merge_stats_dev(self, d_recs, n_shards, n_fields, d_out, stream=0):
        """the library's merge kernel on records already in HBM: (n_shards, n_fields) -> (n_fields,)"""
        self._ck(self.L.ort_merge_stats_dev(self.h, C.c_void_p(d_recs), int(n_shards), int(n_fields), C.c_void_p(d_out),
                                            C.c_void_p(stream)))

    def comm_info(self):
        r, w, v = C.c_int(), C.c_int(), C.c_int()
        self._ck(self.L.ort_comm_info(self.h, C.byref(r), C.byref(w), C.byref(v)))
        return {"rank": r.value, "world": w.value, "nccl_version": v.value}

    def comm_free(self):
        self._ck(self.L.ort_comm_free(self.h))

    def candidates_sharded(self, RtnK, a, h_prime, H, k_rays=64, arith=FAST, aspheric=False, want_aim=False):
        """BASELINE config 5 over the communicator: prelude + aimed sweep of this rank's range of the population, merit
        table (C, 4) complete on every rank (ort_candidates_sharded)."""
        RtnK = _d(RtnK)
        Cn, four, rows = RtnK.shape
        a = _d(a)
        assert four == 4 and a.shape == (rows - 1,)
        out = np.empty((Cn, 4), dtype=np.float64)
        aim = np.full((Cn, AIM_NOUT), np.nan) if want_aim else None
        self._ck(self.L.ort_candidates_sharded(self.h, rows, Cn, _p(RtnK), _p(a), float(h_prime), float(H), int(bool(aspheric)),
                                               int(k_rays), int(k_rays) // 2, int(arith), _p(aim), _p(out)))
        return (out, aim) if want_aim else out

    def candidates_sharded_dev(self, rows, Cn, d_RtnK, a, h_prime, H, ny, nx, d_out, d_aim=0, arith=FAST, aspheric=False,
                               stream=0):
        a = _d(a)
        self._ck(self.L.ort_candidates_sharded_dev(self.h, int(rows), int(Cn), C.c_void_p(d_RtnK), _p(a), float(h_prime),
                                                   float(H), int(bool(aspheric)), int(ny), int(nx), int(arith),
                                                   C.c_void_p(d_aim or 0), C.c_void_p(d_out), C.c_void_p(stream)))

    # ---- 3-D grid ------------------------------------------------------------------------
    def trace3d_grid(self, fields, ys, xs, stop, a_stop, arith=FAST, compact=False,
                     want=("ex", "ey", "mask", "stats"), wavegrad=None, out=None, ext=0, opd_scale=1.0, gather=False):
        """Host-pointer grid sweep.  Returns dict of numpy arrays shaped (n_fields, ny*nx)
        (+ 'stats' structured array).  `out` may supply preallocated (e.g. pinned) arrays.
        gather=True (needs comm_init_rank): ys is this rank's block of y-rows of a sharded grid; 'stats' are the records
        merged over all ranks by the library (all-gather + merge kernel), 'stats_local' this rank's own."""
        farr, nf = make_fields(fields)
        ys, xs = _d(ys), _d(xs)
        per_field = ys.ndim == 2          # ys[n_fields][ny]: every field has its own aimed y-range
        if per_field and ys.shape[0] != nf:
            raise ValueError("ys must be (ny,) or (n_fields, ny)")
        ny, nx = ys.shape[-1], len(xs)
        if "opd" in want:
            ext |= EXT_OPD
        stats = np.zeros(nf, dtype=STATS_DTYPE)
        local = np.zeros(nf, dtype=STATS_DTYPE) if gather else None
        res, go = _host_out(want, out, nf, ny * nx, stats, local)
        op = _opts(arith, compact, per_field, ext, wavegrad, opd_scale, gather)
        self._ck(self.L.ort_trace3d_grid(self.h, farr, nf, _vp(ys), ny, _vp(xs), nx, int(stop),
                                         float(a_stop), C.byref(op), C.byref(go)))
        res["stats"] = stats
        if gather:
            res["stats_local"] = local
        return res

    def trace3d_grid_dev(self, fields, d_ys, ny, d_xs, nx, stop, a_stop, ptrs, stream=0,
                         arith=FAST, compact=False, wavegrad=None, ys_per_field=False, ext=0, opd_scale=1.0, gather=False):
        """Device-pointer grid sweep (enqueue only).  ptrs: dict name -> device address (int).  gather=True: all-gather +
        merge of the statistics records over the communicator behind the sweep, on the same stream (ptrs['stats'] =
        merged, ptrs['stats_local'] = this rank's)."""
        farr, nf = make_fields(fields)
        go = GridOut(*[ptrs.get(k) for k in GRID_OUT_NAMES])
        if ptrs.get("opd"):
            ext |= EXT_OPD
        op = _opts(arith, compact, ys_per_field, ext, wavegrad, opd_scale, gather)
        self._ck(self.L.ort_trace3d_grid_dev(self.h, farr, nf, C.c_void_p(d_ys), int(ny), C.c_void_p(d_xs),
                                             int(nx), int(stop), float(a_stop), C.byref(op), C.byref(go),
                                             C.c_void_p(stream)))

    # ---- through-focus sweep -------------------------------------------------------------
    def trace3d_focus(self, fields, ys, xs, stop, a_stop, foci, arith=FAST, compact=False, want=("stats",)):
        """The grid sweep at M image planes in one pass (ort_trace3d_focus): foci[j] replaces t[rows-2] of the current
        layout.  Returns a dict: 'stats' (n_fields, M) STATS_DTYPE; 'ex', 'ey' (n_fields, M, ny*nx); 'r', 'theta', 'mask',
        'flags' (n_fields, ny*nx), the same for every focus.  With compact=True ex / ey [f, j] hold stats[f, j].n_kept
        entries in push! order (r, theta per field likewise)."""
        farr, nf = make_fields(fields)
        ys, xs = _d(ys), _d(xs)
        per_field = ys.ndim == 2
        if per_field and ys.shape[0] != nf:
            raise ValueError("ys must be (ny,) or (n_fields, ny)")
        foci = _d(np.atleast_1d(foci))
        M = len(foci)
        ny, nx = ys.shape[-1], len(xs)
        stats = np.zeros((nf, M), dtype=STATS_DTYPE)
        res, go = _host_out(want, None, nf, ny * nx, stats, foci=M)
        op = _opts(arith, compact, per_field)
        self._ck(self.L.ort_trace3d_focus(self.h, farr, nf, _vp(ys), ny, _vp(xs), nx, int(stop), float(a_stop), _p(foci), M,
                                          C.byref(op), C.byref(go)))
        res["stats"] = stats
        return res

    def trace3d_focus_dev(self, fields, d_ys, ny, d_xs, nx, stop, a_stop, foci, ptrs, stream=0, arith=FAST, compact=False,
                          ys_per_field=False):
        """Device-pointer through-focus sweep (enqueue only).  ptrs: dict name -> device address; 'ex', 'ey' are
        [n_fields][M][ny*nx], 'r', 'theta', 'mask', 'flags' [n_fields][ny*nx], 'stats' [n_fields][M]."""
        farr, nf = make_fields(fields)
        foci = _d(np.atleast_1d(foci))
        go = GridOut(*[ptrs.get(k) for k in GRID_OUT_NAMES])
        op = _opts(arith, compact, ys_per_field)
        self._ck(self.L.ort_trace3d_focus_dev(self.h, farr, nf, C.c_void_p(d_ys), int(ny), C.c_void_p(d_xs), int(nx),
                                              int(stop), float(a_stop), _p(foci), len(foci), C.byref(op), C.byref(go),
                                              C.c_void_p(stream)))

    # ---- encircled energy ----------------------------------------------------------------
    def spot_energy_dev(self, sets, radii=None, fracs=None, metric="circle", center="centroid", d_counts=0, d_radius=0,
                        stream=0):
        """Encircled / ensquared energy of spot sets already in HBM (ort_spot_energy_dev, enqueue only).  sets: dict with
        n_sets, sets_per_mask, stride and the device addresses ex, ey, mask (0 = compacted segments), stats.  d_counts:
        int64 [n_sets][len(radii)], d_radius: float64 [n_sets][len(fracs)] (device addresses)."""
        ss = SpotSets(*[sets.get(k) or 0 for k in SPOT_SETS_NAMES])
        req, _r, _q = _energy_req(radii, fracs, metric, center)
        self._ck(self.L.ort_spot_energy_dev(self.h, C.byref(ss), C.byref(req), C.c_void_p(d_counts or 0),
                                            C.c_void_p(d_radius or 0), C.c_void_p(stream)))

    def trace3d_energy(self, fields, ys, xs, stop, a_stop, radii=None, fracs=None, foci=None, arith=FAST, metric="circle",
                       center="centroid", ext=0):
        """The grid sweep (foci None) or the through-focus sweep at foci, full grid on the device, and the energy of every
        set on it (ort_trace3d_energy); no spot crosses PCIe.  Returns dict(stats, counts, radius): (n_fields[, M]),
        (n_fields[, M], len(radii)) int64, (n_fields[, M], len(fracs)) float64."""
        farr, nf = make_fields(fields)
        ys, xs = _d(ys), _d(xs)
        per_field = ys.ndim == 2
        if per_field and ys.shape[0] != nf:
            raise ValueError("ys must be (ny,) or (n_fields, ny)")
        fo = None if foci is None else _d(np.atleast_1d(foci))
        M = 0 if fo is None else len(fo)
        req, r, q = _energy_req(radii, fracs, metric, center)
        lead = (nf,) if fo is None else (nf, M)
        stats = np.zeros(lead, dtype=STATS_DTYPE)
        counts = np.zeros(lead + (len(r),), dtype=np.int64)
        radius = np.zeros(lead + (len(q),), dtype=np.float64)
        op = _opts(arith, False, per_field, ext)
        self._ck(self.L.ort_trace3d_energy(self.h, farr, nf, _vp(ys), ys.shape[-1], _vp(xs), len(xs), int(stop),
                                           float(a_stop), _p(fo), M, C.byref(op), C.byref(req), stats.ctypes.data,
                                           counts.ctypes.data if len(r) else None,
                                           radius.ctypes.data if len(q) else None))
        return dict(stats=stats, counts=counts, radius=radius)

    # ---- Zernike fit of the wavefront -----------------------------------------------------
    def wavefront_zernike_dev(self, sets, n_max, r_norm=0.0, d_coef=0, d_resid=0, d_status=0, stream=0):
        """Zernike fit of wavefront sets already in HBM (ort_wavefront_zernike_dev, enqueue only).  sets: dict with n_sets,
        stride and the device addresses opd, r, theta, mask (0 = compacted segments), stats.  d_coef: float64
        [n_sets][zernike_terms(n_max)], d_resid: float64 [n_sets][2], d_status: int32 [n_sets] (device addresses)."""
        ws = WaveSets(*[sets.get(k) or 0 for k in WAVE_SETS_NAMES])
        req = ZernikeReq(int(n_max), 0, float(r_norm))
        self._ck(self.L.ort_wavefront_zernike_dev(self.h, C.byref(ws), C.byref(req), C.c_void_p(d_coef or 0),
                                                  C.c_void_p(d_resid or 0), C.c_void_p(d_status or 0),
                                                  C.c_void_p(stream)))

    def trace3d_zernike(self, fields, ys, xs, stop, a_stop, n_max, r_norm=0.0, arith=FAST, ext=EXT_OPD, opd_scale=1.0):
        """The grid sweep with ORT_EXT_OPD full grid on the device and the Zernike fit of every field on it
        (ort_trace3d_zernike); no ray crosses PCIe.  Returns dict(stats (n_fields,), coef (n_fields, J) float64,
        resid (n_fields, 2) float64 = RMS, PV, status (n_fields,) int32)."""
        farr, nf = make_fields(fields)
        ys, xs = _d(ys), _d(xs)
        per_field = ys.ndim == 2
        if per_field and ys.shape[0] != nf:
            raise ValueError("ys must be (ny,) or (n_fields, ny)")
        stats = np.zeros(nf, dtype=STATS_DTYPE)
        coef = np.zeros((nf, zernike_terms(max(int(n_max), 0))), dtype=np.float64)
        resid = np.zeros((nf, 2), dtype=np.float64)
        status = np.zeros(nf, dtype=np.int32)
        req = ZernikeReq(int(n_max), 0, float(r_norm))
        op = _opts(arith, False, per_field, ext, opd_scale=opd_scale)
        self._ck(self.L.ort_trace3d_zernike(self.h, farr, nf, _vp(ys), ys.shape[-1], _vp(xs), len(xs), int(stop),
                                            float(a_stop), C.byref(op), C.byref(req), stats.ctypes.data,
                                            coef.ctypes.data, resid.ctypes.data, status.ctypes.data))
        return dict(stats=stats, coef=coef, resid=resid, status=status)

    # ---- diffraction PSF of the wavefront ---------------------------------------------------
    def wavefront_psf_dev(self, sets, d_ys, ys_per_set, ny, d_xs, nx, n_u, n_v, du, dv, scale, d_psf=0, d_strehl=0,
                          d_peak=0, d_status=0, stream=0):
        """Diffraction PSF of full-grid wavefront sets already in HBM (ort_wavefront_psf_dev, enqueue only).  sets: dict with
        n_sets, stride = ny * nx and the device addresses opd, mask, stats (r and theta are not read); d_ys
        [ys_per_set ? n_sets : 1][ny], d_xs [nx] device addresses.  d_psf: float64 [n_sets][n_v][n_u], d_strehl: float64
        [n_sets][2], d_peak, d_status: int32 [n_sets] (device addresses)."""
        ws = WaveSets(*[sets.get(k) or 0 for k in WAVE_SETS_NAMES])
        req = PsfReq(int(n_u), int(n_v), float(du), float(dv), float(scale))
        self._ck(self.L.ort_wavefront_psf_dev(self.h, C.byref(ws), C.c_void_p(d_ys or 0), int(ys_per_set), int(ny),
                                              C.c_void_p(d_xs or 0), int(nx), C.byref(req), C.c_void_p(d_psf or 0),
                                              C.c_void_p(d_strehl or 0), C.c_void_p(d_peak or 0),
                                              C.c_void_p(d_status or 0), C.c_void_p(stream)))

    def trace3d_psf(self, fields, ys, xs, stop, a_stop, n_u, n_v, du, dv, scale, arith=FAST, ext=EXT_OPD, opd_scale=1.0):
        """The grid sweep with ORT_EXT_OPD full grid on the device and the diffraction PSF of every field on it
        (ort_trace3d_psf); no ray crosses PCIe.  Returns dict(stats (n_fields,), psf (n_fields, n_v, n_u) float64,
        strehl (n_fields, 2) float64 = strehl_ref, maximum, peak (n_fields,) int32 = iv * n_u + iu, status (n_fields,)
        int32)."""
        farr, nf = make_fields(fields)
        ys, xs = _d(ys), _d(xs)
        per_field = ys.ndim == 2
        if per_field and ys.shape[0] != nf:
            raise ValueError("ys must be (ny,) or (n_fields, ny)")
        stats = np.zeros(nf, dtype=STATS_DTYPE)
        psf = np.zeros((nf, max(int(n_v), 0), max(int(n_u), 0)), dtype=np.float64)
        strehl = np.zeros((nf, 2), dtype=np.float64)
        peak = np.zeros(nf, dtype=np.int32)
        status = np.zeros(nf, dtype=np.int32)
        req = PsfReq(int(n_u), int(n_v), float(du), float(dv), float(scale))
        op = _opts(arith, False, per_field, ext, opd_scale=opd_scale)
        self._ck(self.L.ort_trace3d_psf(self.h, farr, nf, _vp(ys), ys.shape[-1], _vp(xs), len(xs), int(stop),
                                        float(a_stop), C.byref(op), C.byref(req), stats.ctypes.data, psf.ctypes.data,
                                        strehl.ctypes.data, peak.ctypes.data, status.ctypes.data))
        return dict(stats=stats, psf=psf, strehl=strehl, peak=peak, status=status)

    # ---- diffraction MTF of the wavefront ---------------------------------------------------
    def wavefront_mtf_dev(self, sets, d_ys, ys_per_set, ny, d_xs, nx, freqs, scale, d_otf=0, d_status=0, stream=0):
        """Diffraction OTF of full-grid wavefront sets already in HBM (ort_wavefront_mtf_dev, enqueue only).  sets: dict with
        n_sets, stride = ny * nx and the device addresses opd, mask, stats (r and theta are not read); d_ys
        [ys_per_set ? n_sets : 1][ny], d_xs [nx] device addresses; freqs: host array, cycles per image unit.  d_otf:
        float64 [n_sets][2][n_freq][2] (sagittal, tangential; re, im), d_status: int32 [n_sets] (device addresses)."""
        ws = WaveSets(*[sets.get(k) or 0 for k in WAVE_SETS_NAMES])
        req, keep = mtf_req(freqs, scale)
        self._ck(self.L.ort_wavefront_mtf_dev(self.h, C.byref(ws), C.c_void_p(d_ys or 0), int(ys_per_set), int(ny),
                                              C.c_void_p(d_xs or 0), int(nx), C.byref(req), C.c_void_p(d_otf or 0),
                                              C.c_void_p(d_status or 0), C.c_void_p(stream)))
        del keep

    def trace3d_mtf(self, fields, ys, xs, stop, a_stop, freqs, scale, arith=FAST, ext=EXT_OPD, opd_scale=1.0):
        """The grid sweep with ORT_EXT_OPD full grid on the device and the diffraction OTF of every field on it
        (ort_trace3d_mtf); no ray crosses PCIe.  Returns dict(stats (n_fields,), otf (n_fields, 2, n_freq) complex128
        (sagittal, tangential), status (n_fields,) int32)."""
        farr, nf = make_fields(fields)
        ys, xs = _d(ys), _d(xs)
        per_field = ys.ndim == 2
        if per_field and ys.shape[0] != nf:
            raise ValueError("ys must be (ny,) or (n_fields, ny)")
        req, keep = mtf_req(freqs, scale)
        stats = np.zeros(nf, dtype=STATS_DTYPE)
        otf = np.zeros((nf, 2, len(keep), 2), dtype=np.float64)
        status = np.zeros(nf, dtype=np.int32)
        op = _opts(arith, False, per_field, ext, opd_scale=opd_scale)
        self._ck(self.L.ort_trace3d_mtf(self.h, farr, nf, _vp(ys), ys.shape[-1], _vp(xs), len(xs), int(stop),
                                        float(a_stop), C.byref(op), C.byref(req), stats.ctypes.data, otf.ctypes.data,
                                        status.ctypes.data))
        return dict(stats=stats, otf=otf[..., 0] + 1j * otf[..., 1], status=status)

    # ---- arbitrary rays ------------------------------------------------------------------
    def trace3d_rays(self, y0, x0, u0, v0, arith=STRICT, opl=False):
        """-> (xv, yv, k, flags[, opl]); opl=True (EXTENSION) adds the optical path length to the last surface."""
        y0, x0, u0, v0 = _d(y0), _d(x0), _d(u0), _d(v0)
        N, ns = len(y0), self.rows - 1
        xv, yv, k = np.empty((ns, N)), np.empty((ns, N)), np.empty((3, N))
        fl = np.zeros(N, dtype=np.uint8)
        if not opl:
            self._ck(self.L.ort_trace3d_rays(self.h, N, _p(y0), _p(x0), _p(u0), _p(v0), int(arith), _p(xv),
                                             _p(yv), _p(k), fl.ctypes.data_as(_u8p)))
            return xv, yv, k, fl
        ol = np.empty(N)
        self._ck(self.L.ort_trace3d_rays_opl(self.h, N, _p(y0), _p(x0), _p(u0), _p(v0), int(arith), _p(xv),
                                             _p(yv), _p(k), fl.ctypes.data_as(_u8p), _p(ol)))
        return xv, yv, k, fl, ol

    def trace3d_rays_dev(self, N, d_y0, d_x0, d_u0, d_v0, d_xv=0, d_yv=0, d_k=0, d_flags=0, d_opl=0, arith=FAST, stream=0):
        """device-pointer form of trace3d_rays: xv / yv are [rows-1][N], k is [3][N]; 0 = output not wanted"""
        vp = lambda a: C.c_void_p(a or 0)
        self._ck(self.L.ort_trace3d_rays_dev(self.h, int(N), vp(d_y0), vp(d_x0), vp(d_u0), vp(d_v0), int(arith), vp(d_xv),
                                             vp(d_yv), vp(d_k), vp(d_flags), vp(d_opl), vp(stream)))

    def trace2d_batch(self, y0, U0, aspheric=False):
        y0, U0 = _d(y0), _d(U0)
        N, rows = len(y0), self.rows
        yo, Uo, ts = np.empty((rows, N)), np.empty((rows, N)), np.empty((rows, N))
        fl = np.zeros(N, dtype=np.uint8)
        self._ck(self.L.ort_trace2d_batch(self.h, N, _p(y0), _p(U0), int(bool(aspheric)), _p(yo), _p(Uo),
                                          _p(ts), fl.ctypes.data_as(_u8p)))
        return yo, Uo, ts, fl

    def aim2d(self, x_start, other, target, stop, vary_u=False, mode=1, tol=1.0, aspheric=False):
        """N secant solves on the device (one thread each): x such that y_stop(x) == target.
        mode 0: the reference's fixed-step iteration with |f| <= tol; mode 1: root polish, tol = scale."""
        x_start, other, target = np.broadcast_arrays(_d(np.atleast_1d(x_start)), _d(np.atleast_1d(other)),
                                                     _d(np.atleast_1d(target)))
        x_start, other, target = _d(x_start), _d(other), _d(target)
        N = len(x_start)
        out = np.empty(N)
        it = np.zeros(N, dtype=np.int32)
        self._ck(self.L.ort_aim2d(self.h, N, _p(x_start), _p(other), _p(target), int(stop), int(bool(vary_u)), int(mode),
                                  float(tol), int(bool(aspheric)), _p(out), it.ctypes.data_as(_i32p)))
        return out, it

    # ---- paraxial / transfer matrix ------------------------------------------------------
    def paraxial_batch(self, tau, phi, y0, w0, a=None, clip=False, arith=STRICT, table=False):
        tau, phi, y0, w0 = _d(tau), _d(phi), _d(y0), _d(w0)
        a_ = None if a is None else _d(a)
        k, N = len(tau), len(y0)
        y, w = np.empty(N), np.empty(N)
        ci = np.zeros(N, dtype=np.int32)
        ya = np.empty((k + 1, N)) if table else None
        wa = np.empty((k + 1, N)) if table else None
        self._ck(self.L.ort_paraxial_batch(self.h, k, _p(tau), _p(phi), _p(a_), int(bool(clip)), int(arith),
                                           N, _p(y0), _p(w0), _p(y), _p(w), ci.ctypes.data_as(_i32p),
                                           _p(ya), _p(wa)))
        return (y, w, ci, ya, wa) if table else (y, w, ci)

    def paraxial_batch_dev(self, tau, phi, N, d_y0, d_w0, d_y, d_w, d_ci=None, a=None, clip=False,
                           arith=FAST, stream=0):
        tau, phi = _d(tau), _d(phi)
        a_ = None if a is None else _d(a)
        self._ck(self.L.ort_paraxial_batch_dev(self.h, len(tau), _p(tau), _p(phi), _p(a_), int(bool(clip)),
                                               int(arith), int(N), C.c_void_p(d_y0), C.c_void_p(d_w0),
                                               C.c_void_p(d_y), C.c_void_p(d_w), C.c_void_p(d_ci or 0),
                                               None, None, C.c_void_p(stream)))

    def transfer_batch(self, M, tau, taup, v_in, reverse=False):
        """M: 2x2; v_in: (N, 2) rows [y, nu] (= Julia 2xN column-major)."""
        Mc = _d(np.asarray(M, dtype=np.float64).T.reshape(-1))
        v_in = _d(v_in)
        out = np.empty_like(v_in)
        self._ck(self.L.ort_transfer_batch(self.h, _p(Mc), float(tau), float(taup), int(bool(reverse)),
                                           v_in.shape[0], _p(v_in), _p(out)))
        return out

    def transfer_batch_dev(self, M, tau, taup, N, d_in, d_out, reverse=False, stream=0):
        Mc = _d(np.asarray(M, dtype=np.float64).T.reshape(-1))
        self._ck(self.L.ort_transfer_batch_dev(self.h, _p(Mc), float(tau), float(taup), int(bool(reverse)),
                                               int(N), C.c_void_p(d_in), C.c_void_p(d_out),
                                               C.c_void_p(stream)))

    # ---- candidates ----------------------------------------------------------------------
    def trace3d_candidates(self, RtnK, field, ys, xs, stop, a_stop, arith=FAST):
        RtnK = _d(RtnK)
        Cn, four, rows = RtnK.shape
        assert four == 4
        farr, _ = make_fields([field])
        ys, xs = _d(ys), _d(xs)
        out = np.empty((Cn, 4))
        self._ck(self.L.ort_trace3d_candidates(self.h, rows, Cn, _p(RtnK), farr, _p(ys), len(ys), _p(xs),
                                               len(xs), int(stop), float(a_stop), int(arith), _p(out)))
        return out

    def seidel_candidates(self, RtnK, a, h_prime, lam=587.5618e-6, dn=None, per_surface=False):
        """first-order solve + Seidel sums per candidate -> (C, 16) [, (C, 7, rows-1)]"""
        RtnK = _d(RtnK)
        Cn, four, rows = RtnK.shape
        assert four == 4
        a = _d(a)
        dn_ = None if dn is None else _d(dn)
        out = np.empty((Cn, 16))
        per = np.empty((Cn, 7, rows - 1)) if per_surface else None
        self._ck(self.L.ort_seidel_candidates(self.h, rows, Cn, _p(RtnK), _p(a), float(h_prime), float(lam), _p(dn_),
                                              _p(out), _p(per)))
        return (out, per) if per_surface else out

    def vignetting_candidates(self, RtnK, a, h_prime, a_vig=None):
        """vignetting(system, a) per candidate -> dict(M (C, k, 5), code (C, k), FOV (C, 3, 3), un (C,), stop (C,), f (C,))"""
        RtnK = _d(RtnK)
        Cn, four, rows = RtnK.shape
        k = rows - 1
        a = _d(a)
        av = None if a_vig is None else _d(a_vig)
        assert four == 4 and a.shape == (k,) and (av is None or av.shape == (k,))
        out = np.empty((Cn, 6 * k + VIG_TAIL), dtype=np.float64)
        self._ck(self.L.ort_vignetting_candidates(self.h, rows, Cn, _p(RtnK), _p(a), _p(av), float(h_prime), _p(out)))
        return dict(M=out[:, :5 * k].reshape(Cn, 5, k).transpose(0, 2, 1).copy(), code=np.nan_to_num(out[:, 5 * k:6 * k]).astype(np.int32),
                    FOV=out[:, 6 * k:6 * k + 9].reshape(Cn, 3, 3).copy(), un=out[:, 6 * k + 9] == 1.0,
                    stop=np.nan_to_num(out[:, 6 * k + 10]).astype(np.int32), f=out[:, 6 * k + 11].copy())

    def vignetting_candidates_dev(self, rows, Cn, d_RtnK, a, h_prime, d_out, a_vig=None, stream=0):
        a = _d(a)
        av = None if a_vig is None else _d(a_vig)
        self._ck(self.L.ort_vignetting_candidates_dev(self.h, int(rows), int(Cn), C.c_void_p(d_RtnK), _p(a), _p(av),
                                                      float(h_prime), C.c_void_p(d_out), C.c_void_p(stream)))

    def aim_candidates(self, RtnK, a, h_prime, H, aspheric=False):
        """per-candidate full_trace prelude -> (C, 24) records (see ort_b200.h: ort_aim_candidates)"""
        RtnK = _d(RtnK)
        Cn, four, rows = RtnK.shape
        assert four == 4
        a = _d(a)
        assert a.shape == (rows - 1,)
        out = np.empty((Cn, AIM_NOUT), dtype=np.float64)
        self._ck(self.L.ort_aim_candidates(self.h, rows, Cn, _p(RtnK), _p(a), float(h_prime), float(H), int(bool(aspheric)),
                                           _p(out)))
        return out

    def set_polynomials(self, coef=None):
        """EXTENSION: polynomial aspheric terms, coef[row][k] multiplies y^k (row 0 = object space); None clears.
        Call after set_layout (which clears them)."""
        if coef is None:
            self._ck(self.L.ort_set_polynomials(self.h, 0, 0, None))
            return
        c = _d(coef)
        assert c.ndim == 2 and c.shape[0] == self.rows
        self._ck(self.L.ort_set_polynomials(self.h, c.shape[0], c.shape[1], _p(c)))

    def aim_fields(self, surfaces, K, a, h_prime, Hs, aspheric=False):
        """full_trace prelude of ONE system at the relative fields Hs -> (n_fields, 24) records (ort_aim_fields)"""
        S = _d(surfaces)
        R, t, n = _d(S[:, 0]), _d(S[:, 1]), _d(S[:, 2])
        Kc = None if K is None else _d(K)
        a, Hs = _d(a), _d(np.atleast_1d(Hs))
        out = np.empty((len(Hs), AIM_NOUT), dtype=np.float64)
        self._ck(self.L.ort_aim_fields(self.h, len(R), _p(R), _p(t), _p(n), _p(Kc), _p(a), float(h_prime), _p(Hs), len(Hs),
                                       int(bool(aspheric)), _p(out)))
        return out

    def aim_candidates_dev(self, rows, Cn, d_RtnK, a, h_prime, H, d_out, aspheric=False, stream=0):
        a = _d(a)
        self._ck(self.L.ort_aim_candidates_dev(self.h, int(rows), int(Cn), C.c_void_p(d_RtnK), _p(a), float(h_prime),
                                               float(H), int(bool(aspheric)), C.c_void_p(d_out), C.c_void_p(stream)))

    def trace3d_candidates_aimed(self, RtnK, aim, ny, nx, arith=FAST):
        """every candidate over its own aimed pupil grid -> (C, 4) = n_kept, mean_x, mean_y, RMS"""
        RtnK = _d(RtnK)
        Cn, four, rows = RtnK.shape
        aim = _d(aim)
        assert four == 4 and aim.shape == (Cn, AIM_NOUT)
        out = np.empty((Cn, 4), dtype=np.float64)
        self._ck(self.L.ort_trace3d_candidates_aimed(self.h, rows, Cn, _p(RtnK), _p(aim), int(ny), int(nx), int(arith),
                                                     _p(out)))
        return out

    def trace3d_candidates_aimed_dev(self, rows, Cn, d_RtnK, d_aim, ny, nx, d_out, arith=FAST, stream=0):
        self._ck(self.L.ort_trace3d_candidates_aimed_dev(self.h, int(rows), int(Cn), C.c_void_p(d_RtnK), C.c_void_p(d_aim),
                                                         int(ny), int(nx), int(arith), C.c_void_p(d_out),
                                                         C.c_void_p(stream)))

    def seidel_candidates_dev(self, rows, Cn, d_RtnK, a, h_prime, d_out, lam=587.5618e-6, dn=None, stream=0):
        a = _d(a)
        dn_ = None if dn is None else _d(dn)
        self._ck(self.L.ort_seidel_candidates_dev(self.h, int(rows), int(Cn), C.c_void_p(d_RtnK), _p(a), float(h_prime),
                                                  float(lam), _p(dn_), C.c_void_p(d_out), None, C.c_void_p(stream)))

    def trace3d_candidates_dev(self, rows, Cn, d_RtnK, field, d_ys, ny, d_xs, nx, stop, a_stop, d_out,
                               arith=FAST, stream=0):
        farr, _ = make_fields([field])
        self._ck(self.L.ort_trace3d_candidates_dev(self.h, int(rows), int(Cn), C.c_void_p(d_RtnK), farr,
                                                   C.c_void_p(d_ys), int(ny), C.c_void_p(d_xs), int(nx),
                                                   int(stop), float(a_stop), int(arith), C.c_void_p(d_out),
                                                   C.c_void_p(stream)))
