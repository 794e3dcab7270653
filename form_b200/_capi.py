"""ctypes view of the C-ABI in include/formgpu.h (and of libformhost's helpers).

Plain structs are mirrored as numpy dtypes so buffers cross the boundary
without copies.  Nothing here computes: it only declares prototypes and loads
the shared libraries built by ``__graft_entry__.build()`` / ``make``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "lib")

# ---- plain data (include/formgpu.h) ------------------------------------------
POINT4F = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("w", "<f4")])
POINT_FEAT = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("pad", "<f8"), ("scan", "<u8")])
PLANAR_FEAT = np.dtype(
    [("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("pad", "<f8"),
     ("nx", "<f8"), ("ny", "<f8"), ("nz", "<f8"), ("npad", "<f8"), ("scan", "<u8")]
)
POSE = np.dtype([("R", "<f8", (9,)), ("t", "<f8", (3,))])
SCAN_POSE = np.dtype([("scan", "<u8"), ("R", "<f8", (9,)), ("t", "<f8", (3,))])
PAIR = np.dtype([("i", "<u8"), ("j", "<u8")])
PAIR_COUNT = np.dtype([("i", "<u8"), ("n_planar", "<u4"), ("n_point", "<u4")])
MATCH = np.dtype([("scan", "<u8"), ("k", "<u4"), ("found", "<u4"), ("dist_sqrd", "<f8")])

assert POINT4F.itemsize == 16 and POINT_FEAT.itemsize == 40 and PLANAR_FEAT.itemsize == 72
assert POSE.itemsize == 96 and SCAN_POSE.itemsize == 104 and MATCH.itemsize == 24

KG_COUNT = 12
KG_NAMES = ("extract_select", "extract_normals", "extract_pack", "map_build", "assoc_nn", "segment",
            "lin_chunk", "lin_finalize", "err_chunk", "err_finalize", "commit", "export")

OK, ERR_INVALID_ARG, ERR_BAD_SCAN_SIZE, ERR_CAPACITY, ERR_CUDA, ERR_STATE, ERR_UNSUPPORTED = range(7)


class Params(C.Structure):
    """formgpu_params"""

    _fields_ = [
        ("neighbor_points", C.c_int32),
        ("num_sectors", C.c_int32),
        ("planar_feats_per_sector", C.c_int32),
        ("point_feats_per_sector", C.c_int32),
        ("min_points", C.c_int32),
        ("num_columns", C.c_int32),
        ("num_rows", C.c_int32),
        ("max_window_scans", C.c_int32),
        ("planar_threshold", C.c_double),
        ("radius", C.c_double),
        ("min_norm_squared", C.c_double),
        ("max_norm_squared", C.c_double),
        ("max_dist_matching", C.c_double),
        ("min_dist_map", C.c_double),
        ("sigma", C.c_double),
        ("max_batch_scans", C.c_int32),
        ("reserved", C.c_int32),
    ]


class EstParams(C.Structure):
    """formhost_est_params (form/capi_impl.hpp)"""

    _fields_ = [
        ("hot", Params),
        ("new_pose_threshold", C.c_double),
        ("keyscan_match_ratio", C.c_double),
        ("max_num_rematches", C.c_int32),
        ("disable_smoothing", C.c_int32),
        ("max_num_keyscans", C.c_int32),
        ("max_num_recent_scans", C.c_int32),
        ("max_steps_unused_keyscan", C.c_int32),
        ("num_threads", C.c_int32),
        ("device", C.c_int32),
        ("record_trace", C.c_int32),
        ("gtsam_lm_schedule", C.c_int32),
        ("reserved", C.c_int32),
    ]


class Request(C.Structure):
    """formgpu_request: one pending call of one sequence of a batch."""

    _fields_ = [
        ("sequence", C.c_uint32), ("op", C.c_uint32), ("flags", C.c_uint32), ("status", C.c_int32),
        ("scan", C.c_void_p), ("n_points", C.c_size_t), ("scan_idx", C.c_uint64),
        ("planar_out", C.c_void_p), ("planar_cap", C.c_size_t), ("n_planar", C.c_size_t),
        ("point_out", C.c_void_p), ("point_cap", C.c_size_t), ("n_point", C.c_size_t),
        ("poses", C.c_void_p), ("n_poses", C.c_size_t), ("pose_k", C.c_void_p),
        ("pairs", C.c_void_p), ("n_pairs", C.c_size_t),
        ("counts_out", C.c_void_p), ("counts_cap", C.c_size_t), ("n_counts", C.c_size_t),
        ("out", C.c_void_p), ("scans", C.c_void_p), ("n_scans", C.c_size_t),
    ]


(OP_EXTRACT, OP_MAP_REBUILD, OP_ASSOCIATE, OP_ASSOC_LIN, OP_LINEARIZE, OP_ERROR, OP_COMMIT,
 OP_REMOVE) = range(8)
REQ_SCAN_ON_DEVICE = 1
REQ_CLOUD = 2

# ---- raw sensor clouds (formgpu_cloud_format, rule R8) ---------------------------
CLOUD_ABSENT = -1
FIELD_F32, FIELD_F64, FIELD_U8, FIELD_U16, FIELD_U32, FIELD_U32_NS = range(6)
ROW_FROM_FIELD, ROW_FROM_ELEVATION = range(2)
COL_FROM_FIELD, COL_FROM_TIME, COL_FROM_AZIMUTH = range(3)
CLOUD_STATS = np.dtype([(k, "<u8") for k in (
    "records", "placed", "pixels", "dropped_nonfinite", "dropped_zero", "dropped_time", "dropped_row",
    "dropped_col")])


class CloudFormat(C.Structure):
    """formgpu_cloud_format: record layout of a raw cloud and how it is organised."""

    _fields_ = [
        ("stride", C.c_uint32), ("off_x", C.c_int32), ("off_y", C.c_int32), ("off_z", C.c_int32),
        ("xyz_type", C.c_int32), ("off_row", C.c_int32), ("row_type", C.c_int32), ("off_col", C.c_int32),
        ("col_type", C.c_int32), ("off_time", C.c_int32), ("time_type", C.c_int32), ("row_source", C.c_int32),
        ("col_source", C.c_int32), ("azimuth_dir", C.c_int32), ("scan_period", C.c_double),
        ("azimuth_origin", C.c_double), ("beam_elevations", C.POINTER(C.c_double)), ("max_records", C.c_uint64),
    ]

    def beams(self):
        """The beam-elevation table as a numpy array (None without one)."""
        b = getattr(self, "_beams", None)
        return None if b is None else np.array(b)


assert C.sizeof(CloudFormat) == 88

_ROW_FROM = {"field": ROW_FROM_FIELD, "ring": ROW_FROM_FIELD, "row": ROW_FROM_FIELD, "elevation": ROW_FROM_ELEVATION}
_COL_FROM = {"field": COL_FROM_FIELD, "col": COL_FROM_FIELD, "time": COL_FROM_TIME, "azimuth": COL_FROM_AZIMUTH}
_INDEX_TYPES = {np.dtype("u1"): FIELD_U8, np.dtype("<u2"): FIELD_U16, np.dtype("<u4"): FIELD_U32}


def cloud_format(dtype, *, row_from: str | None = None, col_from: str | None = None, scan_period: float = 0.1,
                 azimuth_origin: float = 0.0, azimuth_dir: int = 1, beams=None,
                 max_records: int = 1 << 20) -> CloudFormat:
    """formgpu_cloud_format of the records of a numpy structured dtype.  Fields by name: x, y, z
    (f4 or f8, all three alike), ring or row (u1/u2/u4), col (u1/u2/u4), t or time (f4/f8 seconds
    since the scan started, or u4 nanoseconds).  Row source: the ring / row field when there is one,
    else the beam-elevation table `beams` (radians, one per row, strictly monotonic).  Column source:
    the col field, else the time field, else the azimuth (column c centred at
    azimuth_origin + azimuth_dir * 2 pi c / cols).  `row_from` ("ring" | "elevation") and `col_from`
    ("col" | "time" | "azimuth") override the choice."""
    dt = np.dtype(dtype)
    names = dt.names or ()

    def field(*cands):
        for n in cands:
            if n in names:
                sub, off = dt.fields[n][0], dt.fields[n][1]
                if sub.shape:
                    raise ValueError(f"cloud field {n!r} must be a scalar")
                return n, sub, off
        return None, None, CLOUD_ABSENT

    xyz = [field(a) for a in "xyz"]
    if any(f[0] is None for f in xyz):
        raise ValueError(f"cloud records need fields x, y, z; got {names}")
    kinds = {f[1].newbyteorder("<") if f[1].byteorder == ">" else f[1] for f in xyz}
    if kinds == {np.dtype("<f4")}:
        xyz_type = FIELD_F32
    elif kinds == {np.dtype("<f8")}:
        xyz_type = FIELD_F64
    else:
        raise ValueError(f"x, y, z must all be float32 or all float64; got {sorted(map(str, kinds))}")
    if any(f[1].byteorder == ">" for f in xyz):
        raise ValueError("big-endian coordinates are not supported")
    rname, rtype, roff = field("ring", "row")
    cname, ctype, coff = field("col")
    tname, ttype, toff = field("t", "time")

    def index_type(name, sub):
        if sub is None:
            return 0
        if sub not in _INDEX_TYPES:
            raise ValueError(f"cloud field {name!r}: {sub} is not u1, u2 or u4")
        return _INDEX_TYPES[sub]

    if ttype is None:
        time_type = 0
    elif ttype == np.dtype("<f4"):
        time_type = FIELD_F32
    elif ttype == np.dtype("<f8"):
        time_type = FIELD_F64
    elif ttype == np.dtype("<u4"):
        time_type = FIELD_U32_NS
    else:
        raise ValueError(f"cloud field {tname!r}: {ttype} is not f4, f8 or u4 (nanoseconds)")
    if row_from is None:
        row_from = "ring" if rname else "elevation"
    if col_from is None:
        col_from = "col" if cname else ("time" if tname else "azimuth")
    if row_from not in _ROW_FROM:
        raise ValueError(f"row_from must be one of {sorted(_ROW_FROM)}, not {row_from!r}")
    if col_from not in _COL_FROM:
        raise ValueError(f"col_from must be one of {sorted(_COL_FROM)}, not {col_from!r}")
    f = CloudFormat(stride=dt.itemsize, off_x=xyz[0][2], off_y=xyz[1][2], off_z=xyz[2][2], xyz_type=xyz_type,
                    off_row=roff, row_type=index_type(rname, rtype), off_col=coff, col_type=index_type(cname, ctype),
                    off_time=toff, time_type=time_type, row_source=_ROW_FROM[row_from],
                    col_source=_COL_FROM[col_from], azimuth_dir=int(azimuth_dir), scan_period=float(scan_period),
                    azimuth_origin=float(azimuth_origin), max_records=int(max_records))
    if beams is not None:
        set_beams(f, beams)
    return f


def set_beams(fmt: CloudFormat, beams) -> None:
    """Point fmt.beam_elevations at a copy of `beams` (radians) that lives as long as fmt."""
    arr = (C.c_double * len(beams))(*[float(b) for b in beams])
    fmt._beams = arr
    fmt.beam_elevations = C.cast(arr, C.POINTER(C.c_double))


def check_cloud_format(fmt: CloudFormat, rows: int, cols: int) -> tuple[int, str]:
    """formgpu_cloud_format_check: (status, message); needs no GPU."""
    buf = C.create_string_buffer(512)
    rc = gpu_lib().formgpu_cloud_format_check(C.byref(fmt), rows, cols, buf, len(buf))
    return rc, buf.value.decode()


def default_est_params(rows: int = 64, cols: int = 1024, **overrides) -> EstParams:
    """Estimator::Params defaults (python/bindings.cpp:66-88 of FORM).  Keys of
    formgpu_params and of the estimator-level struct can both be overridden."""
    hot_keys = {f[0] for f in Params._fields_}
    hot = default_params(rows, cols, **{k: v for k, v in overrides.items() if k in hot_keys})
    p = EstParams(hot=hot, new_pose_threshold=1e-4, keyscan_match_ratio=0.1, max_num_rematches=30,
                  disable_smoothing=0, max_num_keyscans=50, max_num_recent_scans=10,
                  max_steps_unused_keyscan=10, num_threads=0, device=0, record_trace=0,
                  gtsam_lm_schedule=0, reserved=0)
    for k, v in overrides.items():
        if k in hot_keys:
            continue
        if not hasattr(p, k):
            raise AttributeError(f"formhost_est_params has no field {k!r}")
        setattr(p, k, v)
    return p


def default_params(rows: int = 64, cols: int = 1024, **overrides) -> Params:
    """Reference defaults (python/bindings.cpp:66-88 of FORM); pure Python so it
    also works where the CUDA library is not built."""
    p = Params(
        neighbor_points=5, num_sectors=6, planar_feats_per_sector=50, point_feats_per_sector=3,
        min_points=5, num_columns=cols, num_rows=rows, max_window_scans=64,
        planar_threshold=1.0, radius=1.0, min_norm_squared=1.0, max_norm_squared=1.0e4,
        max_dist_matching=0.8, min_dist_map=0.1, sigma=0.1, max_batch_scans=1, reserved=0,
    )
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(f"formgpu_params has no field {k!r}")
        setattr(p, k, v)
    return p


def ptr(a):
    """void* of a numpy array (None -> NULL)."""
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


_vp, _sz, _u64, _i = C.c_void_p, C.c_size_t, C.c_uint64, C.c_int
_psz = C.POINTER(C.c_size_t)

# name -> (restype, argtypes); exactly the symbols include/formgpu.h declares
FORMGPU_SYMBOLS = {
    "formgpu_default_params": (None, [C.POINTER(Params)]),
    "formgpu_create": (_i, [C.POINTER(Params), _i, _vp, C.POINTER(_vp)]),
    "formgpu_destroy": (None, [_vp]),
    "formgpu_last_error": (C.c_char_p, [_vp]),
    "formgpu_abi_version": (_i, []),
    "formgpu_extract": (_i, [_vp, _vp, _sz, _u64, _vp, _sz, _psz, _vp, _sz, _psz]),
    "formgpu_alloc_pinned": (_vp, [_sz]),
    "formgpu_free_pinned": (None, [_vp]),
    "formgpu_extract_device": (_i, [_vp, _vp, _sz, _u64, _psz, _psz]),
    "formgpu_max_planar": (_sz, [_vp]),
    "formgpu_max_point": (_sz, [_vp]),
    "formgpu_extract_debug": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _psz, _vp, _psz]),
    "formgpu_map_rebuild": (_i, [_vp, _vp, _sz]),
    "formgpu_associate": (_i, [_vp, _vp, _vp, _sz, _psz]),
    "formgpu_associate_linearize": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp]),
    "formgpu_get_matches": (_i, [_vp, _i, _vp, _sz, _psz]),
    "formgpu_commit_scan": (_i, [_vp, _psz, _psz]),
    "formgpu_remove_scans": (_i, [_vp, _vp, _sz]),
    "formgpu_get_keypoints": (_i, [_vp, _i, _u64, _vp, _sz, _psz]),
    "formgpu_world_keypoints": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp, _sz, _psz]),
    "formgpu_linearize": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "formgpu_error": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "formgpu_profile_enable": (_i, [_vp, _i]),
    "formgpu_profile_read": (_i, [_vp, _vp, _vp]),
    "formgpu_launch_count": (_u64, [_vp]),
    "formgpu_synchronize": (_i, [_vp]),
    "formgpu_set_shard": (_i, [_vp, _i, _i]),
    "formgpu_comm_unique_id": (_i, [_vp]),
    "formgpu_comm_init": (_i, [_vp, _vp, _i, _i]),
    "formgpu_comm_destroy": (_i, [_vp]),
    "formgpu_linearize_device": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "formgpu_error_device": (_i, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "formgpu_batch_create": (_i, [C.POINTER(Params), _i, _vp, _sz, C.POINTER(_vp)]),
    "formgpu_batch_create_mixed": (_i, [C.POINTER(Params), _i, _vp, _sz, C.POINTER(_vp)]),
    "formgpu_batch_destroy": (None, [_vp]),
    "formgpu_batch_size": (_sz, [_vp]),
    "formgpu_batch_ctx": (_vp, [_vp, _sz]),
    "formgpu_batch_submit": (_i, [_vp, _vp, _sz]),
    "formgpu_batch_submit_async": (_i, [_vp, _vp, _sz]),
    "formgpu_batch_wait": (_i, [_vp]),
    "formgpu_batch_done": (_i, [_vp]),
    "formgpu_batch_prefetch_scan": (_i, [_vp, _sz, _vp, _sz]),
    "formgpu_batch_last_error": (C.c_char_p, [_vp]),
    "formgpu_cloud_format_check": (_i, [_vp, _i, _i, _vp, _sz]),
    "formgpu_set_cloud_format": (_i, [_vp, _vp]),
    "formgpu_organize": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "formgpu_extract_cloud": (_i, [_vp, _vp, _sz, _u64, _vp, _sz, _psz, _vp, _sz, _psz]),
    "formgpu_cloud_stats_last": (_i, [_vp, _vp]),
    "formgpu_batch_prefetch_cloud": (_i, [_vp, _sz, _vp, _sz]),
    "formgpu_batch_profile_enable": (_i, [_vp, _i]),
    "formgpu_batch_profile_read": (_i, [_vp, _vp, _vp]),
    "formgpu_batch_launch_count": (_u64, [_vp]),
}

_pest = C.POINTER(EstParams)
_d = C.c_double


def estimator_symbols(prefix: str) -> dict:
    """The C API generated from form/capi_impl.hpp (prefix formhost_ or oracle_)."""
    return {
        f"{prefix}est_create": (_vp, [_pest]),
        f"{prefix}est_destroy": (None, [_vp]),
        f"{prefix}est_register_scan": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp, _sz, _psz]),
        f"{prefix}est_pose": (None, [_vp, _vp]),
        f"{prefix}est_window": (_i, [_vp, _vp, _sz, _psz]),
        f"{prefix}est_stats": (None, [_vp, _vp]),
        f"{prefix}est_map": (_i, [_vp, _vp, _sz, _psz, _vp, _sz, _psz]),
        f"{prefix}est_trace": (_vp, [_vp]),
        f"{prefix}trace_num_scans": (_sz, [_vp]),
        f"{prefix}replay_destroy": (None, [_vp]),
        f"{prefix}replay_run_host": (_d, [_vp, _sz, _sz, _vp]),
        f"{prefix}replay_stats": (None, [_vp, _vp, C.POINTER(_d)]),
        f"{prefix}replay_reset_stats": (None, [_vp]),
    }


# host/src/synth_capi.cpp: exported by libformsynth.so (no CUDA dependency) and by libformhost.so
FORMSYNTH_SYMBOLS = {
    "formhost_synth_shape": (_sz, [_i, C.POINTER(_i), C.POINTER(_i)]),
    "formhost_synth_scan": (_i, [_i, _u64, _u64, _vp, _i]),
    "formhost_synth_gt_pose": (None, [_u64, _u64, _vp]),
    "formhost_synth_stress_scan": (None, [_u64, _u64, _vp, _i]),
    "formhost_synth_stress_pose": (None, [_u64, _u64, _vp]),
    "formhost_pose_expmap": (None, [_vp, _vp]),
    "formhost_pose_logmap": (None, [_vp, _vp]),
    "formhost_pose_logmap_derivative": (None, [_vp, _vp]),
    "formhost_pose_compose": (None, [_vp, _vp, _vp]),
    "formhost_pose_inverse": (None, [_vp, _vp]),
    "formhost_pose_rzryrx": (None, [_d, _d, _d, _vp, _vp]),
    "formhost_pose_normalized": (None, [_vp, _vp]),
}

FORMHOST_SYMBOLS = {
    **FORMSYNTH_SYMBOLS,
    "formhost_default_est_params": (None, [_pest]),
    "formhost_last_error": (C.c_char_p, []),
    "formhost_est_error": (C.c_char_p, [_vp]),
    "formhost_est_ctx": (_vp, [_vp]),
    "formhost_trace_num_ops": (_sz, [_vp]),
    "formhost_replay_create": (_vp, [_vp, _pest, _vp]),
    "formhost_replay_ctx": (_vp, [_vp]),
    "formhost_replay_run_device": (_d, [_vp, _sz, _sz, _vp]),
    "formhost_replay_run_device_multi": (_d, [_vp, _sz, _sz, _sz, _vp]),
    "formhost_pool_create": (_vp, [_pest, _sz, _i]),
    "formhost_pool_create_mixed": (_vp, [_pest, _sz, _i]),
    "formhost_pool_destroy": (None, [_vp]),
    "formhost_pool_stats": (None, [_vp, _vp]),
    "formhost_pool_est_create": (_vp, [_vp, _pest, _sz]),
    "formhost_batch_replay_create": (_vp, [_vp, _sz, _pest, _vp]),
    "formhost_batch_replay_create_mixed": (_vp, [_vp, _sz, _pest, _vp]),
    "formhost_batch_replay_destroy": (None, [_vp]),
    "formhost_batch_replay_batch": (_vp, [_vp]),
    "formhost_batch_replay_run": (_d, [_vp, _sz, _sz, _vp, _i, _psz]),
    "formhost_batch_replay_run_multi": (_d, [_vp, _sz, _sz, _sz, _vp, _i]),
    "formhost_batch_replay_run_pipelined": (_d, [_vp, _sz, _sz, _sz, _sz, _vp, _i]),
    "formhost_batch_replay_stats": (None, [_vp, _i, _vp, C.POINTER(_d)]),
    "formhost_batch_replay_reset_stats": (None, [_vp]),
    "formhost_batch_replay_capture": (None, [_vp, _sz, _i]),
    "formhost_batch_replay_captured": (_sz, [_vp, _sz, _i, _vp, _sz]),
    "formhost_est_set_cloud_format": (_i, [_vp, _vp]),
    "formhost_est_register_cloud": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp, _sz, _psz]),
    "formhost_est_cloud_stats": (_i, [_vp, _vp]),
    **estimator_symbols("formhost_"),
}

REPLAY_STAT_NAMES = (
    "scans", "points", "planar_kp", "point_kp", "assoc_calls", "assoc_queries", "map_rebuilds",
    "map_points", "lin_calls", "lin_pairs", "lin_planar", "lin_point", "err_calls", "err_pairs",
    "err_planar", "err_point", "novel_planar", "novel_point", "assoc_planar", "assoc_point",
)


def _load(path: str, symbols: dict, mode: int = C.RTLD_GLOBAL) -> C.CDLL:
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make`) at the repository root"
        )
    lib = C.CDLL(path, mode=mode)
    for name, (res, args) in symbols.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    return lib


_gpu = None
_host = None
_synth = None
_load_lock = threading.RLock()  # callers load lazily, possibly from worker threads


def gpu_lib() -> C.CDLL:
    """libformgpu.so: the CUDA hot path behind the C-ABI.  No fallback."""
    global _gpu
    if _gpu is None:
        with _load_lock:
            if _gpu is None:
                _gpu = _load(os.path.join(LIB_DIR, "libformgpu.so"), FORMGPU_SYMBOLS)
    return _gpu


def synth_lib() -> C.CDLL:
    """libformsynth.so: the seeded scan generators and the SE(3) hooks of the host side, built
    without any CUDA dependency - what the CPU baseline and the oracle tests load, so that
    they never map the product's CUDA library."""
    global _synth
    if _synth is None:
        path = os.path.join(LIB_DIR, "libformsynth.so")
        if not os.path.exists(path) and os.path.exists(os.path.join(LIB_DIR, "libformhost.so")):
            return host_lib()  # a tree built before libformsynth existed: same symbols, same code
        with _load_lock:
            if _synth is None:
                _synth = _load(path, FORMSYNTH_SYMBOLS, C.DEFAULT_MODE)
    return _synth


def host_lib() -> C.CDLL:
    """libformhost.so: host-side C++ (synthetic scans, Estimator facade)."""
    global _host
    if _host is None:
        with _load_lock:
            if _host is None:
                gpu_lib()  # libformhost links against libformgpu
                _host = _load(os.path.join(LIB_DIR, "libformhost.so"), FORMHOST_SYMBOLS)
    return _host
