"""Python handle on one formgpu context (one sequence on one GPU).

Every method is a single call through the C-ABI of ``include/formgpu.h``;
numpy arrays are passed as raw host buffers.  There is no fallback: a missing
library raises ImportError, a missing GPU raises FormGpuError(ERR_CUDA).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi


class FormGpuError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"formgpu error {code}: {message}")
        self.code = code


class Context:
    def __init__(self, params: _capi.Params | None = None, device: int = 0, stream: int | None = None):
        self._lib = _capi.gpu_lib()
        self.params = params if params is not None else _capi.default_params()
        self.rows, self.cols = self.params.num_rows, self.params.num_columns
        h = C.c_void_p()
        rc = self._lib.formgpu_create(C.byref(self.params), device, C.c_void_p(stream or 0), C.byref(h))
        if rc != 0:
            raise FormGpuError(rc, (self._lib.formgpu_last_error(None) or b"").decode())
        self._h = h
        # cudaStream_t the context's work is ordered on (None: a private stream of its own)
        self.stream_handle = stream or None
        self.max_planar = self._lib.formgpu_max_planar(h)
        self.max_point = self._lib.formgpu_max_point(h)
        self._planar_buf = np.zeros(self.max_planar, dtype=_capi.PLANAR_FEAT)
        self._point_buf = np.zeros(self.max_point, dtype=_capi.POINT_FEAT)

    # -- lifecycle ---------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.formgpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise FormGpuError(rc, (self._lib.formgpu_last_error(self._h) or b"").decode())

    # -- stage 1 -----------------------------------------------------------------
    def extract(self, scan: np.ndarray, scan_idx: int):
        """FeatureExtractor::extract on a host scan; returns (planar, point) records."""
        npl, npt = C.c_size_t(), C.c_size_t()
        self._check(self._lib.formgpu_extract(
            self._h, _capi.ptr(scan), scan.shape[0], scan_idx,
            _capi.ptr(self._planar_buf), self.max_planar, C.byref(npl),
            _capi.ptr(self._point_buf), self.max_point, C.byref(npt)))
        return self._planar_buf[: npl.value].copy(), self._point_buf[: npt.value].copy()

    # -- raw clouds (rule R8) ----------------------------------------------------------
    def set_cloud_format(self, fmt: _capi.CloudFormat):
        """formgpu_set_cloud_format: the record layout of the clouds organize / extract_cloud take."""
        self._check(self._lib.formgpu_set_cloud_format(self._h, C.byref(fmt)))
        self.cloud_format = fmt

    def organize(self, records: np.ndarray):
        """formgpu_organize: -> (scan (rows*cols,) POINT4F, stats CLOUD_STATS record)."""
        records = np.ascontiguousarray(records)
        scan = np.zeros(self.rows * self.cols, dtype=_capi.POINT4F)
        stats = np.zeros(1, dtype=_capi.CLOUD_STATS)
        self._check(self._lib.formgpu_organize(self._h, _capi.ptr(records), len(records), _capi.ptr(scan),
                                               _capi.ptr(stats)))
        return scan, stats[0]

    def extract_cloud(self, records: np.ndarray, scan_idx: int):
        """formgpu_extract_cloud: extract() of a raw cloud; returns (planar, point) records."""
        records = np.ascontiguousarray(records)
        npl, npt = C.c_size_t(), C.c_size_t()
        self._check(self._lib.formgpu_extract_cloud(
            self._h, _capi.ptr(records), len(records), scan_idx,
            _capi.ptr(self._planar_buf), self.max_planar, C.byref(npl),
            _capi.ptr(self._point_buf), self.max_point, C.byref(npt)))
        return self._planar_buf[: npl.value].copy(), self._point_buf[: npt.value].copy()

    def cloud_stats(self):
        """formgpu_cloud_stats_last as a CLOUD_STATS record."""
        stats = np.zeros(1, dtype=_capi.CLOUD_STATS)
        self._check(self._lib.formgpu_cloud_stats_last(self._h, _capi.ptr(stats)))
        return stats[0]

    def extract_device(self, scan_dev_ptr: int, n: int, scan_idx: int):
        npl, npt = C.c_size_t(), C.c_size_t()
        self._check(self._lib.formgpu_extract_device(self._h, C.c_void_p(scan_dev_ptr), n, scan_idx,
                                                     C.byref(npl), C.byref(npt)))
        return npl.value, npt.value

    def extract_debug(self):
        n = self.rows * self.cols
        valid = np.zeros(n, np.uint8)
        pvalid = np.zeros(n, np.uint8)
        curv = np.zeros(n, np.float32)
        pidx = np.zeros(n, np.uint32)
        keep = np.zeros(n, np.uint8)
        cprev = np.zeros(n, np.int32)
        cnext = np.zeros(n, np.int32)
        qidx = np.zeros(n, np.uint32)
        npk, nqk = C.c_size_t(), C.c_size_t()
        self._check(self._lib.formgpu_extract_debug(
            self._h, _capi.ptr(valid), _capi.ptr(pvalid), _capi.ptr(curv), _capi.ptr(pidx),
            _capi.ptr(keep), _capi.ptr(cprev), _capi.ptr(cnext), C.byref(npk), _capi.ptr(qidx),
            C.byref(nqk)))
        k, q = npk.value, nqk.value
        return dict(valid=valid, point_valid=pvalid, curvature=curv, planar_indices=pidx[:k],
                    planar_keep=keep[:k], closest_prev=cprev[:k], closest_next=cnext[:k],
                    point_indices=qidx[:q])

    # -- stage 2 -----------------------------------------------------------------
    def map_rebuild(self, poses: np.ndarray):
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        self._check(self._lib.formgpu_map_rebuild(self._h, _capi.ptr(poses), poses.shape[0]))

    def associate(self, pose) -> np.ndarray:
        pose = np.ascontiguousarray(pose)
        out = np.zeros(max(self.params.max_window_scans, 1), dtype=_capi.PAIR_COUNT)
        n = C.c_size_t()
        self._check(self._lib.formgpu_associate(self._h, _capi.ptr(pose), _capi.ptr(out), out.shape[0],
                                                C.byref(n)))
        return out[: n.value].copy()

    def associate_linearize(self, poses: np.ndarray):
        """One round trip: Matcher::match at the current scan's pose in `poses`, then the
        blocks of every non-empty pair (i, current scan).  Returns (counts, blocks)."""
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        cap = max(self.params.max_window_scans, 1)
        out = np.zeros(cap, dtype=_capi.PAIR_COUNT)
        blocks = np.zeros((cap, 91))
        n = C.c_size_t()
        self._check(self._lib.formgpu_associate_linearize(self._h, _capi.ptr(poses), poses.shape[0],
                                                          _capi.ptr(out), cap, C.byref(n), _capi.ptr(blocks)))
        return out[: n.value].copy(), blocks[: n.value].copy()

    def matches(self, type_: int) -> np.ndarray:
        cap = self.max_planar if type_ == 0 else self.max_point
        out = np.zeros(cap, dtype=_capi.MATCH)
        n = C.c_size_t()
        self._check(self._lib.formgpu_get_matches(self._h, type_, _capi.ptr(out), cap, C.byref(n)))
        return out[: n.value].copy()

    def commit_scan(self):
        a, b = C.c_size_t(), C.c_size_t()
        self._check(self._lib.formgpu_commit_scan(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def remove_scans(self, scans):
        s = np.ascontiguousarray(scans, dtype=np.uint64)
        self._check(self._lib.formgpu_remove_scans(self._h, _capi.ptr(s), s.shape[0]))

    def keypoints(self, type_: int, scan: int) -> np.ndarray:
        n = C.c_size_t()
        self._check(self._lib.formgpu_get_keypoints(self._h, type_, scan, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=_capi.PLANAR_FEAT if type_ == 0 else _capi.POINT_FEAT)
        if n.value:
            self._check(self._lib.formgpu_get_keypoints(self._h, type_, scan, _capi.ptr(out), n.value,
                                                        C.byref(n)))
        return out

    def world_keypoints(self, poses: np.ndarray):
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        W = self.params.max_window_scans
        pl = np.zeros(W * self.max_planar, dtype=_capi.PLANAR_FEAT)
        pt = np.zeros(W * self.max_point, dtype=_capi.POINT_FEAT)
        a, b = C.c_size_t(), C.c_size_t()
        self._check(self._lib.formgpu_world_keypoints(self._h, _capi.ptr(poses), poses.shape[0],
                                                      _capi.ptr(pl), pl.shape[0], C.byref(a),
                                                      _capi.ptr(pt), pt.shape[0], C.byref(b)))
        return pl[: a.value].copy(), pt[: b.value].copy()

    # -- stage 3 -----------------------------------------------------------------
    def linearize(self, pairs: np.ndarray, poses: np.ndarray) -> np.ndarray:
        pairs = np.ascontiguousarray(pairs, dtype=_capi.PAIR)
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        out = np.zeros((pairs.shape[0], 91))
        self._check(self._lib.formgpu_linearize(self._h, _capi.ptr(pairs), pairs.shape[0], _capi.ptr(poses),
                                                poses.shape[0], _capi.ptr(out)))
        return out

    def error(self, pairs: np.ndarray, poses: np.ndarray) -> np.ndarray:
        pairs = np.ascontiguousarray(pairs, dtype=_capi.PAIR)
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        out = np.zeros(pairs.shape[0])
        self._check(self._lib.formgpu_error(self._h, _capi.ptr(pairs), pairs.shape[0], _capi.ptr(poses),
                                            poses.shape[0], _capi.ptr(out)))
        return out

    # -- point-sharded mode ----------------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        """formgpu_comm_unique_id: 128 bytes one rank creates and every rank passes to comm_init."""
        import ctypes as C

        buf = C.create_string_buffer(128)
        rc = _capi.gpu_lib().formgpu_comm_unique_id(buf)
        if rc != 0:
            raise RuntimeError(f"formgpu_comm_unique_id failed ({rc}): NCCL not available?")
        return buf.raw

    def comm_init(self, unique_id: bytes, rank: int, world: int):
        """formgpu_comm_init: make this context rank `rank` of a point-sharded sequence (collective)."""
        import ctypes as C

        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self._lib.formgpu_comm_init(self._h, buf, rank, world))

    def comm_destroy(self):
        self._check(self._lib.formgpu_comm_destroy(self._h))

    def set_shard(self, rank: int, world: int):
        """Stage-3 calls reduce only the rank-th of `world` shares of every pair (the caller
        sums the blocks over the ranks); (0, 1) switches the mode off."""
        self._check(self._lib.formgpu_set_shard(self._h, rank, world))

    def linearize_device(self, pairs: np.ndarray, poses: np.ndarray, out_dev_ptr: int):
        """formgpu_linearize_device: blocks into device memory at out_dev_ptr (91 doubles per
        pair), queued on the context's stream, nothing is waited for."""
        pairs = np.ascontiguousarray(pairs, dtype=_capi.PAIR)
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        self._check(self._lib.formgpu_linearize_device(self._h, _capi.ptr(pairs), pairs.shape[0],
                                                       _capi.ptr(poses), poses.shape[0], C.c_void_p(out_dev_ptr)))

    def error_device(self, pairs: np.ndarray, poses: np.ndarray, out_dev_ptr: int):
        pairs = np.ascontiguousarray(pairs, dtype=_capi.PAIR)
        poses = np.ascontiguousarray(poses, dtype=_capi.SCAN_POSE)
        self._check(self._lib.formgpu_error_device(self._h, _capi.ptr(pairs), pairs.shape[0],
                                                   _capi.ptr(poses), poses.shape[0], C.c_void_p(out_dev_ptr)))

    # -- instrumentation -----------------------------------------------------------
    def profile_enable(self, on: bool = True):
        self._check(self._lib.formgpu_profile_enable(self._h, int(on)))

    def profile_read(self):
        ms = np.zeros(_capi.KG_COUNT)
        launches = np.zeros(_capi.KG_COUNT, np.uint64)
        self._check(self._lib.formgpu_profile_read(self._h, _capi.ptr(ms), _capi.ptr(launches)))
        return {name: dict(ms=float(ms[i]), launches=int(launches[i]))
                for i, name in enumerate(_capi.KG_NAMES)}

    def launch_count(self) -> int:
        return int(self._lib.formgpu_launch_count(self._h))

    def synchronize(self):
        self._check(self._lib.formgpu_synchronize(self._h))
