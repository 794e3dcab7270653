"""form::Estimator (C++ host facade over the CUDA hot path) and the trace
replayer, as Python handles.  ``FORM`` mirrors the evalio pipeline class of the
reference's python/bindings.cpp."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi


class EstimatorBase:
    """Shared wrapper over the C API generated from form/capi_impl.hpp."""

    _prefix = "formhost_"

    def _lib(self):
        return _capi.host_lib()

    def _fn(self, name):
        return getattr(self._lib(), self._prefix + name)

    def _last_error(self) -> str:
        return (self._lib().formhost_last_error() or b"").decode()

    def __init__(self, params: _capi.EstParams):
        self.params = params
        self.rows, self.cols = params.hot.num_rows, params.hot.num_columns
        self._h = self._fn("est_create")(C.byref(params))
        if not self._h:
            raise RuntimeError(f"{self._prefix}est_create failed: {self._last_error()}")
        cap = self.rows * self.cols
        self._planar = np.zeros(cap, dtype=_capi.PLANAR_FEAT)
        self._point = np.zeros(cap, dtype=_capi.POINT_FEAT)

    def close(self):
        if getattr(self, "_h", None):
            self._fn("est_destroy")(self._h)
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

    def register_scan(self, scan: np.ndarray):
        """Estimator::register_scan: returns (planar, point) keypoints of the scan."""
        a, b = C.c_size_t(), C.c_size_t()
        rc = self._fn("est_register_scan")(self._h, _capi.ptr(scan), scan.shape[0],
                                           _capi.ptr(self._planar), self._planar.shape[0], C.byref(a),
                                           _capi.ptr(self._point), self._point.shape[0], C.byref(b))
        if rc != 0:
            raise RuntimeError(f"register_scan failed (rc={rc})")
        return self._planar[: a.value].copy(), self._point[: b.value].copy()

    def pose(self) -> np.ndarray:
        """Estimator::current_lidar_estimate as a POSE record."""
        out = np.zeros(1, dtype=_capi.POSE)
        self._fn("est_pose")(self._h, _capi.ptr(out))
        return out[0]

    def window(self) -> np.ndarray:
        out = np.zeros(256, dtype=_capi.SCAN_POSE)
        n = C.c_size_t()
        rc = self._fn("est_window")(self._h, _capi.ptr(out), out.shape[0], C.byref(n))
        assert rc == 0
        return out[: n.value].copy()

    def stats(self) -> dict:
        out = np.zeros(8, np.uint64)
        self._fn("est_stats")(self._h, _capi.ptr(out))
        names = ("optimize_calls", "lm_iterations", "linearize_calls", "error_calls",
                 "linearized_pairs", "error_pairs", "icp_iterations", "window_size")
        return {k: int(v) for k, v in zip(names, out)}

    def map(self):
        W = max(self.params.hot.max_window_scans, 64)
        pl = np.zeros(W * self.rows * 64, dtype=_capi.PLANAR_FEAT)
        pt = np.zeros(W * self.rows * 64, dtype=_capi.POINT_FEAT)
        a, b = C.c_size_t(), C.c_size_t()
        rc = self._fn("est_map")(self._h, _capi.ptr(pl), pl.shape[0], C.byref(a), _capi.ptr(pt),
                                 pt.shape[0], C.byref(b))
        if rc != 0:
            raise RuntimeError(f"map failed (rc={rc})")
        return pl[: a.value].copy(), pt[: b.value].copy()

    def trace(self):
        return self._fn("est_trace")(self._h)

    def trace_num_scans(self) -> int:
        return int(self._fn("trace_num_scans")(self.trace()))


class Estimator(EstimatorBase):
    """form::Estimator on the CUDA hot path (libformhost.so + libformgpu.so)."""

    def ctx(self):
        return self._lib().formhost_est_ctx(self._h)


def _scan_ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))(*ptrs)
    return arr


class ReplayBase:
    _prefix = "formhost_"

    def _lib(self):
        return _capi.host_lib()

    def _fn(self, name):
        return getattr(self._lib(), self._prefix + name)

    def close(self):
        if getattr(self, "_h", None):
            self._fn("replay_destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run_host(self, first: int, last: int, scans) -> float:
        """Replay scans [first, last) with host scans (list of POINT4F arrays)."""
        arr = _scan_ptr_array([s.ctypes.data for s in scans])
        t = self._fn("replay_run_host")(self._h, first, last, arr)
        if t < 0:
            raise RuntimeError("replay failed")
        return t

    def stats(self) -> dict:
        out = np.zeros(20, np.uint64)
        cs = C.c_double()
        self._fn("replay_stats")(self._h, _capi.ptr(out), C.byref(cs))
        d = {k: int(v) for k, v in zip(_capi.REPLAY_STAT_NAMES, out)}
        d["checksum"] = cs.value
        return d

    def reset_stats(self):
        self._fn("replay_reset_stats")(self._h)


class Replay(ReplayBase):
    """Replays a recorded hot-path trace on a fresh CUDA context."""

    def __init__(self, trace, params: _capi.EstParams, stream: int | None = None):
        self._h = self._lib().formhost_replay_create(trace, C.byref(params), C.c_void_p(stream or 0))
        if not self._h:
            raise RuntimeError("formhost_replay_create failed: " +
                               (self._lib().formhost_last_error() or b"").decode())

    def ctx(self):
        return self._lib().formhost_replay_ctx(self._h)

    def run_device(self, first: int, last: int, dev_ptrs) -> float:
        arr = _scan_ptr_array(list(dev_ptrs))
        t = self._lib().formhost_replay_run_device(self._h, first, last, arr)
        if t < 0:
            raise RuntimeError("replay failed: " + (self._lib().formhost_last_error() or b"").decode())
        return t

    def profile_enable(self, on=True):
        _capi.gpu_lib().formgpu_profile_enable(self.ctx(), int(on))

    def profile_read(self):
        ms = np.zeros(_capi.KG_COUNT)
        launches = np.zeros(_capi.KG_COUNT, np.uint64)
        _capi.gpu_lib().formgpu_profile_read(self.ctx(), _capi.ptr(ms), _capi.ptr(launches))
        return {name: dict(ms=float(ms[i]), launches=int(launches[i]))
                for i, name in enumerate(_capi.KG_NAMES)}

    def launch_count(self) -> int:
        return int(_capi.gpu_lib().formgpu_launch_count(self.ctx()))


def run_device_multi(replays, first: int, last: int, dev_ptrs_per_replay) -> float:
    """Replay scans [first, last) of several sequences concurrently on one GPU (one host
    thread, context and stream per sequence).  Returns the wall time in seconds."""
    n = len(replays)
    handles = (C.c_void_p * n)(*[r._h for r in replays])
    arrays = [_scan_ptr_array(list(p)) for p in dev_ptrs_per_replay]
    outer = (C.c_void_p * n)(*[C.cast(a, C.c_void_p) for a in arrays])
    t = _capi.host_lib().formhost_replay_run_device_multi(handles, n, first, last, outer)
    if t < 0:
        raise RuntimeError("multi-sequence replay failed")
    return t


class BatchReplay:
    """Lock-step replay of the recorded traces of several sequences through
    formgpu_batch_submit: calls of the same kind share one launch per kernel."""

    def __init__(self, traces, params: _capi.EstParams, stream: int | None = None):
        self._lib = _capi.host_lib()
        self.n = len(traces)
        arr = (C.c_void_p * self.n)(*traces)
        self._h = self._lib.formhost_batch_replay_create(arr, self.n, C.byref(params), C.c_void_p(stream or 0))
        if not self._h:
            raise RuntimeError("formhost_batch_replay_create failed: " +
                               (self._lib.formhost_last_error() or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.formhost_batch_replay_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _scan_table(ptrs_per_sequence):
        inner = [_scan_ptr_array(list(p)) for p in ptrs_per_sequence]
        outer = (C.c_void_p * len(inner))(*[C.cast(a, C.c_void_p) for a in inner])
        return inner, outer

    def run(self, first: int, last: int, ptrs_per_sequence, on_device: bool = True):
        """Replay scans [first, last) of every sequence; returns (seconds, submits)."""
        keep, outer = self._scan_table(ptrs_per_sequence)
        rounds = C.c_size_t()
        t = self._lib.formhost_batch_replay_run(self._h, first, last, outer, int(on_device), C.byref(rounds))
        if t < 0:
            raise RuntimeError("batched replay failed: " + (self._lib.formhost_last_error() or b"").decode())
        return t, rounds.value

    def batch(self):
        return self._lib.formhost_batch_replay_batch(self._h)

    def stats(self, seq: int = -1) -> dict:
        out = np.zeros(20, np.uint64)
        cs = C.c_double()
        self._lib.formhost_batch_replay_stats(self._h, seq, _capi.ptr(out), C.byref(cs))
        d = {k: int(v) for k, v in zip(_capi.REPLAY_STAT_NAMES, out)}
        d["checksum"] = cs.value
        return d

    def reset_stats(self):
        self._lib.formhost_batch_replay_reset_stats(self._h)

    def capture_last_scan(self, seq: int, on=True):
        """on: every later run keeps what the calls of its last scan return for sequence `seq`
        (see captured)."""
        self._lib.formhost_batch_replay_capture(self._h, seq, int(on))

    def captured(self, seq: int) -> dict:
        """What the calls of the last scan of sequence `seq` returned in the latest run with
        capture on, in call order: pair counts of every association, 91-double blocks of every
        linearisation, error values, keypoint counts (extracted, then committed) and - for host
        scans - the keypoints."""
        out = {}
        for what, (name, dtype, width) in enumerate((
                ("counts", _capi.PAIR_COUNT, 1), ("blocks", np.float64, 91), ("errors", np.float64, 1),
                ("planar", _capi.PLANAR_FEAT, 1), ("point", _capi.POINT_FEAT, 1), ("keypoint_counts", np.uint64, 1))):
            n = self._lib.formhost_batch_replay_captured(self._h, seq, what, None, 0)
            a = np.zeros(n, dtype=dtype)
            self._lib.formhost_batch_replay_captured(self._h, seq, what, _capi.ptr(a), n)
            out[name] = a.reshape(-1, width) if width > 1 else a
        return out

    def profile_enable(self, on=True):
        _capi.gpu_lib().formgpu_batch_profile_enable(self.batch(), int(on))

    def profile_read(self):
        ms = np.zeros(_capi.KG_COUNT)
        launches = np.zeros(_capi.KG_COUNT, np.uint64)
        _capi.gpu_lib().formgpu_batch_profile_read(self.batch(), _capi.ptr(ms), _capi.ptr(launches))
        return {name: dict(ms=float(ms[i]), launches=int(launches[i]))
                for i, name in enumerate(_capi.KG_NAMES)}

    def launch_count(self) -> int:
        return int(_capi.gpu_lib().formgpu_batch_launch_count(self.batch()))


def run_batches(batch_replays, first: int, last: int, ptrs_per_batch, on_device: bool = True,
                threads: int = 0) -> float:
    """Several BatchReplay objects concurrently on one GPU (one stream per batch), driven by
    `threads` host threads (0: one per batch).  A thread that owns several batches queues a
    round on each of them (formgpu_batch_submit_async) before it waits for the first."""
    n = len(batch_replays)
    handles = (C.c_void_p * n)(*[b._h for b in batch_replays])
    keep = [BatchReplay._scan_table(p) for p in ptrs_per_batch]
    outer = (C.c_void_p * n)(*[C.cast(k[1], C.c_void_p) for k in keep])
    t = _capi.host_lib().formhost_batch_replay_run_pipelined(handles, n, threads, first, last, outer,
                                                             int(on_device))
    if t < 0:
        raise RuntimeError("batched replay failed: " + (_capi.host_lib().formhost_last_error() or b"").decode())
    return t


class EstimatorPool:
    """Many live form::Estimators on one GPU behind a batching dispatcher
    (form/batch_dispatch.hpp): the hot-path calls of the pool's sequences are funnelled
    through formgpu_batch_submit, so calls of the same kind share one launch per kernel.
    Drive each estimator from its own thread (ctypes releases the GIL inside a call)."""

    def __init__(self, params: _capi.EstParams, n_sequences: int, linger_us: int = 200):
        self._lib = _capi.host_lib()
        self.params = params
        self.n = n_sequences
        self._h = self._lib.formhost_pool_create(C.byref(params), n_sequences, linger_us)
        if not self._h:
            raise RuntimeError("formhost_pool_create failed: " + (self._lib.formhost_last_error() or b"").decode())
        self.estimators = [PooledEstimator(self, i) for i in range(n_sequences)]

    def stats(self) -> dict:
        out = np.zeros(2, np.uint64)
        self._lib.formhost_pool_stats(self._h, _capi.ptr(out))
        return {"submits": int(out[0]), "requests": int(out[1])}

    def close(self):
        for e in getattr(self, "estimators", []):
            e.close()
        self.estimators = []
        if getattr(self, "_h", None):
            self._lib.formhost_pool_destroy(self._h)
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


class PooledEstimator(EstimatorBase):
    """form::Estimator of one sequence of an EstimatorPool (same calls as Estimator)."""

    def __init__(self, pool: EstimatorPool, seq: int):
        self.params = pool.params
        self.rows, self.cols = pool.params.hot.num_rows, pool.params.hot.num_columns
        self._h = pool._lib.formhost_pool_est_create(pool._h, C.byref(pool.params), seq)
        if not self._h:
            raise RuntimeError("formhost_pool_est_create failed: " + self._last_error())
        cap = self.rows * self.cols
        self._planar = np.zeros(cap, dtype=_capi.PLANAR_FEAT)
        self._point = np.zeros(cap, dtype=_capi.POINT_FEAT)
