"""Kernel variants that only batched submits use: the many-row extraction kernels (192-thread
select CTAs, thread-per-pick normals; kernels.hpp: kManyRowsMin, FORMGPU_MANY_ROWS_MIN) and, above
that threshold, the latency-shaped ones.  Keypoints - normals included - are compared bit for bit
with the CPU oracle on the synthetic sensor shapes, parameter variants and the edge-case scans of
test_gpu_extract."""
import ctypes as C
import zlib

import numpy as np
import pytest

from form_b200 import _capi, synth
from test_gpu_extract import _random_scan

pytestmark = pytest.mark.gpu


@pytest.fixture
def many_rows(monkeypatch):
    monkeypatch.setenv("FORMGPU_MANY_ROWS_MIN", "1")  # read by formgpu_batch_create


def _batch_extract_vs_oracle(params, scans, rows, cols):
    import oracle_lib

    lib = _capi.gpu_lib()
    n = len(scans)
    h = C.c_void_p()
    assert lib.formgpu_batch_create(C.byref(params), 0, None, n, C.byref(h)) == 0
    try:
        cap_p = lib.formgpu_max_planar(lib.formgpu_batch_ctx(h, 0))
        cap_q = lib.formgpu_max_point(lib.formgpu_batch_ctx(h, 0))
        planar = [np.zeros(cap_p, _capi.PLANAR_FEAT) for _ in range(n)]
        point = [np.zeros(cap_q, _capi.POINT_FEAT) for _ in range(n)]
        reqs = (_capi.Request * n)()
        for s in range(n):
            reqs[s].sequence, reqs[s].op = s, _capi.OP_EXTRACT
            reqs[s].scan, reqs[s].n_points, reqs[s].scan_idx = scans[s].ctypes.data, rows * cols, 3 + s
            reqs[s].planar_out, reqs[s].planar_cap = planar[s].ctypes.data, cap_p
            reqs[s].point_out, reqs[s].point_cap = point[s].ctypes.data, cap_q
        assert lib.formgpu_batch_submit(h, reqs, n) == 0, lib.formgpu_batch_last_error(h)
        ref = oracle_lib.Oracle(params)
        counts = []
        for s in range(n):
            rp, rq = ref.extract(scans[s], 3 + s)
            assert reqs[s].status == 0
            assert reqs[s].n_planar == len(rp) and reqs[s].n_point == len(rq), (s, reqs[s].n_planar, len(rp))
            assert planar[s][: len(rp)].tobytes() == rp.tobytes(), f"planar keypoints of scan {s} not bit-exact"
            assert point[s][: len(rq)].tobytes() == rq.tobytes(), f"point keypoints of scan {s} not bit-exact"
            counts.append((len(rp), len(rq)))
        return counts
    finally:
        lib.formgpu_batch_destroy(h)


@pytest.mark.parametrize("sensor", ["os1-64", "os0-128", "vlp-16", "stress-128x2048"])
def test_many_row_kernels_match_oracle_on_synthetic(many_rows, sensor):
    rows, cols = synth.shape(sensor)
    params = _capi.default_params(rows, cols)
    scans = [synth.scan(sensor, s, k) for s, k in ((0, 0), (2, 31), (5, 57))]
    counts = _batch_extract_vs_oracle(params, scans, rows, cols)
    assert all(p > 100 and q > 10 for p, q in counts)


@pytest.mark.parametrize("overrides", [
    dict(point_feats_per_sector=0),
    dict(planar_feats_per_sector=5, point_feats_per_sector=10),
    dict(neighbor_points=3, num_sectors=4, min_points=8),
    dict(neighbor_points=8, num_sectors=7, planar_threshold=0.05, radius=0.3),
    dict(min_norm_squared=0.01, radius=5.0),
])
def test_many_row_kernels_parameter_variants(many_rows, overrides):
    rows, cols = synth.shape("os1-64")
    params = _capi.default_params(rows, cols, **overrides)
    _batch_extract_vs_oracle(params, [synth.scan("os1-64", 1, 11), synth.scan("os1-64", 4, 2)], rows, cols)


@pytest.mark.parametrize("shape", [(4, 64), (7, 333), (16, 1800), (3, 2048), (1, 512)])
def test_many_row_kernels_edge_cases(many_rows, shape):
    rows, cols = shape
    params = _capi.default_params(rows, cols)
    scans = []
    for kind in ("noise", "ties", "dropouts", "all_invalid", "smooth"):
        rng = np.random.default_rng(zlib.crc32(f"many-{kind}-{rows}-{cols}".encode()))
        scans.append(_random_scan(rng, rows, cols, kind))
    _batch_extract_vs_oracle(params, scans, rows, cols)


def test_large_and_single_scan_batches_match_oracle():
    """Default threshold (kManyRowsMin): a 5 x 64-row batch and a single-scan batch both give the
    oracle's bytes."""
    rows, cols = synth.shape("os1-64")
    params = _capi.default_params(rows, cols)
    scans = [synth.scan("os1-64", s, 9) for s in range(5)]
    _batch_extract_vs_oracle(params, scans, rows, cols)
    _batch_extract_vs_oracle(params, scans[:1], rows, cols)


def test_few_row_variants_still_match_oracle(monkeypatch):
    """FORMGPU_MANY_ROWS_MIN above the launch's row count selects the latency-shaped variants
    (512-thread select CTAs, warp-per-pick normals on four CTAs per row) for a batched submit."""
    monkeypatch.setenv("FORMGPU_MANY_ROWS_MIN", "1000000")
    rows, cols = synth.shape("os1-64")
    params = _capi.default_params(rows, cols)
    _batch_extract_vs_oracle(params, [synth.scan("os1-64", s, 9) for s in range(3)], rows, cols)
    rng = np.random.default_rng(11)
    params = _capi.default_params(7, 333)
    _batch_extract_vs_oracle(params, [_random_scan(rng, 7, 333, k) for k in ("ties", "dropouts", "noise")], 7, 333)
