"""Mixed batches: sequences of different sensor shapes and hot-path parameters in ONE formgpu batch
(formgpu_batch_create_mixed).  Every sequence must compute exactly what its own single context
computes - index work bit-exact, blocks to 1e-12 - whether the batch is replayed from traces or
driven live by pooled estimators; one extraction launch serves all shapes and matches the oracle
bit for bit under both select-kernel variants; the sweep driver writes what stand-alone estimators
produce."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from form_b200 import _capi, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (sensor, sequence, hot-path overrides): three shapes, defaults and non-default parameters
MIXED = [
    ("vlp-16", 0, {}),
    ("vlp-16", 1, dict(num_sectors=4)),
    ("os1-64", 2, dict(num_sectors=8, neighbor_points=3)),
    ("os1-64", 3, dict(point_feats_per_sector=0)),
    ("os0-128", 4, dict(max_dist_matching=1.0, sigma=0.2)),
    ("os0-128", 5, {}),
]


def _same(got, ref, what):
    for k in ref:
        if k == "checksum":
            assert abs(got[k] - ref[k]) <= 1e-12 * abs(ref[k]), (what, k, got[k], ref[k])
        else:
            assert got[k] == ref[k], (what, k, got[k], ref[k])


def test_mixed_replay_matches_single_contexts():
    import torch

    from form_b200.pipeline import BatchReplay, Estimator, Replay

    n = 10
    params, traces, ests, scans = [], [], [], []
    for sensor, seq, ov in MIXED:
        p = _capi.default_est_params(*synth.shape(sensor), record_trace=1, **ov)
        sc = [synth.scan(sensor, seq, k) for k in range(n)]
        e = Estimator(p)
        for s in sc:
            e.register_scan(s)
        params.append(p)
        ests.append(e)
        traces.append(e.trace())
        scans.append(sc)
    dev = [[torch.from_numpy(s.view(np.uint8)).cuda() for s in sc] for sc in scans]
    torch.cuda.synchronize()
    dptrs = [[d.data_ptr() for d in seq] for seq in dev]
    hptrs = [[s.ctypes.data for s in sc] for sc in scans]
    singles = []
    for t, p, pp in zip(traces, params, dptrs):
        r = Replay(t, p)
        r.run_device(0, n, pp)
        singles.append(r.stats())
        r.close()
    assert len({st["points"] for st in singles}) == 3  # three shapes, each counted with its own size

    def check(br, what):
        for s, ref in enumerate(singles):
            _same(br.stats(s), ref, (what, MIXED[s]))

    bd = BatchReplay(traces, params)
    _, rounds = bd.run(0, n, dptrs, on_device=True)
    assert rounds > 0
    check(bd, "device")
    bd2 = BatchReplay(traces, params)
    bd2.run(0, n, dptrs, on_device=True)
    for s in range(len(MIXED)):
        assert bd2.stats(s) == bd.stats(s)  # run to run identical
    bh = BatchReplay(traces, params)
    bh.run(0, n, hptrs, on_device=False)  # host scans, next scan prefetched (default)
    check(bh, "host, prefetch")
    os.environ["FORM_REPLAY_PREFETCH"] = "0"
    try:
        bn = BatchReplay(traces, params)
        bn.run(0, n, hptrs, on_device=False)
    finally:
        del os.environ["FORM_REPLAY_PREFETCH"]
    check(bn, "host, no prefetch")
    for s in range(len(MIXED)):
        assert bn.stats(s) == bh.stats(s)
    # the homogeneous constructor is the mixed one with one params repeated
    same = BatchReplay(traces[:2], [params[0], params[0]])
    single_params = BatchReplay(traces[:2], params[0])
    same.run(0, n, dptrs[:2], on_device=True)
    single_params.run(0, n, dptrs[:2], on_device=True)
    assert same.stats(0) == single_params.stats(0) and same.stats(1) == single_params.stats(1)
    for b in (bd, bd2, bh, bn, same, single_params):
        b.close()
    for e in ests:
        e.close()


@pytest.mark.parametrize("many_rows_min", ["1", "100000000"])  # 192-thread many-row / 512-thread few-row select
def test_one_extraction_launch_of_three_shapes_matches_the_oracle(monkeypatch, many_rows_min):
    import oracle_lib

    monkeypatch.setenv("FORMGPU_MANY_ROWS_MIN", many_rows_min)  # read by formgpu_batch_create
    items = [("vlp-16", 0, {}), ("os1-64", 1, dict(num_sectors=8, planar_feats_per_sector=30)),
             ("os0-128", 2, {}), ("vlp-16", 3, dict(neighbor_points=3, point_feats_per_sector=0)),
             ("os1-64", 4, {})]
    params = [_capi.default_params(*synth.shape(sensor), **ov) for sensor, _, ov in items]
    scans = [synth.scan(sensor, seq, 2) for sensor, seq, _ in items]
    lib = _capi.gpu_lib()
    n = len(items)
    h = C.c_void_p()
    assert lib.formgpu_batch_create_mixed((_capi.Params * n)(*params), 0, None, n, C.byref(h)) == 0
    try:
        reqs = (_capi.Request * n)()
        outs = []
        for s in range(n):
            ctx = lib.formgpu_batch_ctx(h, s)
            cap_p, cap_q = lib.formgpu_max_planar(ctx), lib.formgpu_max_point(ctx)
            outs.append((np.zeros(cap_p, _capi.PLANAR_FEAT), np.zeros(cap_q, _capi.POINT_FEAT)))
            reqs[s].sequence, reqs[s].op = s, _capi.OP_EXTRACT
            reqs[s].scan, reqs[s].n_points, reqs[s].scan_idx = scans[s].ctypes.data, len(scans[s]), 7 + s
            reqs[s].planar_out, reqs[s].planar_cap = outs[s][0].ctypes.data, cap_p
            reqs[s].point_out, reqs[s].point_cap = outs[s][1].ctypes.data, cap_q
        lib.formgpu_batch_profile_read(h, None, None)
        launches = np.zeros(_capi.KG_COUNT, np.uint64)
        assert lib.formgpu_batch_submit(h, reqs, n) == 0, lib.formgpu_batch_last_error(h)
        lib.formgpu_batch_profile_read(h, None, _capi.ptr(launches))
        # ONE launch per extraction kernel for the whole mix of shapes
        assert [int(launches[g]) for g in range(3)] == [1, 1, 1]
        for s in range(n):
            rp, rq = oracle_lib.Oracle(params[s]).extract(scans[s], 7 + s)
            assert reqs[s].status == 0
            assert (reqs[s].n_planar, reqs[s].n_point) == (len(rp), len(rq)), items[s]
            assert outs[s][0][: len(rp)].tobytes() == rp.tobytes(), f"planar keypoints of {items[s]}"
            assert outs[s][1][: len(rq)].tobytes() == rq.tobytes(), f"point keypoints of {items[s]}"
        # a scan of another sequence's size is refused for this one
        reqs[0].n_points = len(scans[2])
        assert lib.formgpu_batch_submit(h, reqs, n) == _capi.ERR_BAD_SCAN_SIZE
        assert reqs[0].status == _capi.ERR_BAD_SCAN_SIZE and reqs[2].status == 0
    finally:
        lib.formgpu_batch_destroy(h)


def test_pooled_mixed_estimators_match_standalone_estimators():
    """2 sensors x 2 sequences x 3 variants (disable_smoothing among them), live, in ONE pool."""
    from concurrent.futures import ThreadPoolExecutor

    from form_b200.pipeline import Estimator, EstimatorPool

    n_scans = 8
    variants = [{}, dict(point_feats_per_sector=0), dict(disable_smoothing=1)]
    runs = [(sensor, seq, ov) for sensor in ("vlp-16", "os1-64") for seq in (0, 6) for ov in variants]
    params = [_capi.default_est_params(*synth.shape(sensor), **ov) for sensor, _, ov in runs]
    scans = {(sensor, seq): [synth.scan(sensor, seq, k) for k in range(n_scans)]
             for sensor in ("vlp-16", "os1-64") for seq in (0, 6)}
    alone = []
    for (sensor, seq, _), p in zip(runs, params):
        with Estimator(p) as e:
            kps = [e.register_scan(sc) for sc in scans[sensor, seq]]
            alone.append((kps, e.pose(), e.stats(), e.window()))
    with EstimatorPool(params) as pool:
        assert pool.n == len(runs)

        def drive(i):
            e = pool.estimators[i]
            kps = [e.register_scan(sc) for sc in scans[runs[i][0], runs[i][1]]]
            return kps, e.pose(), e.stats(), e.window()

        with ThreadPoolExecutor(len(runs)) as ex:
            pooled = list(ex.map(drive, range(len(runs))))
        st = pool.stats()
    for i in range(len(runs)):
        kps, pose, stats, window = pooled[i]
        rk, rpose, rstats, rwindow = alone[i]
        for (pl, pt), (rpl, rpt) in zip(kps, rk):
            assert pl.tobytes() == rpl.tobytes() and pt.tobytes() == rpt.tobytes(), runs[i]
        assert stats == rstats, (runs[i], stats, rstats)
        assert np.array_equal(window["scan"], rwindow["scan"]), runs[i]
        assert np.max(np.abs(pose["t"] - rpose["t"])) < 1e-7 and np.max(np.abs(pose["R"] - rpose["R"])) < 1e-7
    assert st["requests"] > st["submits"] > 0


def test_pool_rejects_an_estimator_whose_hot_path_params_differ_from_its_sequence():
    from form_b200.pipeline import EstimatorPool

    a = _capi.default_est_params(16, 1800)
    b = _capi.default_est_params(64, 1024, point_feats_per_sector=0)
    with EstimatorPool([a, b]) as pool:
        lib = pool._lib
        for seq, wrong in ((0, b), (1, a), (1, _capi.default_est_params(64, 1024)),
                           (0, _capi.default_est_params(16, 1800, max_window_scans=32))):
            assert not lib.formhost_pool_est_create(pool._h, C.byref(wrong), seq)
            msg = lib.formhost_last_error()
            assert b"hot-path parameters differ" in msg and f"sequence {seq}".encode() in msg, msg
    # the homogeneous pool checks the same way
    with EstimatorPool(a, 2) as pool:
        assert not pool._lib.formhost_pool_est_create(pool._h, C.byref(b), 1)


_ATTRIBUTE_SCRIPT = r"""
import sys
sys.path[:0] = [{root!r}, {tests!r}]
from form_b200 import _capi, synth
from form_b200.context import Context
import oracle_lib
small = _capi.default_params(16, 1800)   # ~94 KB of normals shared memory
large = _capi.default_params(64, 1024)   # ~54 KB, created after it
a = Context(small)
b = Context(large)
for ctx, p, sensor in ((a, small, "vlp-16"), (b, large, "os1-64")):
    scan = synth.scan(sensor, 3, 1)
    planar, point = ctx.extract(scan, 1)
    rp, rq = oracle_lib.Oracle(p).extract(scan, 1)
    assert len(rp) > 0 and planar.tobytes() == rp.tobytes(), sensor
    assert point.tobytes() == rq.tobytes(), sensor
print("ok")
"""


def test_smaller_context_created_later_keeps_the_larger_shared_memory_attribute():
    """The kernels' max-dynamic-shared-memory attributes are process-wide: a fresh process creates
    a 16x1800 context, then a 64x1024 one, and both must still extract (single-context path)."""
    script = _ATTRIBUTE_SCRIPT.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_sweep_writes_evalio_files_equal_to_standalone_runs(tmp_path):
    from form_b200 import sweep, trajectory
    from form_b200.pipeline import Estimator

    n = 10
    summary = sweep.main(["--sensor", "vlp-16", "--sensor", "os1-64", "--sequences", "1", "--scans", str(n),
                          "--variant", "form", "--variant", "no_points:point_feats_per_sector=0,max_dist_map=0.2",
                          "--out", str(tmp_path)])
    assert len(summary) == 4
    rows = (tmp_path / "summary.csv").read_text().strip().splitlines()
    assert rows[0] == "variant,sequence,scans,hz,ate_rmse" and len(rows) == 5
    for sensor in ("vlp-16", "os1-64"):
        d = tmp_path / "synthetic" / sensor / "1"
        assert sorted(os.listdir(d)) == ["form.csv", "gt.csv", "no_points.csv"]
        meta, _, t_gt, _ = trajectory.read_evalio_csv(d / "gt.csv")
        assert meta["sequence"] == f"synthetic/{sensor}/1" and len(t_gt) == n
        for name, ov in (("form", {}), ("no_points", dict(point_feats_per_sector=0, max_dist_map=0.2))):
            meta, _, t, R = trajectory.read_evalio_csv(d / f"{name}.csv")
            assert meta["status"] == "complete" and meta["name"] == name
            with Estimator(sweep.est_params(*synth.shape(sensor), ov)) as e:
                ref = []
                for k in range(n):
                    e.register_scan(synth.scan(sensor, 1, k))
                    ref.append(e.pose().copy())
            assert np.max(np.abs(t - np.stack([r["t"] for r in ref]))) < 1e-7, (sensor, name)
            assert np.max(np.abs(R - np.stack([r["R"].reshape(3, 3) for r in ref]))) < 1e-7, (sensor, name)
