"""Raw sensor clouds on the B200: formgpu_organize against the synthetic scans and against the numpy
restatement of rule R8 (tests/cloud_model.py), the estimator and pool fed clouds against the same
runs fed organised scans, batched / mixed submissions with FORMGPU_REQ_CLOUD, the error paths, and
the run_sequence / sweep drivers on a directory of clouds."""
import ctypes as C
import math

import numpy as np
import pytest

import cloud_model
from form_b200 import _capi, clouds, synth
from form_b200.context import Context, FormGpuError

pytestmark = pytest.mark.gpu

COMBOS = [(("ring", "t"), "ring", "time"), (("ring",), "ring", "azimuth"), ((), "elevation", "azimuth"),
          (("row", "col"), "ring", "col")]


def _stats(rec):
    return {k: int(rec[k]) for k in _capi.CLOUD_STATS.names}


@pytest.mark.parametrize("sensor", sorted(synth.SENSORS))
def test_organize_reproduces_the_synthetic_scan(sensor):
    rows, cols = synth.shape(sensor)
    ref = synth.scan(sensor, 2, 5)
    with Context(_capi.default_params(rows, cols)) as ctx:
        for fields, row_from, col_from in COMBOS:
            for order in ("firing", "shuffled"):
                for f64 in (False, True):
                    rec = clouds.synth_cloud(sensor, 2, 5, order=order, fields=fields, f64=f64, duplicates=2)
                    fmt = clouds.synth_format(sensor, rec, row_from=row_from, col_from=col_from)
                    ctx.set_cloud_format(fmt)
                    scan, st = ctx.organize(rec)
                    assert scan.tobytes() == ref.tobytes(), (fields, order, f64)
                    _, model = cloud_model.organize(rec, fmt, rows, cols)
                    assert _stats(st) == model
                    assert _stats(ctx.cloud_stats()) == model


def _adversarial(rows, cols, rng, beams):
    """Points on column and beam boundaries (+-1 ulp), many-way equal-range collisions, zeros,
    NaN / Inf, rings and times out of range."""
    out = []
    for b in range(cols):
        phi = 2.0 * math.pi * (b - 0.5) / cols
        for d in (-1, 0, 1):
            a = np.nextafter(phi, phi + d) if d else phi
            r = rng.uniform(1, 30)
            out.append((r * math.cos(a), r * math.sin(a), rng.uniform(-2, 2)))
    for j in range(rows - 1):
        mu = (beams[j] + beams[j + 1]) * 0.5
        for d in (-1, 0, 1):
            e = np.nextafter(mu, mu + d) if d else mu
            a, r = rng.uniform(0, 2 * math.pi), rng.uniform(1, 30)
            out.append((r * math.cos(e) * math.cos(a), r * math.cos(e) * math.sin(a), r * math.sin(e)))
    xyz = np.array(out)
    # the same point many times at equal range (ties go to the lower record index), and its mirror
    tie = np.repeat(xyz[:50], 8, axis=0)
    tie[1::2] *= np.array([1.0, -1.0, 1.0])
    xyz = np.concatenate([xyz, tie, rng.uniform(-40, 40, (4000, 3))])
    n = len(xyz) + 6
    dt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("ring", "<u2"), ("col", "<u2"), ("t", "<f4")])
    rec = np.zeros(n, dt)
    rec["x"][:-6], rec["y"][:-6], rec["z"][:-6] = xyz.T
    rec["x"][-6:] = [0.0, -0.0, np.nan, np.inf, 1.0, 2.0]
    rec["y"][-6:] = [0.0, 0.0, 1.0, 1.0, -np.inf, 0.0]
    rec["ring"] = rng.integers(0, rows + 3, n)
    rec["col"] = rng.integers(0, cols + 5, n)
    rec["t"] = rng.uniform(-0.01, 0.11, n).astype(np.float32)
    rec["t"][:4] = [0.0, np.nextafter(np.float32(0.1), np.float32(0)), 0.1, -0.0]
    return rec


@pytest.mark.parametrize("sensor", ["vlp-16", "os0-128"])
def test_organize_matches_the_numpy_rule_on_adversarial_clouds(sensor):
    rows, cols = synth.shape(sensor)
    beams = clouds.beam_elevations(sensor)
    rng = np.random.default_rng(7)
    rec = _adversarial(rows, cols, rng, beams)
    with Context(_capi.default_params(rows, cols)) as ctx:
        for row_from, col_from, extra in (("ring", "time", {}), ("ring", "col", {}), ("elevation", "azimuth", {}),
                                          ("elevation", "azimuth", dict(azimuth_dir=-1, azimuth_origin=0.7)),
                                          ("ring", "azimuth", dict(azimuth_origin=-2.0))):
            table = beams[::-1] if extra.get("azimuth_dir") == -1 else beams  # top-down table too
            fmt = _capi.cloud_format(rec.dtype, row_from=row_from, col_from=col_from, max_records=len(rec),
                                     beams=table if row_from == "elevation" else None, **extra)
            ctx.set_cloud_format(fmt)
            scan, st = ctx.organize(rec)
            ref, model = cloud_model.organize(rec, fmt, rows, cols)
            assert scan.tobytes() == ref.tobytes(), (row_from, col_from, extra)
            assert _stats(st) == model, (row_from, col_from, extra)
            assert model["dropped_zero"] == 2 and model["dropped_nonfinite"] == 3
            assert model["placed"] > model["pixels"]
        # u32 nanoseconds as time
        dt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("ring", "u1"), ("t", "<u4")])
        ns = np.zeros(len(rec), dt)
        for k in ("x", "y", "z"):
            ns[k] = rec[k]
        ns["ring"] = np.minimum(rec["ring"], 255)
        ns["t"] = rng.integers(0, 120_000_000, len(rec), dtype=np.uint32)
        fmt = _capi.cloud_format(dt, max_records=len(ns))
        ctx.set_cloud_format(fmt)
        scan, st = ctx.organize(ns)
        ref, model = cloud_model.organize(ns, fmt, rows, cols)
        assert scan.tobytes() == ref.tobytes() and _stats(st) == model and model["dropped_time"] > 0


def test_estimator_register_cloud_equals_register_scan():
    from form_b200.pipeline import Estimator, EstimatorPool

    sensor, seq, n = "vlp-16", 3, 30
    rows, cols = synth.shape(sensor)
    p = _capi.default_est_params(rows, cols)
    scans = [synth.scan(sensor, seq, k) for k in range(n)]
    recs = [clouds.synth_cloud(sensor, seq, k, order="shuffled", duplicates=2) for k in range(n)]
    fmt = clouds.synth_format(sensor, recs[0], row_from="ring", col_from="time")

    def run(est, inputs, cloud):
        out = []
        for x in inputs:
            kp = est.register_cloud(x) if cloud else est.register_scan(x)
            out.append((kp[0].tobytes(), kp[1].tobytes(), est.pose().tobytes()))
        return out, est.stats(), est.window().tobytes()

    with Estimator(p) as a:
        ref = run(a, scans, False)
    with Estimator(p) as b:
        b.set_cloud_format(fmt)
        got = run(b, recs, True)
        assert _stats(b.cloud_stats())["records"] == len(recs[-1])
    assert got == ref
    # pooled: a cloud sequence and an organised-scan sequence in one pool
    import threading

    with EstimatorPool([p, p], cloud_formats=[fmt, None]) as pool:
        res = [None, None]
        th = [threading.Thread(target=lambda i=i: res.__setitem__(i, run(pool.estimators[i], recs if i == 0 else scans,
                                                                          i == 0))) for i in range(2)]
        for t in th:
            t.start()
        for t in th:
            t.join()
    # the two sequences of the pool are bit-identical; against a stand-alone estimator a pool differs
    # in the fp64 summation order of its stage-3 reductions only: same keypoints and ICP / LM counts,
    # poses to 1e-7 (as tests/test_gpu_mixed_batch.py)
    assert res[0] == res[1]
    (steps, stats, window), (rsteps, rstats, rwindow) = res[0], ref
    assert [s[:2] for s in steps] == [s[:2] for s in rsteps] and stats == rstats
    for s, r in zip(steps, rsteps):
        a, b = np.frombuffer(s[2], _capi.POSE)[0], np.frombuffer(r[2], _capi.POSE)[0]
        assert np.max(np.abs(a["t"] - b["t"])) < 1e-7 and np.max(np.abs(a["R"] - b["R"])) < 1e-7


class _Batch:
    def __init__(self, params):
        self.lib = _capi.gpu_lib()
        self.h = C.c_void_p()
        arr = (_capi.Params * len(params))(*params)
        assert self.lib.formgpu_batch_create_mixed(arr, 0, None, len(params), C.byref(self.h)) == 0
        self.outs = []
        for i in range(len(params)):
            c = self.lib.formgpu_batch_ctx(self.h, i)
            cp, cq = self.lib.formgpu_max_planar(c), self.lib.formgpu_max_point(c)
            self.outs.append((np.zeros(cp, _capi.PLANAR_FEAT), np.zeros(cq, _capi.POINT_FEAT)))

    def ctx(self, i):
        return self.lib.formgpu_batch_ctx(self.h, i)

    def extract(self, inputs, scan_idx, cloud_flags):
        reqs = (_capi.Request * len(inputs))()
        for s, x in enumerate(inputs):
            reqs[s].sequence, reqs[s].op, reqs[s].flags = s, _capi.OP_EXTRACT, cloud_flags[s]
            reqs[s].scan, reqs[s].n_points, reqs[s].scan_idx = x.ctypes.data, len(x), scan_idx
            reqs[s].planar_out, reqs[s].planar_cap = self.outs[s][0].ctypes.data, len(self.outs[s][0])
            reqs[s].point_out, reqs[s].point_cap = self.outs[s][1].ctypes.data, len(self.outs[s][1])
        rc = self.lib.formgpu_batch_submit(self.h, reqs, len(inputs))
        res = [(reqs[s].status, self.outs[s][0][: reqs[s].n_planar].tobytes(),
                self.outs[s][1][: reqs[s].n_point].tobytes()) for s in range(len(inputs))]
        return rc, res

    def close(self):
        self.lib.formgpu_batch_destroy(self.h)


def test_mixed_batch_with_clouds_equals_single_contexts():
    sensors = ["vlp-16", "os1-64", "os0-128", "vlp-16"]
    combos = [("ring", "time", False), None, ("elevation", "azimuth", True), ("ring", "col", False)]
    params = [_capi.default_params(*synth.shape(s)) for s in sensors]
    b = _Batch(params)
    try:
        fmts = []
        for i, (s, c) in enumerate(zip(sensors, combos)):
            if c is None:
                fmts.append(None)
                continue
            fields = {"time": ("ring", "t"), "azimuth": (), "col": ("ring", "col")}[c[1]]
            rec = clouds.synth_cloud(s, i, 0, fields=fields, f64=c[2])
            fmt = clouds.synth_format(s, rec, row_from=c[0], col_from=c[1])
            assert _capi.gpu_lib().formgpu_set_cloud_format(b.ctx(i), C.byref(fmt)) == 0
            fmts.append((fmt, fields, c[2]))
        flags = [0 if f is None else _capi.REQ_CLOUD for f in fmts]
        runs = []
        for prefetch in (False, True, False):
            for k in range(3):
                inputs = [synth.scan(s, i, k) if f is None else
                          clouds.synth_cloud(s, i, k, fields=f[1], f64=f[2], order="shuffled", duplicates=1)
                          for i, (s, f) in enumerate(zip(sensors, fmts))]
                if prefetch:
                    for i, f in enumerate(fmts):
                        if f is not None:
                            assert _capi.gpu_lib().formgpu_batch_prefetch_cloud(
                                b.h, i, inputs[i].ctypes.data, len(inputs[i])) == 0
                rc, res = b.extract(inputs, k, flags)
                assert rc == 0 and all(r[0] == 0 for r in res)
                for i, f in enumerate(fmts):
                    if f is None:
                        continue
                    st = np.zeros(1, _capi.CLOUD_STATS)
                    assert _capi.gpu_lib().formgpu_cloud_stats_last(b.ctx(i), _capi.ptr(st)) == 0
                    _, model = cloud_model.organize(inputs[i], f[0], *synth.shape(sensors[i]))
                    assert _stats(st[0]) == model
                runs.append(res)
        # the same scans on single contexts, organised inputs
        for i, s in enumerate(sensors):
            with Context(params[i]) as ctx:
                for k in range(3):
                    pl, pt = ctx.extract(synth.scan(s, i, k), k)
                    for r in range(3):
                        assert runs[3 * r + k][i][1] == pl.tobytes() and runs[3 * r + k][i][2] == pt.tobytes(), (i, k, r)
    finally:
        b.close()


def test_cloud_errors_single_and_batched():
    rows, cols = synth.shape("vlp-16")
    rec = clouds.synth_cloud("vlp-16", 0, 0)
    with Context(_capi.default_params(rows, cols)) as ctx:
        with pytest.raises(FormGpuError) as e:
            ctx.organize(rec)
        assert e.value.code == _capi.ERR_STATE and "no cloud format" in str(e.value)
        with pytest.raises(FormGpuError) as e:
            ctx.extract_cloud(rec, 0)
        assert e.value.code == _capi.ERR_STATE
        bad = _capi.cloud_format(rec.dtype, scan_period=0.0)
        with pytest.raises(FormGpuError) as e:
            ctx.set_cloud_format(bad)
        assert e.value.code == _capi.ERR_INVALID_ARG and "scan_period" in str(e.value)
        ctx.set_cloud_format(_capi.cloud_format(rec.dtype, max_records=len(rec) - 1))
        with pytest.raises(FormGpuError) as e:
            ctx.organize(rec)
        assert e.value.code == _capi.ERR_CAPACITY
        ctx.set_cloud_format(_capi.cloud_format(rec.dtype, max_records=len(rec)))
        pl, pt = ctx.extract_cloud(rec, 0)
        rpl, rpt = Context(_capi.default_params(rows, cols)).extract(synth.scan("vlp-16", 0, 0), 0)
        assert pl.tobytes() == rpl.tobytes() and pt.tobytes() == rpt.tobytes()
    params = [_capi.default_params(rows, cols)] * 3
    b = _Batch(params)
    try:
        fmt = _capi.cloud_format(rec.dtype, max_records=100)
        assert _capi.gpu_lib().formgpu_set_cloud_format(b.ctx(1), C.byref(fmt)) == 0
        scan = synth.scan("vlp-16", 0, 0)
        rc, res = b.extract([rec, rec, scan], 0, [_capi.REQ_CLOUD, _capi.REQ_CLOUD, 0])
        assert rc == _capi.ERR_STATE
        assert [r[0] for r in res] == [_capi.ERR_STATE, _capi.ERR_CAPACITY, 0]
        with Context(params[2]) as ctx:
            rpl, rpt = ctx.extract(scan, 0)
        assert res[2][1] == rpl.tobytes() and res[2][2] == rpt.tobytes()
        assert _capi.gpu_lib().formgpu_batch_prefetch_cloud(b.h, 0, rec.ctypes.data, len(rec)) == _capi.ERR_STATE
        assert _capi.gpu_lib().formgpu_batch_prefetch_cloud(b.h, 1, rec.ctypes.data, len(rec)) == _capi.ERR_CAPACITY
    finally:
        b.close()


def test_run_sequence_and_sweep_on_a_cloud_directory(tmp_path):
    from form_b200 import run_sequence, sweep, trajectory

    n = 12
    d = tmp_path / "log"
    clouds.write_dir(str(d), [clouds.synth_cloud("vlp-16", 0, k, order="shuffled") for k in range(n)])
    run_sequence.main(["--sensor", "vlp-16", "--scans", str(n), "--out", str(tmp_path / "synth")])
    run_sequence.main(["--clouds", str(d), "--rows", "16", "--cols", "1800", "--out", str(tmp_path / "cloud")])
    _, s0, t0, r0 = trajectory.read_evalio_csv(tmp_path / "synth" / "form.csv")
    meta, s1, t1, r1 = trajectory.read_evalio_csv(tmp_path / "cloud" / "form.csv")
    assert meta["sequence"] == "log/log" and not (tmp_path / "cloud" / "gt.csv").exists()
    rows0 = (tmp_path / "synth" / "form.csv").read_text().splitlines()
    rows1 = (tmp_path / "cloud" / "form.csv").read_text().splitlines()
    assert [r for r in rows0 if not r.startswith("#")] == [r for r in rows1 if not r.startswith("#")]
    summary = sweep.main(["--log", f"mylog={d}", "--rows", "16", "--cols", "1800", "--sensor", "vlp-16",
                          "--sequences", "0", "--scans", str(n), "--out", str(tmp_path / "sw")])
    assert [(r["sequence"], r["ate_rmse"] == "") for r in summary] == [("synthetic/vlp-16/0", False), ("log/mylog", True)]
    a = (tmp_path / "sw" / "synthetic" / "vlp-16" / "0" / "form.csv").read_text().splitlines()
    c = (tmp_path / "sw" / "log" / "mylog" / "form.csv").read_text().splitlines()
    assert [r for r in a if not r.startswith("#")] == [r for r in c if not r.startswith("#")]
    _, _, tp, rp = trajectory.read_evalio_csv(tmp_path / "sw" / "log" / "mylog" / "form.csv")
    assert np.max(np.abs(tp - t0)) < 1e-7 and np.max(np.abs(rp - r0)) < 1e-7  # pool against stand-alone
    lines = (tmp_path / "sw" / "summary.csv").read_text().splitlines()
    assert lines[2].startswith("form,log/mylog,12,") and lines[2].endswith(",")
