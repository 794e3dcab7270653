"""Raw sensor clouds without a GPU: rule R8's numpy restatement against the synthetic scans,
formgpu_cloud_format_check (fails before any CUDA call, with a message), the dtype -> format helper,
the readers of form_b200/clouds.py, and the exported symbols."""
import ctypes as C
import math

import numpy as np
import pytest

import cloud_model
from form_b200 import _capi, clouds, synth

COMBOS = [(("ring", "t"), "ring", "time"), (("ring",), "ring", "azimuth"), ((), "elevation", "azimuth"),
          (("row", "col"), "ring", "col")]


def test_new_symbols_are_declared_bound_and_exported():
    for name in ("formgpu_cloud_format_check", "formgpu_set_cloud_format", "formgpu_organize",
                 "formgpu_extract_cloud", "formgpu_cloud_stats_last", "formgpu_batch_prefetch_cloud"):
        assert name in _capi.FORMGPU_SYMBOLS
        assert hasattr(_capi.gpu_lib(), name)
    for name in ("formhost_est_set_cloud_format", "formhost_est_register_cloud", "formhost_est_cloud_stats"):
        assert name in _capi.FORMHOST_SYMBOLS
        assert hasattr(_capi.host_lib(), name)
    assert _capi.gpu_lib().formgpu_abi_version() == 1
    assert _capi.KG_COUNT == 12 and _capi.REQ_CLOUD == 2
    assert C.sizeof(_capi.CloudFormat) == 88 and _capi.CLOUD_STATS.itemsize == 64
    assert C.sizeof(_capi.Request) == 176  # formgpu_request keeps its layout


@pytest.mark.parametrize("sensor", sorted(synth.SENSORS))
@pytest.mark.parametrize("fields, row_from, col_from", COMBOS)
@pytest.mark.parametrize("order", ["firing", "shuffled"])
def test_synth_cloud_round_trips_through_the_rule(sensor, fields, row_from, col_from, order):
    rows, cols = synth.shape(sensor)
    rec = clouds.synth_cloud(sensor, 1, 4, order=order, fields=fields, duplicates=3, f64=order == "shuffled")
    fmt = clouds.synth_format(sensor, rec, row_from=row_from, col_from=col_from)
    assert _capi.check_cloud_format(fmt, rows, cols) == (0, "")
    scan, stats = cloud_model.organize(rec, fmt, rows, cols)
    ref = synth.scan(sensor, 1, 4)
    assert scan.tobytes() == ref.tobytes()
    live = int(np.count_nonzero((ref["x"] != 0) | (ref["y"] != 0) | (ref["z"] != 0)))
    assert stats["pixels"] == live and stats["placed"] == len(rec) > live
    assert stats["records"] == len(rec)


def test_synth_cloud_layout():
    rec = clouds.synth_cloud("vlp-16", 0, 0)
    assert rec.dtype.names == ("x", "y", "z", "ring", "col", "t") and rec.dtype.itemsize == 20
    assert not np.any((rec["x"] == 0) & (rec["y"] == 0) & (rec["z"] == 0))
    key = rec["col"].astype(np.int64) * 16 + rec["ring"]
    assert np.all(np.diff(key) > 0)  # firing order: column by column, bottom ring first
    assert np.array_equal(np.floor(rec["t"].astype(np.float64) * 1800 / 0.1).astype(int), rec["col"])
    shuffled = clouds.synth_cloud("vlp-16", 0, 0, order="shuffled")
    assert not np.array_equal(shuffled, rec)
    assert np.array_equal(np.sort(shuffled, order=["col", "ring"]), rec)
    with pytest.raises(ValueError, match="order"):
        clouds.synth_cloud("vlp-16", 0, 0, order="random")


def test_dtype_to_format():
    dt = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("intensity", "<f4"), ("ring", "u1"), ("time", "<u4")])
    f = _capi.cloud_format(dt)
    assert (f.stride, f.off_x, f.off_y, f.off_z, f.xyz_type) == (33, 0, 8, 16, _capi.FIELD_F64)
    assert (f.off_row, f.row_type, f.row_source) == (28, _capi.FIELD_U8, _capi.ROW_FROM_FIELD)
    assert (f.off_time, f.time_type, f.col_source) == (29, _capi.FIELD_U32_NS, _capi.COL_FROM_TIME)
    assert f.off_col == _capi.CLOUD_ABSENT
    g = _capi.cloud_format(clouds.KITTI_DTYPE, beams=np.radians(np.linspace(-15, 15, 16)))
    assert (g.row_source, g.col_source, g.off_row, g.off_time) == (_capi.ROW_FROM_ELEVATION, _capi.COL_FROM_AZIMUTH, -1, -1)
    assert np.allclose(g.beams(), np.radians(np.linspace(-15, 15, 16)))
    h = _capi.cloud_format(clouds.cloud_dtype(fields=("row", "col", "t")), col_from="azimuth", azimuth_dir=-1)
    assert (h.row_source, h.col_source, h.azimuth_dir) == (_capi.ROW_FROM_FIELD, _capi.COL_FROM_AZIMUTH, -1)
    with pytest.raises(ValueError, match="x, y, z"):
        _capi.cloud_format(np.dtype([("x", "<f4"), ("y", "<f4")]))
    with pytest.raises(ValueError, match="float32 or all float64"):
        _capi.cloud_format(np.dtype([("x", "<f4"), ("y", "<f8"), ("z", "<f4")]))
    with pytest.raises(ValueError, match="u1, u2 or u4"):
        _capi.cloud_format(np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("ring", "<f4")]))
    with pytest.raises(ValueError, match="row_from"):
        _capi.cloud_format(clouds.cloud_dtype(), row_from="up")


def _good():
    return _capi.cloud_format(clouds.cloud_dtype(), max_records=1000)


@pytest.mark.parametrize("change, match", [
    (dict(stride=0), "stride"),
    (dict(off_x=18), "x: offset 18 does not fit a 20-byte record"),
    (dict(off_z=-1), "z: offset -1"),
    (dict(xyz_type=_capi.FIELD_U16), "x: unsupported field type"),
    (dict(off_time=19), "time: offset 19"),
    (dict(row_type=_capi.FIELD_F32), "row: unsupported"),
    (dict(scan_period=0.0), "scan_period"),
    (dict(scan_period=float("nan")), "scan_period"),
    (dict(max_records=0), "max_records"),
    (dict(max_records=1 << 32), "max_records"),
    (dict(off_row=-1), "row source FIELD needs a ring"),
    (dict(col_source=_capi.COL_FROM_FIELD, off_col=-1), "column source FIELD needs a col"),
    (dict(col_source=_capi.COL_FROM_TIME, off_time=-1), "column source TIME needs a time"),
    (dict(col_source=_capi.COL_FROM_AZIMUTH, azimuth_dir=0), "azimuth_dir"),
    (dict(row_source=7), "unknown row source"),
    (dict(row_source=_capi.ROW_FROM_ELEVATION), "needs beam_elevations"),
])
def test_format_check_rejects_bad_formats_with_a_message(change, match):
    f = _good()
    for k, v in change.items():
        setattr(f, k, v)
    rc, msg = _capi.check_cloud_format(f, 16, 1800)
    assert rc == _capi.ERR_INVALID_ARG and match in msg, msg


@pytest.mark.parametrize("beams, match", [
    ([0.1, 0.2, 0.2, 0.3], "strictly monotonic (beam 2)"),
    ([0.3, 0.2, 0.25, 0.1], "strictly monotonic (beam 2)"),
    ([0.1, 0.2, 1.6, 1.7], "not in (-pi/2, pi/2)"),
])
def test_format_check_rejects_bad_beam_tables(beams, match):
    f = _capi.cloud_format(clouds.cloud_dtype(fields=()), beams=beams)
    rc, msg = _capi.check_cloud_format(f, 4, 100)
    assert rc == _capi.ERR_INVALID_ARG and match in msg, msg
    ok = _capi.cloud_format(clouds.cloud_dtype(fields=()), beams=[0.3, 0.2, 0.1, -0.1])  # top-down is fine
    assert _capi.check_cloud_format(ok, 4, 100) == (0, "")


def test_set_cloud_format_validates_before_touching_the_gpu():
    """A bad format fails the same way on a context-less check and is named in the message; a
    context is needed for set_cloud_format itself, so here only the null context is checked."""
    lib = _capi.gpu_lib()
    f = _good()
    f.scan_period = -1.0
    assert lib.formgpu_set_cloud_format(None, C.byref(f)) == _capi.ERR_INVALID_ARG
    assert lib.formgpu_cloud_format_check(None, 16, 1800, None, 0) == _capi.ERR_INVALID_ARG
    assert lib.formgpu_organize(None, None, 0, None, None) == _capi.ERR_INVALID_ARG


def test_rule_drops_and_counts_by_reason():
    """Hand-made records, one per outcome, against the restatement's counters."""
    dt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("ring", "<u2"), ("t", "<f4")])
    rec = np.array([(1, 0, 0, 0, 0.0), (np.nan, 0, 0, 0, 0.0), (0, 0, 0, 0, 0.0), (-0.0, 0, 0, 1, 0.0),
                    (1, 1, 0, 0, 0.1), (1, 1, 0, 0, -1e-9), (1, 1, 0, 4, 0.05), (2, 0, 0, 0, 0.0),
                    (1, 0, 0, 0, 0.0)], dtype=dt)
    fmt = _capi.cloud_format(dt, max_records=100)
    scan, st = cloud_model.organize(rec, fmt, 4, 16)
    assert st == dict(records=9, placed=3, pixels=1, dropped_nonfinite=1, dropped_zero=2, dropped_time=2,
                      dropped_row=1, dropped_col=0)
    # the nearest of the three points of pixel (0, 0) wins; of the two equal ones, the lower index
    assert scan[0].tolist() == (1.0, 0.0, 0.0, 0.0) and not scan[1:].tolist().count((1.0, 0.0, 0.0, 0.0))


def test_azimuth_rule_nearest_centre():
    cols = 8
    ang = 2 * math.pi * np.arange(cols) / cols
    dt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("ring", "u1")])
    rec = np.zeros(cols, dt)
    rec["x"], rec["y"], rec["z"] = 5 * np.cos(ang + 0.3), 5 * np.sin(ang + 0.3), 1
    for direction, origin, expect in ((1, 0.0, np.arange(cols)), (-1, 0.0, (-np.arange(cols)) % cols),
                                      (1, 2 * math.pi / cols, (np.arange(cols) - 1) % cols)):
        f = _capi.cloud_format(dt, col_from="azimuth", azimuth_dir=direction, azimuth_origin=origin)
        scan, _ = cloud_model.organize(rec, f, 1, cols)
        got = [int(np.nonzero(scan["x"] == r["x"])[0][0]) for r in rec]
        assert got == expect.tolist(), direction


def test_readers(tmp_path):
    a = [clouds.synth_cloud("vlp-16", 0, k) for k in range(3)]
    clouds.write_dir(str(tmp_path / "npy"), a)
    back = clouds.read_dir(str(tmp_path / "npy"))
    assert [b.tobytes() for b in back] == [x.tobytes() for x in a]
    kitti = tmp_path / "kitti"
    kitti.mkdir()
    for k in range(2):
        np.arange(12 * (k + 1), dtype="<f4").tofile(kitti / f"{k:06d}.bin")
    got = clouds.read_dir(str(kitti))
    assert got[0].dtype == clouds.KITTI_DTYPE and len(got[0]) == 3 and len(got[1]) == 6
    assert got[1]["z"].tolist() == [2, 6, 10, 14, 18, 22]
    (kitti / "000009.npy").write_bytes(b"")
    with pytest.raises(ValueError, match="mixes"):
        clouds.read_dir(str(kitti))
    bad = tmp_path / "bad"
    bad.mkdir()
    np.arange(5, dtype="<f4").tofile(bad / "0.bin")
    with pytest.raises(ValueError, match="whole number"):
        clouds.read_dir(str(bad))
    (tmp_path / "empty").mkdir()
    with pytest.raises(ValueError, match="no .npy"):
        clouds.read_dir(str(tmp_path / "empty"))


def test_command_line_cloud_flags(tmp_path):
    import argparse

    ap = argparse.ArgumentParser()
    clouds.add_format_args(ap)
    beams = tmp_path / "beams.txt"
    beams.write_text("\n".join(str(v) for v in np.linspace(-15, 15, 16)))
    args = ap.parse_args(["--row-from", "elevation", "--col-from", "azimuth", "--beams", str(beams),
                          "--max-records", "5000"])
    f = clouds.format_from_args(clouds.KITTI_DTYPE, args, 16)
    assert f.row_source == _capi.ROW_FROM_ELEVATION and f.max_records == 5000
    assert np.allclose(f.beams(), np.radians(np.linspace(-15, 15, 16)))
    with pytest.raises(ValueError, match="16 beam elevations for 32 rows"):
        clouds.format_from_args(clouds.KITTI_DTYPE, args, 32)
    from form_b200 import sweep

    assert sweep.parse_log("mylog=/data/x") == ("mylog", "/data/x")
    with pytest.raises(ValueError, match="NAME=DIR"):
        sweep.parse_log("/data/x")
    with pytest.raises(SystemExit):
        sweep.main(["--log", "a=" + str(tmp_path), "--out", str(tmp_path / "o")])  # no --rows / --cols
