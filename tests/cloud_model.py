"""Rule R8 (DESIGN.md §4) restated in numpy: a raw cloud -> the organised row-major scan and the
outcome counters, with the arithmetic of form_b200/csrc/organize.cu (f64 decisions, no fused
multiply-add, boundary tables from the C library's cos / sin through Python's math module).
formgpu_organize must match it bit for bit."""
from __future__ import annotations

import math

import numpy as np

from form_b200 import _capi

_NP = {_capi.FIELD_F32: "<f4", _capi.FIELD_F64: "<f8", _capi.FIELD_U8: "u1", _capi.FIELD_U16: "<u2",
       _capi.FIELD_U32: "<u4", _capi.FIELD_U32_NS: "<u4"}


def _field(raw: np.ndarray, off: int, type_: int) -> np.ndarray:
    """Column of a field at byte offset `off` of every record (raw: (n, stride) uint8)."""
    dt = np.dtype(_NP[type_])
    return np.ascontiguousarray(raw[:, off:off + dt.itemsize]).view(dt).reshape(-1)


def tables(fmt, rows: int, cols: int, beams=None):
    """(azimuth boundaries [cols + 1] (cos, sin), beam midpoints [rows - 1] ascending (cos, sin), desc)."""
    az = np.zeros((cols + 1, 2))
    for b in range(cols + 1):
        phi = fmt.azimuth_origin + float(fmt.azimuth_dir) * (2.0 * math.pi * (b - 0.5) / cols)
        az[b] = (math.cos(phi), math.sin(phi))
    el = np.zeros((max(rows - 1, 0), 2))
    desc = False
    if fmt.row_source == _capi.ROW_FROM_ELEVATION:
        asc = [float(v) for v in beams]
        if rows > 1 and asc[1] < asc[0]:
            desc = True
            asc = asc[::-1]
        for j in range(rows - 1):
            mu = (asc[j] + asc[j + 1]) * 0.5
            el[j] = (math.cos(mu), math.sin(mu))
    return az, el, desc


def _azimuth_column(x, y, az, cols, direction):
    def past(b):
        s = y * az[b, 0] - x * az[b, 1]
        if direction < 0:
            s = -s
        return s >= 0.0

    m = cols // 2
    first = past(np.zeros_like(x, dtype=np.int64)) & ~past(np.full(x.shape, m, dtype=np.int64))
    lo = np.where(first, 0, m)
    hi = np.where(first, m, cols)
    while True:
        open_ = hi - lo > 1
        if not open_.any():
            return lo
        mid = (lo + hi) // 2
        p = past(np.where(open_, mid, 0))
        lo = np.where(open_ & p, mid, lo)
        hi = np.where(open_ & ~p, mid, hi)


def _elevation_row(x, y, z, el, rows, desc):
    rho = np.sqrt(x * x + y * y)
    lo = np.zeros(x.shape, dtype=np.int64)
    hi = np.full(x.shape, rows - 1, dtype=np.int64)
    while True:
        open_ = lo < hi
        if not open_.any():
            break
        mid = np.where(open_, (lo + hi) // 2, 0)
        above = z * el[mid, 0] - rho * el[mid, 1] >= 0.0
        lo = np.where(open_ & above, mid + 1, lo)
        hi = np.where(open_ & ~above, mid, hi)
    return rows - 1 - lo if desc else lo


def organize(records: np.ndarray, fmt, rows: int, cols: int, beams=None):
    """-> (scan: (rows*cols,) POINT4F, stats: dict of the formgpu_cloud_stats counters)."""
    n = len(records)
    raw = np.ascontiguousarray(records).view(np.uint8).reshape(n, fmt.stride) if n else np.zeros((0, fmt.stride), np.uint8)
    if beams is None and fmt.row_source == _capi.ROW_FROM_ELEVATION:
        beams = fmt.beams()
    az, el, desc = tables(fmt, rows, cols, beams)
    x, y, z = (_field(raw, o, fmt.xyz_type).astype(np.float32) for o in (fmt.off_x, fmt.off_y, fmt.off_z))
    with np.errstate(all="ignore"):
        finite = np.isfinite(x) & np.isfinite(y) & np.isfinite(z)
        zero = (x == 0) & (y == 0) & (z == 0)
        if fmt.off_time >= 0:
            tv = _field(raw, fmt.off_time, fmt.time_type)
            t = tv.astype(np.float64) * 1e-9 if fmt.time_type == _capi.FIELD_U32_NS else tv.astype(np.float64)
            bad_time = ~((t >= 0.0) & (t < fmt.scan_period))
        else:
            t = np.zeros(n)
            bad_time = np.zeros(n, bool)
        xd, yd, zd = x.astype(np.float64), y.astype(np.float64), z.astype(np.float64)
        if fmt.row_source == _capi.ROW_FROM_FIELD:
            v = _field(raw, fmt.off_row, fmt.row_type).astype(np.int64)
            row = np.where(v < rows, v, -1)
        else:
            row = _elevation_row(xd, yd, zd, el, rows, desc)
        if fmt.col_source == _capi.COL_FROM_FIELD:
            v = _field(raw, fmt.off_col, fmt.col_type).astype(np.int64)
            col = np.where(v < cols, v, -1)
        elif fmt.col_source == _capi.COL_FROM_TIME:
            q = (t * float(cols)) / fmt.scan_period
            col = np.minimum(np.floor(np.where(bad_time, 0.0, q)).astype(np.int64), cols - 1)
        else:
            col = _azimuth_column(xd, yd, az, cols, fmt.azimuth_dir)
        n2 = (x * x + z * z) + (y * y + np.float32(0.0))
    code = np.full(n, 1)  # placed
    code[~finite] = 3
    code[finite & zero] = 4
    rest = finite & ~zero
    code[rest & bad_time] = 5
    rest &= ~bad_time
    code[rest & (row < 0)] = 6
    rest &= row >= 0
    code[rest & (col < 0)] = 7
    placed = code == 1
    pix = row[placed] * cols + col[placed]
    key = (n2[placed].view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.nonzero(placed)[0].astype(np.uint64)
    keys = np.full(rows * cols, np.iinfo(np.uint64).max, dtype=np.uint64)
    np.minimum.at(keys, pix, key)
    won = keys != np.iinfo(np.uint64).max
    idx = (keys[won] & np.uint64(0xffffffff)).astype(np.int64)
    scan = np.zeros(rows * cols, dtype=_capi.POINT4F)
    scan["x"][won], scan["y"][won], scan["z"][won] = x[idx], y[idx], z[idx]
    stats = dict(records=n, placed=int(placed.sum()), pixels=int(won.sum()),
                 dropped_nonfinite=int((code == 3).sum()), dropped_zero=int((code == 4).sum()),
                 dropped_time=int((code == 5).sum()), dropped_row=int((code == 6).sum()),
                 dropped_col=int((code == 7).sum()))
    return scan, stats
