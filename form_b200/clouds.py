"""Raw sensor clouds: what a LiDAR driver or a recorded log delivers before any organisation -
unordered records, missing returns absent - and the readers and synthetic source this project
feeds to formgpu_organize / Estimator.register_cloud (rule R8, DESIGN.md §4).

    read_dir(DIR)             a directory of scans: .npy structured arrays (fields x, y, z and any of
                              ring|row, col, t|time) or KITTI-style .bin float32 x, y, z, intensity
    synth_cloud(sensor, s, k) scan k of synthetic sequence s as the cloud a driver would emit
    write_dir(DIR, clouds)    the inverse of read_dir for .npy clouds
"""
from __future__ import annotations

import math
import os

import numpy as np

from . import _capi, synth

KITTI_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("i", "<f4")])


def list_dir(path: str) -> list[str]:
    """The scan files of a directory in name order: all .npy or all .bin, not a mix."""
    names = sorted(n for n in os.listdir(path) if n.endswith((".npy", ".bin")))
    kinds = {os.path.splitext(n)[1] for n in names}
    if not names:
        raise ValueError(f"{path}: no .npy or .bin scans")
    if len(kinds) > 1:
        raise ValueError(f"{path}: mixes .npy and .bin scans")
    return [os.path.join(path, n) for n in names]


def read_scan(path: str) -> np.ndarray:
    """One cloud as a structured array: a .npy structured array as stored, or a KITTI .bin as
    KITTI_DTYPE records."""
    if path.endswith(".bin"):
        raw = np.fromfile(path, dtype="<f4")
        if raw.size % 4:
            raise ValueError(f"{path}: {raw.size} floats is not a whole number of x, y, z, i records")
        return raw.view(KITTI_DTYPE).copy()
    a = np.load(path, allow_pickle=False)
    if a.dtype.names is None or a.ndim != 1:
        raise ValueError(f"{path}: expected a 1-d structured array with fields x, y, z, got {a.dtype} {a.shape}")
    return np.ascontiguousarray(a)


def read_dir(path: str) -> list[np.ndarray]:
    """Every cloud of a directory, in file-name order; all of them share one record layout."""
    clouds = [read_scan(p) for p in list_dir(path)]
    if len({c.dtype for c in clouds}) > 1:
        raise ValueError(f"{path}: the scans do not share one record layout")
    return clouds


def write_dir(path: str, clouds) -> list[str]:
    """Store clouds as 000000.npy, 000001.npy, ... (read_dir reads them back in order)."""
    os.makedirs(path, exist_ok=True)
    out = []
    for k, c in enumerate(clouds):
        p = os.path.join(path, f"{k:06d}.npy")
        np.save(p, np.ascontiguousarray(c), allow_pickle=False)
        out.append(p)
    return out


def beam_elevations(sensor: str) -> np.ndarray:
    """Beam elevations (radians, bottom beam first) of a synthetic sensor, one per row."""
    fov = {"os1-64": 16.6, "os0-128": 45.0, "vlp-16": 15.0, "stress-128x2048": 45.0}[sensor]
    rows, _ = synth.shape(sensor)
    deg = math.pi / 180.0
    return np.array([(-fov + 2.0 * fov * r / (rows - 1)) * deg for r in range(rows)])


def cloud_dtype(f64: bool = False, fields=("ring", "col", "t")) -> np.dtype:
    """Packed record layout of synth_cloud: x, y, z (f4 or f8), then ring (u2), col (u2), t (f4)."""
    kinds = {"ring": "<u2", "row": "<u2", "col": "<u2", "t": "<f4"}
    f = "<f8" if f64 else "<f4"
    return np.dtype([("x", f), ("y", f), ("z", f)] + [(n, kinds[n]) for n in fields])


def synth_cloud(sensor: str, sequence_id: int, k: int, *, order: str = "firing", duplicates: int = 0,
                f64: bool = False, fields=("ring", "col", "t"), scan_period: float = 0.1,
                seed: int = 0) -> np.ndarray:
    """Scan k of synthetic sequence `sequence_id` as a driver emits it: the no-returns are dropped,
    every point carries its ring, column and time since the scan started
    (t = (col + 0.5) * scan_period / cols, so floor(t * cols / scan_period) is its column), and the
    records come in firing order (column by column, bottom ring first) or, with order="shuffled", in
    a seeded random order.  `duplicates` > 0 adds that many colliding records per 64 points - an
    exact copy or a copy pushed 1 % to 50 % farther along its ray - which organisation must resolve
    back to the original point.  Organised with synth.shape(sensor) the cloud is synth.scan(...)
    byte for byte."""
    rows, cols = synth.shape(sensor)
    scan = synth.scan(sensor, sequence_id, k).reshape(rows, cols)
    xyz = np.stack([scan["x"], scan["y"], scan["z"]], axis=-1)
    live = ~((xyz[..., 0] == 0) & (xyz[..., 1] == 0) & (xyz[..., 2] == 0))
    # firing order: column-major, ring 0 (bottom) first
    cc, rr = np.nonzero(live.T)
    pts = xyz[rr, cc]
    rng = np.random.default_rng(seed * 1000003 + sequence_id * 1009 + k)
    if duplicates > 0:
        m = len(pts) * duplicates // 64
        pick = rng.choice(len(pts), size=m, replace=True)
        scale = np.where(rng.random(m) < 0.5, 1.0, 1.0 + rng.uniform(0.01, 0.5, m)).astype(np.float32)
        dup = (pts[pick] * scale[:, None]).astype(np.float32)
        pts = np.concatenate([pts, dup])
        rr = np.concatenate([rr, rr[pick]])
        cc = np.concatenate([cc, cc[pick]])
    if order == "shuffled":
        perm = rng.permutation(len(pts))
    elif order == "firing":
        perm = np.argsort(cc * rows + rr, kind="stable")  # duplicates next to their originals
    else:
        raise ValueError(f"order must be 'firing' or 'shuffled', not {order!r}")
    out = np.zeros(len(pts), dtype=cloud_dtype(f64, fields))
    for a, name in enumerate("xyz"):
        out[name] = pts[perm, a]
    if "ring" in fields or "row" in fields:
        out["ring" if "ring" in fields else "row"] = rr[perm]
    if "col" in fields:
        out["col"] = cc[perm]
    if "t" in fields:
        out["t"] = ((cc[perm] + 0.5) * scan_period / cols).astype(np.float32)
    return out


def synth_format(sensor: str, records: np.ndarray, *, row_from: str | None = None, col_from: str | None = None,
                 scan_period: float = 0.1, max_records: int | None = None) -> _capi.CloudFormat:
    """formgpu_cloud_format for synth_cloud records of `sensor` (beam table of the synthetic sensor
    when rows come from elevation)."""
    rows, cols = synth.shape(sensor)
    beams = beam_elevations(sensor) if row_from == "elevation" else None
    return _capi.cloud_format(records.dtype, row_from=row_from, col_from=col_from, scan_period=scan_period,
                              beams=beams, max_records=max_records or 2 * rows * cols)


def format_from_args(dtype, args, rows: int) -> _capi.CloudFormat:
    """formgpu_cloud_format from the command-line flags of run_sequence / sweep (--row-from,
    --col-from, --scan-period, --beams FILE of elevations in degrees, --max-records)."""
    beams = None
    if args.beams:
        beams = np.radians(np.loadtxt(args.beams, dtype=np.float64).reshape(-1))
        if len(beams) != rows:
            raise ValueError(f"{args.beams}: {len(beams)} beam elevations for {rows} rows")
    return _capi.cloud_format(dtype, row_from=args.row_from, col_from=args.col_from, scan_period=args.scan_period,
                              beams=beams, max_records=args.max_records)


def add_format_args(ap) -> None:
    """The cloud-format flags shared by run_sequence and sweep."""
    ap.add_argument("--rows", type=int, help="scan rows of the recorded sensor (default: the --sensor shape)")
    ap.add_argument("--cols", type=int, help="scan columns of the recorded sensor (default: the --sensor shape)")
    ap.add_argument("--row-from", choices=["ring", "elevation"],
                    help="row source (default: the ring / row field, else elevation)")
    ap.add_argument("--col-from", choices=["col", "time", "azimuth"],
                    help="column source (default: col field, else time field, else azimuth)")
    ap.add_argument("--scan-period", type=float, default=0.1, help="seconds per revolution (default 0.1)")
    ap.add_argument("--beams", help="text file of beam elevations in degrees, one per row (--row-from elevation)")
    ap.add_argument("--max-records", type=int, default=0,
                    help="record capacity per scan (default: the largest scan of the log)")
