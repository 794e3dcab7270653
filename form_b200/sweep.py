"""Sequences x parameter variants, run live through one mixed EstimatorPool - this project's
counterpart of `evalio run -c config.yaml` for FORM's experiments (several sensors, several logs,
ablations such as `point_feats_per_sector: 0` or `disable_smoothing: true`).

    python -m form_b200.sweep --sensor vlp-16 --sensor os1-64 --sequences 0,1 --scans 100 \\
        --variant form --variant no_points:point_feats_per_sector=0 \\
        --variant fixed_lag_off:disable_smoothing=true --out sweeps

A variant is `NAME` (FORM's defaults) or `NAME:key=value,key=value` with the parameter names of
FORM.default_params() (python/bindings.cpp), applied as FORM.set_params applies them
(`max_dist_map` sets the map's `min_dist_map`).  Every (sensor, sequence, variant) is one
PooledEstimator on its own thread; all of them share one pool (one formgpu batch) unless
--pool-size caps the estimators per pool.  Output, in evalio's CSV layout:
OUT/synthetic/<sensor>/<seq>/<variant>.csv per run, gt.csv once per sequence, and OUT/summary.csv
(variant, sequence, scans, hz, ATE rmse against ground truth).

Recorded logs join the same pool: `--log NAME=DIR` (repeatable) names a directory of raw clouds
(form_b200/clouds.py: .npy structured arrays or KITTI .bin), organised on the GPU through
register_cloud.  Their shape and record format come from --rows/--cols and the cloud flags of
run_sequence (--row-from, --col-from, --scan-period, --beams).  Every scan of the log is run; its
runs land in OUT/log/NAME/<variant>.csv, and a log has no ground truth, so its ate_rmse stays empty.

    python -m form_b200.sweep --log mylog=DIR --rows 16 --cols 1800 --sensor vlp-16 --out sweeps
"""
from __future__ import annotations

import argparse
import csv
import os
import threading
import time

import numpy as np

from . import _capi, clouds, synth, trajectory
from .pipeline import EstimatorPool
from .run_sequence import relative_gt

# FORM.default_params() (python/bindings.cpp) -> (field of formhost_est_params, type); "hot." fields
# live in formgpu_params.  The mapping is FORM.set_params'.
PARAM_FIELDS = {
    "neighbor_points": ("hot.neighbor_points", int),
    "num_sectors": ("hot.num_sectors", int),
    "planar_threshold": ("hot.planar_threshold", float),
    "planar_feats_per_sector": ("hot.planar_feats_per_sector", int),
    "point_feats_per_sector": ("hot.point_feats_per_sector", int),
    "radius": ("hot.radius", float),
    "min_points": ("hot.min_points", int),
    "max_dist_matching": ("hot.max_dist_matching", float),
    "new_pose_threshold": ("new_pose_threshold", float),
    "max_num_rematches": ("max_num_rematches", int),
    "disable_smoothing": ("disable_smoothing", bool),
    "max_num_keyscans": ("max_num_keyscans", int),
    "max_num_recent_scans": ("max_num_recent_scans", int),
    "max_steps_unused_keyscan": ("max_steps_unused_keyscan", int),
    "keyscan_match_ratio": ("keyscan_match_ratio", float),
    "max_dist_map": ("hot.min_dist_map", float),  # bindings.cpp: the name differs from the field
    "num_threads": ("num_threads", int),
}


def _value(key: str, text: str):
    kind = PARAM_FIELDS[key][1]
    t = text.strip()
    if kind is bool:
        if t.lower() in ("true", "1", "yes", "on"):
            return True
        if t.lower() in ("false", "0", "no", "off"):
            return False
        raise ValueError(f"{key}: expected true or false, got {text!r}")
    if kind is int:
        v = float(t)
        if v != int(v):
            raise ValueError(f"{key}: expected an integer, got {text!r}")
        return int(v)
    return float(t)


def parse_variant(spec: str) -> tuple[str, dict]:
    """`NAME` or `NAME:key=value,...` -> (name, {key: value}) with FORM.default_params() keys."""
    name, _, body = spec.partition(":")
    name = name.strip()
    if not name or "/" in name or name in (".", ".."):
        raise ValueError(f"variant {spec!r}: needs a name usable as a file name")
    if name == "gt":
        raise ValueError("variant name 'gt' is taken by the ground-truth file")
    overrides = {}
    for item in filter(None, (s.strip() for s in body.split(","))):
        key, eq, val = item.partition("=")
        key = key.strip()
        if not eq:
            raise ValueError(f"variant {name!r}: {item!r} is not key=value")
        if key not in PARAM_FIELDS:
            raise ValueError(f"variant {name!r}: unknown parameter {key!r}; valid keys: "
                             + ", ".join(sorted(PARAM_FIELDS)))
        overrides[key] = _value(key, val)
    return name, overrides


def parse_variants(specs) -> list[tuple[str, dict]]:
    out, seen = [], set()
    for spec in specs:
        name, overrides = parse_variant(spec)
        if name in seen:
            raise ValueError(f"duplicate variant name {name!r}")
        seen.add(name)
        out.append((name, overrides))
    return out


def est_params(rows: int, cols: int, overrides: dict) -> _capi.EstParams:
    """formhost_est_params of a sensor shape with FORM.default_params()-named overrides."""
    p = _capi.default_est_params(rows, cols)
    for key, value in overrides.items():
        if key not in PARAM_FIELDS:
            raise ValueError(f"unknown parameter {key!r}; valid keys: " + ", ".join(sorted(PARAM_FIELDS)))
        field, kind = PARAM_FIELDS[key]
        target = p.hot if field.startswith("hot.") else p
        setattr(target, field.split(".")[-1], int(value) if kind is bool else kind(value))
    return p


def parse_log(spec: str) -> tuple[str, str]:
    """`NAME=DIR` -> (name, dir)."""
    name, eq, path = spec.partition("=")
    name = name.strip()
    if not eq or not name or not path or "/" in name or name in (".", ".."):
        raise ValueError(f"--log {spec!r}: expected NAME=DIR with a NAME usable as a file name")
    return name, path


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--sensor", action="append", choices=sorted(synth.SENSORS),
                    help="sensor (repeatable; default os1-64 when no --log is given)")
    ap.add_argument("--sequences", default="0", help="comma-separated sequence ids")
    ap.add_argument("--scans", type=int, default=100)
    ap.add_argument("--rate-hz", type=float, default=10.0)
    ap.add_argument("--variant", action="append",
                    help="NAME or NAME:key=value,... (repeatable; default: one variant 'form')")
    ap.add_argument("--log", action="append", default=[], help="NAME=DIR: a recorded log of raw clouds (repeatable)")
    ap.add_argument("--pool-size", type=int, default=0,
                    help="estimators per pool (default 0: every run in one pool)")
    ap.add_argument("--linger-us", type=int, default=200)
    ap.add_argument("--out", default="sweeps")
    clouds.add_format_args(ap)
    args = ap.parse_args(argv)

    sensors = args.sensor or ([] if args.log else ["os1-64"])
    sequences = [int(s) for s in args.sequences.split(",") if s.strip()]
    try:
        variants = parse_variants(args.variant or ["form"])
        logs = [parse_log(spec) for spec in args.log]
    except ValueError as e:
        ap.error(str(e))
    if len({name for name, _ in logs}) != len(logs):
        ap.error("duplicate --log name")
    if logs and not (args.rows and args.cols):
        ap.error("--log needs the scan shape of the recorded sensor: --rows and --cols")
    if args.scans < 1 or (sensors and not sequences):
        ap.error("need at least one scan and one sequence")

    # a source is ("synthetic", sensor, seq) or ("log", name); a run is (source, variant, overrides)
    sources = [("synthetic", sensor, seq) for sensor in sensors for seq in sequences] + [("log", n) for n, _ in logs]
    scans, formats, shapes = {}, {}, {}
    for sensor in sensors:
        for seq in sequences:
            scans["synthetic", sensor, seq] = [synth.scan(sensor, seq, k) for k in range(args.scans)]
            shapes["synthetic", sensor, seq] = synth.shape(sensor)
    for name, path in logs:
        recs = clouds.read_dir(path)
        max_records = args.max_records if args.max_records > 0 else max(len(c) for c in recs)
        fmt_args = argparse.Namespace(**{**vars(args), "max_records": max_records})
        try:
            formats["log", name] = clouds.format_from_args(recs[0].dtype, fmt_args, args.rows)
        except ValueError as e:
            ap.error(f"--log {name}: {e}")
        scans["log", name] = recs
        shapes["log", name] = (args.rows, args.cols)
    runs = [(src, name, overrides) for src in sources for name, overrides in variants]
    params = [est_params(*shapes[src], overrides) for src, _, overrides in runs]
    cloud_formats = [formats.get(src) for src, _, _ in runs]

    size = args.pool_size if args.pool_size > 0 else len(runs)
    pools = [EstimatorPool(params[i:i + size], linger_us=args.linger_us, cloud_formats=cloud_formats[i:i + size])
             for i in range(0, len(runs), size)]
    estimators = [est for pool in pools for est in pool.estimators]
    poses = [[] for _ in runs]
    steps = [[] for _ in runs]
    errors = [None] * len(runs)

    def drive(i):
        src = runs[i][0]
        register = estimators[i].register_cloud if src[0] == "log" else estimators[i].register_scan
        try:
            for scan in scans[src]:
                t0 = time.perf_counter()
                register(scan)
                steps[i].append(time.perf_counter() - t0)
                poses[i].append(estimators[i].pose().copy())
        except Exception as e:  # reported after every thread has finished
            errors[i] = e

    threads = [threading.Thread(target=drive, args=(i,)) for i in range(len(runs))]
    try:
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    finally:
        for pool in pools:
            pool.close()
    for i, e in enumerate(errors):
        if e is not None:
            raise RuntimeError(f"run {runs[i][0][1:]} {runs[i][1]!r} failed: {e}") from e

    summary = []
    for src in sources:
        n = len(scans[src])
        stamps = [k / args.rate_hz for k in range(n)]
        seq_name = f"synthetic/{src[1]}/{src[2]}" if src[0] == "synthetic" else f"log/{src[1]}"
        d = os.path.join(args.out, seq_name)
        os.makedirs(d, exist_ok=True)
        gt = None
        if src[0] == "synthetic":
            gt = [relative_gt(src[2], k) for k in range(n)]
            trajectory.write_evalio_csv(os.path.join(d, "gt.csv"), stamps, gt, name="gt", pipeline="gt",
                                        sequence=seq_name)
        for i, (s_, name, overrides) in enumerate(runs):
            if s_ != src:
                continue
            trajectory.write_evalio_csv(os.path.join(d, f"{name}.csv"), stamps, poses[i], name=name,
                                        params=overrides, total_elapsed=sum(steps[i]),
                                        max_step_elapsed=max(steps[i]), sequence=seq_name)
            row = dict(variant=name, sequence=seq_name, scans=n, hz=round(n / sum(steps[i]), 3), ate_rmse="")
            if gt is not None:
                err = [float(np.linalg.norm(a["t"] - b["t"])) for a, b in zip(poses[i], gt)]
                row["ate_rmse"] = round(float(np.sqrt(np.mean(np.square(err)))), 6)
            summary.append(row)
            ate = f"ATE rmse vs ground truth = {row['ate_rmse']:.4f} m" if gt is not None else "no ground truth"
            print(f"{seq_name} [{name}]: {n} scans, hz = {row['hz']:.1f}, {ate}")
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "summary.csv"), "w", newline="") as f:
        w = csv.DictWriter(f, fieldnames=["variant", "sequence", "scans", "hz", "ate_rmse"])
        w.writeheader()
        w.writerows(summary)
    print(f"{len(runs)} runs in {len(pools)} pool(s) -> {args.out}/summary.csv")
    return summary


if __name__ == "__main__":
    main()
