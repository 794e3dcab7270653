"""Run form::Estimator over a synthetic sequence and write the trajectory (and the ground truth)
in evalio's CSV layout - what `evalio run -M form` produces for FORM's experiment scripts
(/root/reference/README.md:51-55, experiments/env.py:157-198: per-run `hz`, `status`).

    python -m form_b200.run_sequence --sensor os1-64 --scans 200 --out out_dir [--disable-smoothing]

A recorded log - a directory of raw clouds, .npy structured arrays or KITTI .bin files, see
form_b200/clouds.py - runs through Estimator.register_cloud, organised on the GPU:

    python -m form_b200.run_sequence --clouds DIR --rows 16 --cols 1800 [--row-from ring|elevation]
        [--col-from col|time|azimuth] [--scan-period 0.1] [--beams FILE] --out out_dir

It has no ground truth, so only form.csv is written.
"""
from __future__ import annotations

import argparse
import os
import time

import numpy as np

from . import _capi, clouds, synth, trajectory
from .pipeline import Estimator


def relative_gt(seq: int, k: int):
    """Ground-truth pose of scan k in the frame of scan 0 (the estimator starts at identity)."""
    g0, gk = synth.gt_pose(seq, 0), synth.gt_pose(seq, k)
    R0 = g0["R"].reshape(3, 3)
    out = np.zeros((), dtype=_capi.POSE)
    out["R"] = (R0.T @ gk["R"].reshape(3, 3)).reshape(9)
    out["t"] = R0.T @ (gk["t"] - g0["t"])
    return out


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--sensor", default="os1-64", choices=sorted(synth.SENSORS))
    ap.add_argument("--sequence", type=int, default=0)
    ap.add_argument("--scans", type=int, default=200)
    ap.add_argument("--rate-hz", type=float, default=10.0)
    ap.add_argument("--out", default="trajectories")
    ap.add_argument("--disable-smoothing", action="store_true")
    ap.add_argument("--point-feats-per-sector", type=int, default=3)
    ap.add_argument("--clouds", help="directory of raw clouds (a recorded log) instead of the synthetic sequence")
    clouds.add_format_args(ap)
    args = ap.parse_args(argv)
    if args.clouds:
        return run_clouds(args)

    rows, cols = synth.shape(args.sensor)
    overrides = dict(disable_smoothing=int(args.disable_smoothing), point_feats_per_sector=args.point_feats_per_sector)
    p = _capi.default_est_params(rows, cols, **overrides)
    scans = [synth.scan(args.sensor, args.sequence, k) for k in range(args.scans)]
    stamps = [k / args.rate_hz for k in range(args.scans)]
    poses, step = [], []
    with Estimator(p) as est:
        for scan in scans:
            t0 = time.perf_counter()
            est.register_scan(scan)
            step.append(time.perf_counter() - t0)
            poses.append(est.pose().copy())
    gt = [relative_gt(args.sequence, k) for k in range(args.scans)]
    os.makedirs(args.out, exist_ok=True)
    seq_name = f"synthetic/{args.sensor}/{args.sequence}"
    trajectory.write_evalio_csv(os.path.join(args.out, "form.csv"), stamps, poses, params=overrides,
                                total_elapsed=sum(step), max_step_elapsed=max(step), sequence=seq_name)
    trajectory.write_evalio_csv(os.path.join(args.out, "gt.csv"), stamps, gt, name="gt", pipeline="gt",
                                sequence=seq_name)
    err = [float(np.linalg.norm(a["t"] - b["t"])) for a, b in zip(poses, gt)]
    print(f"{seq_name}: {args.scans} scans, hz = {args.scans / sum(step):.1f}, "
          f"ATE rmse vs ground truth = {np.sqrt(np.mean(np.square(err))):.4f} m -> {args.out}/form.csv, gt.csv")


def log_shape(args) -> tuple[int, int]:
    """Scan shape of a recorded log: --rows / --cols, defaulting to the --sensor shape."""
    rows, cols = synth.shape(args.sensor)
    return args.rows or rows, args.cols or cols


def run_clouds(args):
    rows, cols = log_shape(args)
    scans = clouds.read_dir(args.clouds)
    if args.max_records <= 0:
        args.max_records = max(len(c) for c in scans)
    fmt = clouds.format_from_args(scans[0].dtype, args, rows)
    overrides = dict(disable_smoothing=int(args.disable_smoothing), point_feats_per_sector=args.point_feats_per_sector)
    p = _capi.default_est_params(rows, cols, **overrides)
    stamps = [k / args.rate_hz for k in range(len(scans))]
    poses, step = [], []
    with Estimator(p) as est:
        est.set_cloud_format(fmt)
        for cloud in scans:
            t0 = time.perf_counter()
            est.register_cloud(cloud)
            step.append(time.perf_counter() - t0)
            poses.append(est.pose().copy())
    os.makedirs(args.out, exist_ok=True)
    seq_name = f"log/{os.path.basename(os.path.normpath(args.clouds))}"
    trajectory.write_evalio_csv(os.path.join(args.out, "form.csv"), stamps, poses, params=overrides,
                                total_elapsed=sum(step), max_step_elapsed=max(step), sequence=seq_name)
    print(f"{seq_name}: {len(scans)} clouds, hz = {len(scans) / sum(step):.1f} -> {args.out}/form.csv "
          "(no ground truth)")


if __name__ == "__main__":
    main()
