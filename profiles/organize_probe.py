"""Raw clouds on the GPU (rule R8): what organisation costs per scan, for each sensor shape.

  single   formgpu_organize on one context: CUDA events on the context's stream around the call
           (record upload, clear + scatter + gather, counters' copy), host records in page-locked
           memory; and the same with the organised scan (what formgpu_extract uploads instead)
  batch    one formgpu_batch_submit of --seqs EXTRACT requests of that shape, CUDA events on the
           batch's stream around the submission: FORMGPU_REQ_CLOUD against organised host scans
  e2e      an EstimatorPool of --e2e-seqs live estimators (one thread each), --scans scans each after
           --warmup untimed ones: register_cloud against register_scan, scans/s over the wall time

Clouds come from clouds.synth_cloud (ring + time fields, shuffled, no duplicates).  The card's name
and power limit are read in the same run.  The JSON goes to --out (default: a temporary directory).

usage: python profiles/organize_probe.py [--sensors vlp-16,os1-64,os0-128,stress-128x2048] [--out DIR]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from form_b200 import _capi, clouds, synth  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return out[0]


_PINNED = []  # the tensors that own the page-locked buffers


def pinned_copy(a: np.ndarray) -> np.ndarray:
    import torch

    t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
    _PINNED.append(t)
    out = t.numpy().view(a.dtype)
    out[:] = a
    return out


def timed(stream, fn, reps):
    """Device milliseconds per call: events on `stream` around `reps` calls (each call waits)."""
    import torch

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    a.record(stream)
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / reps, (time.perf_counter() - t0) * 1e3 / reps


def probe_single(sensor, reps):
    import torch

    from form_b200.context import Context

    rows, cols = synth.shape(sensor)
    stream = torch.cuda.Stream()
    rec = pinned_copy(clouds.synth_cloud(sensor, 0, 0, order="shuffled"))
    scan = pinned_copy(synth.scan(sensor, 0, 0))
    with Context(_capi.default_params(rows, cols), stream=stream.cuda_stream) as ctx:
        ctx.set_cloud_format(clouds.synth_format(sensor, rec, row_from="ring", col_from="time"))
        lib, h = ctx._lib, ctx._h
        st = np.zeros(1, _capi.CLOUD_STATS)
        dev_ms, host_ms = timed(stream, lambda: lib.formgpu_organize(h, _capi.ptr(rec), len(rec), None, _capi.ptr(st)),
                                reps)
        pl, pt = np.zeros(ctx.max_planar, _capi.PLANAR_FEAT), np.zeros(ctx.max_point, _capi.POINT_FEAT)
        a, b = C.c_size_t(), C.c_size_t()
        ex_cloud, _ = timed(stream, lambda: lib.formgpu_extract_cloud(h, _capi.ptr(rec), len(rec), 0, _capi.ptr(pl),
                                                                      len(pl), C.byref(a), _capi.ptr(pt), len(pt),
                                                                      C.byref(b)), reps)
        ex_scan, _ = timed(stream, lambda: lib.formgpu_extract(h, _capi.ptr(scan), len(scan), 0, _capi.ptr(pl), len(pl),
                                                               C.byref(a), _capi.ptr(pt), len(pt), C.byref(b)), reps)
    return dict(records=len(rec), record_bytes=int(rec.nbytes), scan_bytes=int(scan.nbytes),
                organize_ms=dev_ms, organize_host_ms=host_ms, extract_cloud_ms=ex_cloud, extract_scan_ms=ex_scan)


def probe_batch(sensor, seqs, reps):
    import torch

    rows, cols = synth.shape(sensor)
    lib = _capi.gpu_lib()
    stream = torch.cuda.Stream()
    h = C.c_void_p()
    params = _capi.default_params(rows, cols)
    assert lib.formgpu_batch_create(C.byref(params), 0, C.c_void_p(stream.cuda_stream), seqs, C.byref(h)) == 0
    try:
        recs = [pinned_copy(clouds.synth_cloud(sensor, s, 0, order="shuffled")) for s in range(seqs)]
        scans = [pinned_copy(synth.scan(sensor, s, 0)) for s in range(seqs)]
        fmt = clouds.synth_format(sensor, recs[0], row_from="ring", col_from="time")
        outs = []
        for s in range(seqs):
            c = lib.formgpu_batch_ctx(h, s)
            assert lib.formgpu_set_cloud_format(c, C.byref(fmt)) == 0
            outs.append((pinned_copy(np.zeros(lib.formgpu_max_planar(c), _capi.PLANAR_FEAT)),
                         pinned_copy(np.zeros(lib.formgpu_max_point(c), _capi.POINT_FEAT))))

        def reqs_for(inputs, flags):
            reqs = (_capi.Request * seqs)()
            for s in range(seqs):
                reqs[s].sequence, reqs[s].op, reqs[s].flags = s, _capi.OP_EXTRACT, flags
                reqs[s].scan, reqs[s].n_points = inputs[s].ctypes.data, len(inputs[s])
                reqs[s].planar_out, reqs[s].planar_cap = outs[s][0].ctypes.data, len(outs[s][0])
                reqs[s].point_out, reqs[s].point_cap = outs[s][1].ctypes.data, len(outs[s][1])
            return reqs

        rc, rs = reqs_for(recs, _capi.REQ_CLOUD), reqs_for(scans, 0)
        out = {}
        for name, reqs in (("cloud", rc), ("scan", rs), ("cloud_again", rc)):
            dev, host = timed(stream, lambda: lib.formgpu_batch_submit(h, reqs, seqs), reps)
            out[name] = dict(submit_ms=dev, submit_host_ms=host)
        return out
    finally:
        lib.formgpu_batch_destroy(h)


def probe_e2e(sensor, seqs, scans, warmup):
    from form_b200.pipeline import EstimatorPool

    rows, cols = synth.shape(sensor)
    p = _capi.default_est_params(rows, cols)
    total = warmup + scans
    data = {s: [synth.scan(sensor, s, k) for k in range(total)] for s in range(seqs)}
    recs = {s: [clouds.synth_cloud(sensor, s, k, order="shuffled") for k in range(total)] for s in range(seqs)}
    fmt = clouds.synth_format(sensor, recs[0][0], row_from="ring", col_from="time",
                              max_records=max(len(r) for v in recs.values() for r in v))
    res = {}
    for arm in ("scan", "cloud", "scan_again", "cloud_again"):
        cloud = arm.startswith("cloud")
        with EstimatorPool(p, seqs, cloud_formats=[fmt] * seqs if cloud else None) as pool:
            barrier = threading.Barrier(seqs + 1)
            done = threading.Barrier(seqs + 1)

            def drive(s, est):
                reg = est.register_cloud if cloud else est.register_scan
                src = recs[s] if cloud else data[s]
                for k in range(warmup):
                    reg(src[k])
                barrier.wait()
                for k in range(warmup, total):
                    reg(src[k])
                done.wait()

            th = [threading.Thread(target=drive, args=(s, e)) for s, e in enumerate(pool.estimators)]
            for t in th:
                t.start()
            barrier.wait()
            t0 = time.perf_counter()
            done.wait()
            dt = time.perf_counter() - t0
            for t in th:
                t.join()
        res[arm] = dict(scans_per_s=seqs * scans / dt, seconds=dt)
    return res


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--sensors", default="vlp-16,os1-64,os0-128,stress-128x2048")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--seqs", type=int, default=32, help="sequences of the batched and e2e arms")
    ap.add_argument("--e2e-seqs", type=int, default=16, help="live estimators of the e2e arm")
    ap.add_argument("--scans", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import torch

    assert torch.cuda.is_available(), "organize_probe measures on a GPU; there is none"
    out = dict(card=card(), reps=args.reps, seqs=args.seqs, e2e_seqs=args.e2e_seqs, scans=args.scans,
               warmup=args.warmup, sensors={})
    print(out["card"], flush=True)
    for sensor in args.sensors.split(","):
        r = dict(single=probe_single(sensor, args.reps), batch=probe_batch(sensor, args.seqs, max(args.reps // 4, 10)),
                 e2e=probe_e2e(sensor, args.e2e_seqs, args.scans, args.warmup))
        out["sensors"][sensor] = r
        print(sensor, json.dumps(r), flush=True)
    d = args.out or tempfile.mkdtemp(prefix="organize_probe_")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "organize_probe.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("->", os.path.join(d, "organize_probe.json"))


if __name__ == "__main__":
    main()
