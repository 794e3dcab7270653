"""Mixed batches against homogeneous ones: what putting sequences of different sensors, or of
different hot-path parameters, into the same formgpu batch does to the batched engine's rate.

Two workloads, each replayed (recorded traces, device-resident scans) in two arms with the same
number of batches and host threads, driven by pipeline.run_batches as bench.py drives its value leg:

  M  32 x vlp-16 (16x1800), 32 x os1-64 (64x1024), 32 x os0-128 (128x1024) sequences
  V  128 os0-128 sequences in 4 hot-path variants of 32 (defaults; point_feats_per_sector=0;
     num_sectors=8 + planar_feats_per_sector=30; max_dist_matching=1.0 + min_dist_map=0.2)

  mixed  every batch holds an equal share of every group (sensor or variant)
  split  every batch holds one group only - the best that homogeneous batches allow

Traces are recorded live (Estimator, host smoother in the loop, one per sequence with its own
params) as bench.py records them; `--preroll` + `--warmup` untimed scans fill every fixed-lag
window before the timed `--steps` scans.  Reported per arm: scans/s, Mpoints/s (each scan counts
its own rows x cols), launches per scan, and per-kernel-group device milliseconds per scan from a
separate, profiled replay (ONE batch per arm's grouping: all sequences for mixed, one batch per
group for split), plus the card's name and power limit read in the same run.

usage: python profiles/mixed_batch.py [--workload M,V] [--steps 150] [--repeats 3] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from form_b200 import _capi, synth  # noqa: E402

WORKLOADS = {
    "M": [("vlp-16", {}), ("os1-64", {}), ("os0-128", {})],
    "V": [("os0-128", {}), ("os0-128", dict(point_feats_per_sector=0)),
          ("os0-128", dict(num_sectors=8, planar_feats_per_sector=30)),
          ("os0-128", dict(max_dist_matching=1.0, min_dist_map=0.2))],
}
GROUP_NAMES = {
    "M": ["vlp-16", "os1-64", "os0-128"],
    "V": ["defaults", "point_feats_per_sector=0", "num_sectors=8,planar_feats_per_sector=30",
          "max_dist_matching=1.0,min_dist_map=0.2"],
}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()
    return out[1] if len(out) > 1 else out[0]


def sum_stats(list_of_stats):
    out = {}
    for st in list_of_stats:
        for k, v in st.items():
            out[k] = out.get(k, 0) + v
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="M,V")
    ap.add_argument("--arms", default="mixed,split")
    ap.add_argument("--per-group", type=int, default=32, help="sequences per sensor / variant")
    ap.add_argument("--preroll", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--batches", type=int, default=12)
    ap.add_argument("--threads", type=int, default=0, help="host threads (0: min(batches, cores - 1))")
    ap.add_argument("--repeats", type=int, default=3, help="timed passes per arm (arms alternate)")
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "mixed_batch"),
                    help="directory of the JSON result")
    args = ap.parse_args()

    import torch

    from form_b200.pipeline import BatchReplay, Estimator, run_batches

    gpu = card()
    W0 = args.preroll + args.warmup
    S = W0 + args.steps
    G = args.batches
    T = args.threads or max(1, min(G, (len(os.sched_getaffinity(0)) or 1) - 1))
    os.makedirs(args.out, exist_ok=True)
    results = {"gpu": gpu, "batches": G, "host_threads": T,
               "preroll": args.preroll, "warmup": args.warmup, "steps": args.steps, "workloads": {}}
    pool = ThreadPoolExecutor(max_workers=16)
    for wl in [w.strip() for w in args.workload.split(",") if w.strip()]:
        groups = WORKLOADS[wl]
        N = args.per_group
        # sequence (group g, slot j): its params, its sensor's scans (variants replay the same logs)
        seqs = [(g, j) for g in range(len(groups)) for j in range(N)]
        params = {g: _capi.default_est_params(*synth.shape(sensor), record_trace=1, **ov)
                  for g, (sensor, ov) in enumerate(groups)}
        logs = sorted({(groups[g][0], j) for g, j in seqs})
        dev = {}

        def upload(log):
            sensor, j = log
            host = np.stack([synth.scan(sensor, j, k, 1) for k in range(S)])
            return log, host, torch.from_numpy(host.view(np.float32).reshape(S, -1)).cuda()

        t0 = time.time()
        hosts = {}
        for log, host, d in pool.map(upload, logs):
            hosts[log], dev[log] = host, d
        torch.cuda.synchronize()

        def record(s):
            g, j = s
            e = Estimator(params[g])
            for k in range(S):
                e.register_scan(hosts[groups[g][0], j][k])
            return e

        ests = dict(zip(seqs, pool.map(record, seqs)))
        del hosts
        t_setup = time.time() - t0
        ptr = {s: [dev[groups[s[0]][0], s[1]][k].data_ptr() for k in range(S)] for s in seqs}

        def arm_batches(arm):
            if arm == "mixed":  # batch b: slots j = b, b + G, ... of EVERY group
                return [[(g, j) for j in range(N) for g in range(len(groups)) if j % G == b] for b in range(G)]
            per = max(1, G // len(groups))  # split: every group over G / groups batches
            out = []
            for g in range(len(groups)):
                for b in range(per):
                    out.append([(g, j) for j in range(N) if j % per == b])
            return [b for b in out if b]

        def make(batch):
            return BatchReplay([ests[s].trace() for s in batch], [params[s[0]] for s in batch])

        def timed(arm):
            batches = arm_batches(arm)
            reps = [make(b) for b in batches]
            ptrs = [[ptr[s] for s in b] for b in batches]
            run_batches(reps, 0, W0, ptrs, True, T)  # pre-roll + warm-up
            for r in reps:
                r.reset_stats()
            l0 = sum(r.launch_count() for r in reps)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            run_batches(reps, W0, S, ptrs, True, T)
            torch.cuda.synchronize()
            b.record()
            torch.cuda.synchronize()
            t = a.elapsed_time(b) / 1e3
            st = sum_stats([r.stats() for r in reps])
            launches = sum(r.launch_count() for r in reps) - l0
            for r in reps:
                r.close()
            return dict(seconds=t, scans=st["scans"], points=st["points"], launches=launches,
                        batch_sizes=[len(x) for x in batches])

        def profiled(arm):
            """ONE batch per group of the arm's grouping, replayed one after the other with CUDA
            events around every kernel group (inflates short launches by a few us)."""
            grouping = [seqs] if arm == "mixed" else [[s for s in seqs if s[0] == g] for g in range(len(groups))]
            ms, scans = {}, 0
            for grp in grouping:
                rp = make(grp)
                rp.run(0, W0, [ptr[s] for s in grp])
                rp.reset_stats()
                rp.profile_read()
                rp.profile_enable(True)
                rp.run(W0, S, [ptr[s] for s in grp])
                for name, v in rp.profile_read().items():
                    if v["launches"]:
                        ms[name] = ms.get(name, 0.0) + v["ms"]
                scans += rp.stats()["scans"]
                rp.close()
            return {k: round(1e3 * v / scans, 3) for k, v in sorted(ms.items())}  # us per scan

        arms = [a.strip() for a in args.arms.split(",") if a.strip()]
        runs = {a: [] for a in arms}
        for _ in range(args.repeats):
            for a in arms:
                runs[a].append(timed(a))
        out = {"groups": GROUP_NAMES[wl], "sequences": len(seqs), "setup_s": round(t_setup, 1), "arms": {}}
        for a in arms:
            rates = [r["scans"] / r["seconds"] for r in runs[a]]
            mpts = [r["points"] / r["seconds"] / 1e6 for r in runs[a]]
            last = runs[a][-1]
            out["arms"][a] = {
                "scans_per_s": [round(x, 1) for x in rates],
                "mpoints_per_s": [round(x, 1) for x in mpts],
                "launches_per_scan": round(last["launches"] / last["scans"], 3),
                "batch_sizes": last["batch_sizes"],
                "kernel_group_us_per_scan": profiled(a),
            }
            print(f"[{wl}] {a:5s}: scans/s {out['arms'][a]['scans_per_s']}, Mpoints/s "
                  f"{out['arms'][a]['mpoints_per_s']}, launches/scan {out['arms'][a]['launches_per_scan']}",
                  flush=True)
        results["workloads"][wl] = out
        for e in ests.values():
            e.close()
        del dev, ests
        torch.cuda.empty_cache()
    path = os.path.join(args.out, "mixed_batch.json")
    with open(path, "w") as f:
        json.dump(results, f, indent=1)
    print(f"{gpu}: -> {path}")


if __name__ == "__main__":
    main()
