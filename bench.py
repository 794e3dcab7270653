#!/usr/bin/env python
"""bench.py - FORM per-scan hot path (feature + association + linearisation) on B200.

Contract (see the round brief): `python bench.py --gpus N --steps K --warmup W`
prints ONE JSON line on rank 0.  A step = the hot-path work of one scan of one sequence
(extraction, reparative map rebuild, every ICP association, every LM linearisation,
novel-keypoint commit), replayed from a trace that one untimed run of the real pipeline
(form::Estimator with the host smoother) records; the host smoother itself is therefore
not inside the timed region (BASELINE.md 2).

Workload: BASELINE.json configs[1] - synthetic OS0-128 (128x1024) sequences.  A single
sequence is a chain of ~45 dependent device calls per scan over < 1 MB each and cannot
fill a B200 (DESIGN.md 5), so the throughput metric is measured the way the path shards
(SURVEY 8e: independent sequences): M independent sequences per GPU, advanced in lock
step through formgpu_batch_submit - calls of the same kind share ONE launch per kernel.

  value     scans/s, whole job over all ranks: M sequences per GPU, scans resident in HBM
  e2e       same job through the host-buffer C-ABI: every scan comes from pinned host
            memory (H2D inside the timed region), keypoints and blocks go back (D2H)
  roofline  dominant kernel group of the batched run: algorithmic bytes / CUDA-event time
            vs the measured HBM peak (+ every other group under roofline.kernel_groups)
  single_sequence   the latency mode: ONE sequence per GPU (value / e2e / kernel times)
  cpu_baseline      the same multi-sequence job on the CPU oracle (kind "port"): one
            single-threaded replay per host core, --cpu-sample scans each; plus the reference's own
            threading (one sequence, parallel_for over keypoints) for comparison

`--impl reference` times the CPU oracle on the same job, --steps scans per sequence.  The
reference cannot be built as shipped here (no Eigen / GTSAM / TBB); its C++ sources do compile, unmodified, over API stand-ins
into oracle/_ref, but that library is a checker (restated Eigen arithmetic, serial TBB, restated
GTSAM optimiser), not a representative build: it is timed only as labelled extra rows
(reference_code_stage1, reference_code_pipeline), where it is the SLOWER of the two CPU codes.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

SENSOR_OF_WORKLOAD = {
    "os0-128": "configs[1]: synthetic OS0-128 (128x1024) sequences, fixed-lag window",
    "os1-64": "configs[0]/[3]: synthetic OS1-64 (64x1024) sequences",
    "vlp-16": "configs[2]: sparse VLP-16 (16x1800) sequences",
    "stress-128x2048": "configs[4]: dense 128x2048 stress scans",
}
METRIC = "scans/sec (feature+assoc+linearize hot path)"
DTYPE = "f32 index arithmetic, f64 transforms/normal equations"


def host_cores() -> int:
    """Host cores this process may run on (affinity-aware: a rank pinned to a share of the box,
    or `taskset`, sees that share)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, smax = [], set(), None
        try:
            with open(self.path) as f:
                for line in f:
                    c = [x.strip() for x in line.split(",")]
                    if len(c) < 9:
                        continue
                    try:
                        sm.append(float(c[1]))
                        smax = float(c[2])
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                        "sw_power_cap"), c[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = smax
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def algorithmic_bytes(s: dict, group: str) -> float:
    """Compulsory HBM bytes of one kernel group over the replayed region (DESIGN.md 5):
    every input read once, every output written once; re-reads that hit L2/smem are
    not counted."""
    if group == "lin_chunk":
        # pair-moment kernel: every correspondence of an association streamed ONCE (lossless f32
        # SoA, 36 B planar / 24 B point); the 1056 B cache entries it writes are < 2 % of that
        return 36.0 * s["assoc_planar"] + 24.0 * s["assoc_point"]
    if group == "lin_finalize":
        # cached evaluation: 1056 B entry read + 728 B block written per pair
        return (1056.0 + 728.0) * s["lin_pairs"]
    if group == "err_chunk":
        return 0.0
    if group == "err_finalize":
        return (1056.0 + 8.0) * s["err_pairs"]
    if group in ("extract_select", "extract_normals", "extract_pack"):
        # scan read (16 B/pt) + keypoint records written (32 B planar, 16 B point)
        return 16.0 * s["points"] + 32.0 * s["planar_kp"] + 16.0 * s["point_kp"]
    if group == "assoc_nn":
        # query record + 27 hash slots (16 B) + one 32 B candidate sector per probed voxel
        # (lower bound) + 16 B match record
        return s["assoc_queries"] * (32.0 + 27 * 16.0 + 32.0 + 16.0)
    if group == "segment":
        return s["assoc_queries"] * (16.0 + 36.0 + 32.0)
    return 0.0  # map_build / commit: the replay does not count their units


def ncu_capture(group: str):
    """DRAM traffic of one launch of a kernel group, MEASURED by `ncu --set full` (dram__bytes_read.sum
    + dram__bytes_write.sum) and committed with the launch it belongs to in profiles/ncu_capture.json
    (written from the .ncu-rep by profiles/ncu_capture.py).  Not scaled to this run: the entry names
    its own launch (queries, duration), so the reader can compare bytes per unit."""
    path = os.path.join(ROOT, "profiles", "ncu_capture.json")
    try:
        with open(path) as f:
            return json.load(f).get(group)
    except (OSError, ValueError):
        return None



def whole_step_bytes(s: dict) -> float:
    """SURVEY 8(d) B_scan - the REFERENCE ALGORITHM's compulsory traffic (every linearisation
    streams its correspondences) - with this implementation's record sizes."""
    return (16.0 * s["points"] + 32.0 * s["planar_kp"] + 16.0 * s["point_kp"]
            + s["assoc_queries"] * (32.0 + 27 * 16.0 + 32.0 + 16.0)
            + 36.0 * (s["lin_planar"] + s["err_planar"]) + 24.0 * (s["lin_point"] + s["err_point"])
            + 728.0 * s["lin_pairs"] + 8.0 * s["err_pairs"]
            + 32.0 * s["novel_planar"] + 16.0 * s["novel_point"])


def own_step_bytes(s: dict) -> float:
    """The same step with THIS implementation's algorithm: correspondences are streamed once per
    association (pair-moment cache), linearisations read and write per-pair records only."""
    return (16.0 * s["points"] + 32.0 * s["planar_kp"] + 16.0 * s["point_kp"]
            + s["assoc_queries"] * (32.0 + 27 * 16.0 + 32.0 + 16.0)
            + 36.0 * s["assoc_planar"] + 24.0 * s["assoc_point"]
            + (1056.0 + 728.0) * s["lin_pairs"] + (1056.0 + 8.0) * s["err_pairs"]
            + 32.0 * s["novel_planar"] + 16.0 * s["novel_point"])


def sum_stats(list_of_stats):
    out = {}
    for st in list_of_stats:
        for k, v in st.items():
            out[k] = out.get(k, 0) + v
    return out


def sequence_id(rank: int, m: int) -> int:
    """Distinct synthetic sequence per (GPU, slot)."""
    return rank * 1000 + m


DUMP_BUDGET = 64 << 20  # bytes of .npy data that --dump-outputs may write


def dump_sequences(M: int) -> list:
    """The sequences (slots of rank 0) whose outputs --dump-outputs writes: 8 drawn with a fixed
    seed from the first 32, which every automatic --sequences-per-gpu has, so that runs on hosts
    with different free memory still dump the same sequences."""
    pool = min(M, 32)
    return sorted(int(m) for m in np.random.default_rng(0).choice(pool, size=min(pool, 8), replace=False))


def write_outputs(out_dir: str, dumped: dict):
    """DIR/<leg>_<name>.npy, float64, one row per record; column 0 is the sequence.  `leg` is
    `value` (device-resident scans) or `e2e` (host scans, so the keypoints come back too); every
    record of the last timed scan of each dumped sequence, in call order.  Over DUMP_BUDGET, rows
    are thinned by a fixed seed."""
    def columns(a):
        if a.dtype.names is None:
            return a.reshape(a.shape[0], int(np.prod(a.shape[1:]))).astype(np.float64)
        return np.stack([a[f].astype(np.float64) for f in a.dtype.names], axis=1)

    names = {"counts": "pair_counts", "blocks": "blocks", "errors": "errors", "keypoint_counts": "keypoint_counts",
             "planar": "planar_keypoints", "point": "point_keypoints"}
    arrays = {}
    for leg, per_seq in dumped.items():
        for name, file_name in names.items():
            out = np.concatenate([np.column_stack([np.full(len(c[name]), float(m)), columns(c[name])])
                                  for m, c in sorted(per_seq.items())])
            if len(out):  # value leg: no keypoints come back; fused LM schedule: no error calls
                arrays[f"{leg}_{file_name}"] = out
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BUDGET:
        rng = np.random.default_rng(0)
        for k, a in arrays.items():
            keep = int(len(a) * DUMP_BUDGET / total * 0.99)
            arrays[k] = a[np.sort(rng.choice(len(a), size=keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    import torch

    from form_b200 import _capi, synth
    from form_b200.pipeline import BatchReplay, Estimator, Replay, run_batches

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rows, cols = synth.shape(args.sensor)
    n_points = rows * cols
    W, K = args.warmup, args.steps
    P0 = max(0, args.preroll)
    W0 = P0 + W  # first timed scan
    S = W0 + K
    cores = host_cores()
    sched_cores = args.emulate_cores if args.emulate_cores > 0 else cores  # cores of the timed region
    M = args.sequences_per_gpu
    if M <= 0:
        # auto: 128 sequences keep the GPU ~8 % busier than 64 (measured), but their scans take
        # S x 2 MiB of page-locked host memory each - only when every rank of the box has ample room
        import psutil

        per_seq = S * n_points * 16
        # the largest multiple of 16 (at most 128, at least 32) whose page-locked scans fit this rank's
        # share of the free host memory twice over
        share = psutil.virtual_memory().available / max(world, 1)
        M = int(max(32, min(128, (share / (2 * per_seq)) // 16 * 16)))
    # G batches (one stream each) driven by T host threads: a thread queues a round on each of
    # its batches (formgpu_batch_submit_async) before it waits for the first, so G rounds are in
    # flight however few cores the rank has.  T never exceeds the rank's spare cores, so the
    # waiting threads spin without competing with each other (no FORMGPU_YIELD_WAIT).
    spare = max(1, sched_cores // max(world, 1) - 1)
    G = max(1, min(args.batches_per_gpu, M))
    T = max(1, min(G, spare, args.host_threads if args.host_threads > 0 else G))
    p = _capi.default_est_params(rows, cols, record_trace=1, device=local_rank)
    pool = ThreadPoolExecutor(max_workers=max(1, min(16, cores // max(world, 1))))

    # ---- M synthetic sequences: pinned host copies and device-resident copies ----
    t0 = time.time()
    host_pinned = True
    try:
        pinned = [torch.empty((S, n_points, 4), dtype=torch.float32).pin_memory() for _ in range(M)]
    except RuntimeError:  # not enough lockable host memory: pageable scans (slower e2e, same results)
        host_pinned = False
        pinned = [torch.empty((S, n_points, 4), dtype=torch.float32) for _ in range(M)]
    host_np = [t.numpy().view(_capi.POINT4F).reshape(S, n_points) for t in pinned]

    def gen(job):
        m, k = job
        host_np[m][k][:] = synth.scan(args.sensor, sequence_id(rank, m), k, 1)

    list(pool.map(gen, [(m, k) for m in range(M) for k in range(S)]))
    dev = [t.cuda(non_blocking=True) for t in pinned]
    torch.cuda.synchronize()
    dev_ptrs = [[d[k].data_ptr() for k in range(S)] for d in dev]
    host_ptrs = [[h[k].ctypes.data for k in range(S)] for h in host_np]
    t_gen = time.time() - t0

    # ---- untimed recording pass: the real pipeline (host smoother in the loop) per sequence ----
    t0 = time.time()

    def record(m):
        e = Estimator(_capi.default_est_params(rows, cols, record_trace=1, device=local_rank))
        for k in range(S):
            e.register_scan(host_np[m][k])
        return e

    ests = list(pool.map(record, range(M)))
    t_record = time.time() - t0
    traces = [e.trace() for e in ests]
    est_stats = sum_stats([e.stats() for e in ests])
    g0, gk = synth.gt_pose(sequence_id(rank, 0), 0), synth.gt_pose(sequence_id(rank, 0), S - 1)
    rel_gt = g0["R"].reshape(3, 3).T @ (gk["t"] - g0["t"])
    final_err = float(np.linalg.norm(ests[0].pose()["t"] - rel_gt))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    groups = [list(range(g, M, G)) for g in range(G)]
    dumped = {}  # leg -> {sequence: what the calls of its last timed scan returned}

    def timed_batched(ptr_table, on_device, leg):
        """G concurrent batches replay scans W..S of their sequences; device time by CUDA
        events on the current stream around a full-device synchronize on both sides."""
        reps = [BatchReplay([traces[i] for i in grp], p) for grp in groups]
        gptrs = [[ptr_table[i] for i in grp] for grp in groups]
        run_batches(reps, 0, W0, gptrs, on_device, T)  # pre-roll + warm-up: fills every fixed-lag window
        for r_ in reps:
            r_.reset_stats()
        if args.dump_outputs:  # only the dumped sequences copy their records inside the timed region
            for m in dump_sequences(M):
                reps[m % G].capture_last_scan(m // G)
        launches0 = sum(r_.launch_count() for r_ in reps)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        t_host = run_batches(reps, W0, S, gptrs, on_device, T)
        torch.cuda.synchronize()
        b.record()
        torch.cuda.synchronize()
        t_dev = a.elapsed_time(b) / 1e3
        st = sum_stats([r_.stats() for r_ in reps])
        launches = sum(r_.launch_count() for r_ in reps) - launches0
        if args.dump_outputs:
            dumped[leg] = {m: reps[m % G].captured(m // G) for m in dump_sequences(M)}
        for r_ in reps:
            r_.close()
        return t_dev, t_host, st, launches

    if args.emulate_cores > 0:  # development aid: the timed legs run on a share of the box's cores
        os.sched_setaffinity(0, sorted(os.sched_getaffinity(0))[: args.emulate_cores])
    # ---- value: scans resident in HBM ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    if args.only_profile:  # development aid: only the per-kernel-group event timing
        sampler.stop()
        rp = BatchReplay(traces, p)
        rp.run(0, W0, dev_ptrs)
        rp.reset_stats()
        rp.profile_read()
        rp.profile_enable(True)
        rp.run(W0, S, dev_ptrs)
        prof = rp.profile_read()
        rp.close()
        return {g: round(1e3 * v["ms"] / (M * K), 2) for g, v in sorted(prof.items()) if v["launches"]} if rank == 0 else None
    if args.only_e2e:  # development aid: only the host-buffer leg
        t_e2e, _, _, _ = timed_batched(host_ptrs, False, "e2e")
        sampler.stop()
        return {"sequences_per_gpu": M, "batches_per_gpu": G, "e2e": round(M * K / t_e2e, 2)} if rank == 0 else None
    t_value, t_value_host, stats_d, gpu_launches = timed_batched(dev_ptrs, True, "value")
    if args.only_value:  # development aid (configuration sweeps): not a bench line
        sampler.stop()
        return {"sequences_per_gpu": M, "batches_per_gpu": G, "value": round(M * K / t_value, 2),
                "setup_s": round(t_gen + t_record, 1)} if rank == 0 else None
    # ---- e2e: pinned host scans in, f64 keypoints + blocks out, through the same C-ABI ----
    t_e2e, _, stats_h, _ = timed_batched(host_ptrs, False, "e2e")
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, dumped)

    # ---- per-kernel-group CUDA-event timing of the same region: ONE batch with all M
    # sequences, events around every launch (this inflates short launches by a few us) ----
    rp = BatchReplay(traces, p)
    rp.run(0, W0, dev_ptrs)
    rp.reset_stats()
    rp.profile_read()
    rp.profile_enable(True)
    t_prof, rounds = rp.run(W0, S, dev_ptrs)
    prof = rp.profile_read()
    rp.profile_enable(False)
    stats_p = rp.stats()
    rp.close()

    # ---- latency mode: ONE sequence, the single-context entry points ----
    single = run_single(torch, Replay, traces[0], p, dev_ptrs[0], host_np[0], W0, S, n_points)

    # max over ranks, whole-job aggregate
    if dist is not None:
        t = torch.tensor([t_value, t_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_value, t_e2e = float(t[0]), float(t[1])
    total_scans = world * M * K
    value = total_scans / t_value
    e2e_value = total_scans / t_e2e

    result = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        kernel_ms = {g: v["ms"] for g, v in prof.items() if v["launches"]}
        total_kernel_ms = sum(kernel_ms.values()) or 1.0
        dom = max(kernel_ms, key=kernel_ms.get)
        kg = {}
        for g, ms in sorted(kernel_ms.items()):
            ab = algorithmic_bytes(stats_p, g)
            n = prof[g]["launches"]
            kg[g] = {"ms_per_scan": round(ms / (M * K), 6), "launches": n,
                     "avg_launch_us": round(1e3 * ms / n, 2),
                     "algorithmic_MB_per_launch": round(ab / n / 1e6, 3),
                     "achieved_GBps": round(ab / (ms / 1e3) / 1e9, 1),
                     "frac": round(ab / (ms / 1e3) / 1e9 / peak, 4),
                     "share_of_gpu_time": round(ms / total_kernel_ms, 4)}
        cap = ncu_capture(dom)
        roofline = {
            "bound": "hbm", "kernel": dom, "achieved": kg[dom]["achieved_GBps"], "peak": peak,
            "unit": "GB/s", "frac": kg[dom]["frac"],
            # measured DRAM bytes of ONE launch of this kernel (ncu --set full), with the launch it
            # was measured on; null when no capture of the dominant kernel is committed
            "traffic": cap["dram_bytes"] if cap else None,
            "traffic_capture": cap,
            "dram_frac": round(cap["dram_GBps"] / peak, 4) if cap else None,
            "note": "frac = SURVEY 8(d) algorithmic bytes (the reference algorithm's probes: 27 hash slots "
                    "per query) / CUDA-event time; the kernel keeps its working set in L1/L2 and is bound "
                    "by instruction issue and L2 latency, so dram_frac (measured DRAM bytes / time / peak) "
                    "is what it really asks of HBM",
            "peak_source": peak_src,
            "algorithmic_bytes_per_launch": round(kg[dom]["algorithmic_MB_per_launch"] * 1e6),
            "avg_launch_us": kg[dom]["avg_launch_us"], "launches": kg[dom]["launches"],
            "kernel_share_of_gpu_time": kg[dom]["share_of_gpu_time"],
            "measured_on": f"one batch of all {M} sequences, CUDA events around every launch "
                           f"({rounds} submits, {round(M * K / t_prof, 1)} scans/s under profiling)",
            "kernel_groups": kg,
            "whole_step_algorithmic_GBps": round(whole_step_bytes(stats_d) / t_value / 1e9, 2),
            "whole_step_frac": round(whole_step_bytes(stats_d) / t_value / 1e9 / peak, 4),
            "whole_step_note": "reference algorithm's compulsory bytes per step (every linearisation "
                               "streams its correspondences) / measured step time",
            "own_algorithm_step_GBps": round(own_step_bytes(stats_d) / t_value / 1e9, 2),
            "own_algorithm_step_frac": round(own_step_bytes(stats_d) / t_value / 1e9 / peak, 4),
        }
        h2d = 16.0 * n_points  # the scan (requests are < 1% of it)
        d2h = (72.0 * stats_h["planar_kp"] + 40.0 * stats_h["point_kp"] + 728.0 * stats_h["lin_pairs"]
               + 8.0 * stats_h["err_pairs"] + stats_h["assoc_calls"] * 4 * 4 * (p.hot.max_window_scans + 1)) / (M * K)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_multi(args, rows, cols, W0, S, host_np)
        n_seq_scans = M * S
        result = {
            "metric": METRIC, "value": round(value, 3),
            "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(1e3 * t_value / (M * K), 5), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic", "mpoints_per_s": round(value * n_points / 1e6, 3),
            "config": {
                "workload": SENSOR_OF_WORKLOAD[args.sensor] + f"; {M} independent sequences per GPU "
                            f"advanced in lock step (formgpu_batch_submit), {G} concurrent batches",
                "sensor": args.sensor, "rows": rows, "cols": cols, "scans_per_sequence": S,
                "preroll_scans": P0,
                "steady_state": f"{P0} untimed pre-roll scans + {W} warm-up scans per sequence precede the "
                                f"timed ones, so the fixed-lag window is at its steady size from the first "
                                f"timed scan whatever --warmup is",
                "sequences_per_gpu": M, "batches_per_gpu": G, "sequences": world * M,
                "host_threads_per_gpu": T,
                "host_wait": "spin; a thread pipelines its batches (submit_async to each, then wait)",
                "step": "hot-path calls of one scan of one sequence, replayed from the recorded pipeline "
                        "trace; `steps` timed scans per sequence after `warmup` untimed ones",
                "l2": f"inputs larger than L2: every round touches {M} scans + {M} maps (> 126 MB); no flush",
                "timing": "CUDA events around the timed region with a device-wide synchronize on both "
                          "sides (work runs on one stream per batch), max over ranks",
                "host_wall_s_value_leg": round(t_value_host, 4),
                "icp_iterations_per_scan": round(est_stats["icp_iterations"] / n_seq_scans, 2),
                "lm_iterations_per_scan": round(est_stats["lm_iterations"] / n_seq_scans, 2),
                "lm_schedule": "fused: trial steps are linearised (error = f/2), accepted blocks reused",
                "stage3": "pair-moment cache: correspondences streamed once per association, every "
                          "linearize / error call is a per-pair 13x13 congruence (moments.cu)",
                "correspondences_streamed_per_step": round((stats_d["assoc_planar"] + stats_d["assoc_point"]) / (M * K)),
                "window_size_mean": round(est_stats["window_size"] / M, 1),
                "pipeline_final_position_error_m": round(final_err, 4),
                "assoc_calls_per_step": round(stats_d["assoc_calls"] / (M * K), 2),
                "linearize_calls_per_step": round(stats_d["lin_calls"] / (M * K), 2),
                "correspondences_linearized_per_step": round((stats_d["lin_planar"] + stats_d["lin_point"]) / (M * K)),
                "keypoints_per_scan": round((stats_d["planar_kp"] + stats_d["point_kp"]) / (M * K)),
                "parallelism": f"{world} GPU(s) x {M} independent sequences, no collective",
                "recording_pass_s": round(t_record, 2), "scan_generation_s": round(t_gen, 2),
                "host_scans_pinned": host_pinned,
            },
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 3), "unit": "scans/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": round(1e3 * t_e2e / (M * K), 5)},
            "gpu_launches": int(gpu_launches),
            "roofline": roofline,
            "single_sequence": single,
            "live_pipeline": {
                "value": round(M * S / t_record, 2), "unit": "scans/s",
                "what": f"the untimed recording pass: {M} live form::Estimators (host smoother, key-scan "
                        f"logic and LM in the loop, one private context each) on {pool._max_workers} host "
                        f"threads, all {S} scans per sequence - the drop-in rate with nothing replayed"},
            "cpu_baseline": cpu,
        }
        if cpu:
            result["config"]["speedup_value_vs_cpu"] = round(value / cpu["value"], 2)
            result["config"]["speedup_e2e_vs_cpu"] = round(e2e_value / cpu["value"], 2)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return result


# ---------------------------------------------------------------------------------------------
# --mode sharded: BASELINE.json configs[4] - ONE dense 128x2048 sequence against a map of about a
# million occupied voxels, point-sharded over the ranks (formgpu_comm_init): strong scaling
# ---------------------------------------------------------------------------------------------
STRESS_TILES = 40  # far tiles that seed the map: ~25 k planar + ~5 k point voxels each
STRESS_ICP = 4     # associate_linearize calls per scan (ICP iterations)
STRESS_FULL = 2    # full-window linearisations per scan
STRESS_KEEP = 8    # scans of the driven tile kept in the window


def run_sharded(args, rank, world, local_rank):
    import torch

    from form_b200 import _capi, synth
    from form_b200.context import Context
    from helpers import perturbed, scan_poses

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sensor = "stress-128x2048"
    rows, cols = synth.shape(sensor)
    n_points = rows * cols
    W, K = args.warmup, args.steps
    S = W + K
    params = _capi.default_params(rows, cols)
    scans = [synth.stress_scan(0, k) for k in range(S)]
    pinned = [torch.from_numpy(s.view(np.uint8)).pin_memory() for s in scans]
    dev = [t.cuda() for t in pinned]
    host_np = [t.numpy().view(_capi.POINT4F) for t in pinned]
    seeds = [synth.stress_scan(t, 0) for t in range(1, STRESS_TILES + 1)]
    torch.cuda.synchronize()
    side = torch.cuda.Stream()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    rng0 = np.random.default_rng(5)  # same stream on every rank: identical calls
    trial_pose = [[perturbed(synth.stress_pose(0, k), rng0, 0.002 / (it + 1), 0.02 / (it + 1))
                   for it in range(STRESS_ICP)] for k in range(S)]

    def one_pass(on_device, profile=False):
        """Seeds the map, then drives scans 0..S-1 of tile 0; returns (seconds of the timed scans,
        work counters, kernel-group profile, launches)."""
        st = dict(points=0, planar_kp=0, point_kp=0, assoc_calls=0, assoc_queries=0, assoc_corr=0,
                  lin_calls=0, lin_pairs=0, lin_corr=0)
        with torch.cuda.stream(side), Context(params, device=local_rank, stream=side.cuda_stream) as ctx:
            if world > 1:  # a fresh NCCL id per communicator (rank 0 creates, torch.distributed carries it)
                ident = [Context.comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(ident, src=0)
                ctx.comm_init(ident[0], rank, world)
            poses, counts_of = {}, {}
            ctx.map_rebuild(scan_poses([], []))
            for t, scan in enumerate(seeds, start=1):
                ctx.extract(scan, t)
                poses[t] = synth.stress_pose(t, 0)
                ctx.associate(poses[t])
                ctx.commit_scan()
            seed_arr = scan_poses(sorted(poses), [poses[s] for s in sorted(poses)])  # never changes
            n_seed = len(poses)

            def window_poses():
                own = sorted(poses)[n_seed:]  # the driven tile's scans (ids >= 1000)
                return np.concatenate([seed_arr, scan_poses(own, [poses[s] for s in own])])

            mine = []
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = 0
            for k in range(S):
                if k == W:
                    if profile:
                        ctx.profile_read()
                        ctx.profile_enable(True)
                    for key in st:
                        st[key] = 0
                    l0 = ctx.launch_count()
                    barrier()
                    a.record(side)
                idx = 1000 + k
                if on_device:
                    n_pl, n_pt = ctx.extract_device(dev[k].data_ptr(), n_points, idx)
                else:
                    pl, pt = ctx.extract(host_np[k], idx)
                    n_pl, n_pt = len(pl), len(pt)
                ctx.map_rebuild(window_poses())
                counts = None
                for it in range(STRESS_ICP):
                    poses[idx] = trial_pose[k][it]
                    counts, _ = ctx.associate_linearize(window_poses())
                    corr = int(counts["n_planar"].sum() + counts["n_point"].sum())
                    st["assoc_calls"] += 1
                    st["assoc_queries"] += n_pl + n_pt
                    st["assoc_corr"] += corr
                    st["lin_calls"] += 1
                    st["lin_pairs"] += len(counts)
                    st["lin_corr"] += corr
                counts_of[idx] = counts
                all_poses = window_poses()
                pairs = np.zeros(sum(len(c) for c in counts_of.values()), dtype=_capi.PAIR)
                at = 0
                for j in sorted(counts_of):
                    pairs["i"][at:at + len(counts_of[j])] = counts_of[j]["i"]
                    pairs["j"][at:at + len(counts_of[j])] = j
                    at += len(counts_of[j])
                for _ in range(STRESS_FULL):
                    if len(pairs):
                        ctx.linearize(pairs, all_poses)
                        st["lin_calls"] += 1
                        st["lin_pairs"] += len(pairs)
                        st["lin_corr"] += sum(int(c["n_planar"].sum() + c["n_point"].sum()) for c in counts_of.values())
                ctx.commit_scan()
                mine.append(idx)
                if len(mine) > STRESS_KEEP:
                    old = mine.pop(0)
                    ctx.remove_scans([old])
                    poses.pop(old)
                    counts_of.pop(old)
                    for j in counts_of:
                        counts_of[j] = counts_of[j][counts_of[j]["i"] != old]
                st["points"] += n_points
                st["planar_kp"] += n_pl
                st["point_kp"] += n_pt
            ctx.synchronize()
            b.record(side)
            torch.cuda.synchronize()
            seconds = a.elapsed_time(b) / 1e3
            prof = ctx.profile_read() if profile else None
            launches = ctx.launch_count() - l0
            if world > 1:
                ctx.comm_destroy()
        return seconds, st, prof, launches

    sampler = ClockSampler(local_rank)
    sampler.start()
    t_value, st, _, launches = one_pass(True)
    t_e2e, st_h, _, _ = one_pass(False)
    barrier()
    clocks = sampler.stop()
    _, st_p, prof, _ = one_pass(True, profile=True)
    if dist is not None:
        t = torch.tensor([t_value, t_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_value, t_e2e = float(t[0]), float(t[1])
    result = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        kernel_ms = {g: v["ms"] for g, v in prof.items() if v["launches"]}
        total_ms = sum(kernel_ms.values()) or 1.0
        ab_of = {"assoc_nn": st_p["assoc_queries"] * (32.0 + 27 * 16.0 + 32.0 + 16.0),
                 "segment": st_p["assoc_queries"] * (16.0 + 36.0 + 32.0),
                 "lin_chunk": 36.0 * st_p["assoc_corr"],
                 "lin_finalize": (1056.0 + 728.0) * st_p["lin_pairs"],
                 "extract_select": 16.0 * st_p["points"], "extract_normals": 16.0 * st_p["points"],
                 "extract_pack": 32.0 * st_p["planar_kp"] + 16.0 * st_p["point_kp"]}
        kg = {}
        for g, ms in sorted(kernel_ms.items()):
            n = prof[g]["launches"]
            ab = ab_of.get(g, 0.0) / max(world, 1) if g in ("assoc_nn", "lin_chunk") else ab_of.get(g, 0.0)
            kg[g] = {"ms_per_scan": round(ms / K, 5), "launches": n, "avg_launch_us": round(1e3 * ms / n, 2),
                     "algorithmic_MB_per_launch": round(ab / n / 1e6, 3),
                     "achieved_GBps": round(ab / (ms / 1e3) / 1e9, 1), "frac": round(ab / (ms / 1e3) / 1e9 / peak, 4),
                     "share_of_gpu_time": round(ms / total_ms, 4)}
        dom = max(kernel_ms, key=kernel_ms.get)
        cap = ncu_capture(dom + "_single")
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_sharded(args, rows, cols, scans, seeds)
        value, e2e_value = K / t_value, K / t_e2e
        result = {
            "metric": METRIC, "value": round(value, 3), "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(1e3 * t_value / K, 4), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "mpoints_per_s": round(value * n_points / 1e6, 3),
            "config": {
                "workload": SENSOR_OF_WORKLOAD[sensor] + f"; ONE sequence point-sharded over {world} GPU(s) "
                            f"(formgpu_comm_init): map seeded with {STRESS_TILES} far tiles (~1.2 M occupied voxels, "
                            f"1.5 M points) + the last {STRESS_KEEP} scans of the driven tile",
                "sensor": sensor, "rows": rows, "cols": cols,
                "step": f"extract + reparative rebuild of the whole map + {STRESS_ICP} x associate_linearize at "
                        f"perturbed poses + {STRESS_FULL} x linearize of every pair of the driven tile + commit "
                        f"(fixed schedule, no smoother in the loop)",
                "parallelism": f"{world} rank(s): keypoint-sharded association (all-gather of matches), "
                               f"correspondence-sharded pair moments, ncclAllReduce of 91 doubles per pair; "
                               f"extraction and map rebuild replicated",
                "l2": "the map (1.5 M points x 32 B + 16 MB hash) exceeds L2 and is rebuilt every step; no flush",
                "timing": "CUDA events on the context's stream, barrier + device synchronize on both sides, max over ranks",
                "keypoints_per_scan": round((st["planar_kp"] + st["point_kp"]) / K),
                "correspondences_per_association": round(st["assoc_corr"] / max(st["assoc_calls"], 1)),
            },
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 3), "unit": "scans/s", "h2d_bytes_per_step": 16 * n_points,
                    "d2h_bytes_per_step": int((72.0 * st_h["planar_kp"] + 40.0 * st_h["point_kp"] + 728.0 * st_h["lin_pairs"]) / K),
                    "ms_per_step": round(1e3 * t_e2e / K, 4)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": kg[dom]["achieved_GBps"], "peak": peak, "unit": "GB/s",
                         "frac": kg[dom]["frac"], "traffic": cap["dram_bytes"] if cap else None, "traffic_capture": cap,
                         "peak_source": peak_src, "kernel_groups": kg},
            "cpu_baseline": cpu,
        }
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return result


def cpu_baseline_sharded(args, rows, cols, scans, seeds):
    """The same fixed schedule on the CPU oracle (all host threads over keypoints, as the
    reference's TBB loops), bounded sample of 3 scans after the map is seeded."""
    import oracle_lib
    from form_b200 import _capi, synth
    from helpers import perturbed, scan_poses

    params = _capi.default_params(rows, cols)
    ref = oracle_lib.Oracle(params)
    rng = np.random.default_rng(5)
    poses, counts_of = {}, {}
    ref.map_rebuild(scan_poses([], []))
    for t, scan in enumerate(seeds, start=1):
        ref.extract(scan, t)
        poses[t] = synth.stress_pose(t, 0)
        ref.associate(poses[t])
        ref.commit_scan()
    n = min(3, len(scans))
    t0 = time.perf_counter()
    for k in range(n):
        idx = 1000 + k
        ref.extract(scans[k], idx)
        window = sorted(poses)
        ref.map_rebuild(scan_poses(window, [poses[s] for s in window]))
        counts = None
        for it in range(STRESS_ICP):
            poses[idx] = perturbed(synth.stress_pose(0, k), rng, 0.002 / (it + 1), 0.02 / (it + 1))
            now = sorted(poses)
            all_poses = scan_poses(now, [poses[s] for s in now])
            counts = ref.associate(poses[idx])
            if len(counts):
                pairs = np.zeros(len(counts), dtype=_capi.PAIR)
                pairs["i"], pairs["j"] = counts["i"], idx
                ref.linearize(pairs, all_poses)
        counts_of[idx] = counts
        now = sorted(poses)
        all_poses = scan_poses(now, [poses[s] for s in now])
        pairs = np.array([(int(c["i"]), j) for j in sorted(counts_of) for c in counts_of[j]], dtype=_capi.PAIR)
        for _ in range(STRESS_FULL):
            if len(pairs):
                ref.linearize(pairs, all_poses)
        ref.commit_scan()
    dt = time.perf_counter() - t0
    return {"value": round(n / dt, 4), "unit": "scans/s", "cores": host_cores(), "kind": "port",
            "sample": f"{n} scans of the same fixed schedule on the oracle after seeding the map, {round(dt, 1)} s; "
                      f"worker threads over keypoints where the reference uses TBB"}


def run_single(torch, Replay, trace, p, dev_ptrs, scans_np, W, S, n_points):
    """Latency mode: one sequence through the single-context entry points.  Per-step CUDA
    events on the launching stream, 256 MiB L2 flush between steps (outside the intervals)."""
    K = S - W
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    pinned_np = [scans_np[k] for k in range(S)]

    def timed(run):
        ms = []
        for s in range(W, S):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            run(s, s + 1)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return sum(ms) / 1e3

    rep_d = Replay(trace, p, stream=stream)
    rep_d.run_device(0, W, dev_ptrs)
    t_d = timed(lambda a, b: rep_d.run_device(a, b, dev_ptrs))
    rep_d.close()
    rep_h = Replay(trace, p, stream=stream)
    rep_h.run_host(0, W, pinned_np)
    t_h = timed(lambda a, b: rep_h.run_host(a, b, pinned_np))
    rep_h.close()
    rep_p = Replay(trace, p, stream=stream)
    rep_p.run_device(0, W, dev_ptrs)
    rep_p.reset_stats()
    rep_p.profile_read()
    rep_p.profile_enable(True)
    for s in range(W, S):
        flush.zero_()
        rep_p.run_device(s, s + 1, dev_ptrs)
    prof = rep_p.profile_read()
    rep_p.profile_enable(False)
    st = rep_p.stats()
    rep_p.close()
    peak, _ = measured_peaks()
    kernel_ms = {g: v["ms"] for g, v in prof.items() if v["launches"]}
    dom = max(kernel_ms, key=kernel_ms.get)
    ab = algorithmic_bytes(st, dom)
    return {
        "what": "ONE sequence per GPU through the single-context C-ABI calls (latency mode): "
                "~45 dependent device calls per scan",
        "value": round(K / t_d, 3), "unit": "scans/s", "ms_per_scan": round(1e3 * t_d / K, 4),
        "e2e": round(K / t_h, 3), "e2e_ms_per_scan": round(1e3 * t_h / K, 4),
        "mpoints_per_s": round(K / t_d * n_points / 1e6, 2),
        "l2": "256 MiB buffer written between timed steps (outside the timed intervals)",
        "dominant_kernel": dom,
        "dominant_frac_of_hbm_peak": round(ab / (kernel_ms[dom] / 1e3) / 1e9 / peak, 5),
        "dominant_avg_launch_us": round(1e3 * kernel_ms[dom] / prof[dom]["launches"], 2),
        "kernel_ms_per_scan": {g: round(v / K, 5) for g, v in sorted(kernel_ms.items())},
    }


def cpu_multi_sequence(rows, cols, W, last, scans_of, n_workers, gtsam_schedule=1, live=None):
    """The multi-sequence job on the CPU oracle: one single-threaded worker per host core,
    each recording (untimed) and then replaying the hot-path calls of scans W..last-1 of its
    own sequence after an untimed window warm-up.  gtsam_schedule=1: the reference's LM schedule
    (one linearisation per iteration + one error evaluation per trial); 0: the fused schedule
    our arm replays (every trial linearised).  `live` (a dict) receives the rate of the recording
    pass itself - the whole pipeline with the host smoother in the loop - over scans W..last-1.
    Returns (scans/s over all workers, seconds)."""
    import oracle_lib
    from form_b200 import _capi

    p = _capi.default_est_params(rows, cols, record_trace=1, gtsam_lm_schedule=gtsam_schedule, num_threads=1)
    oracle_lib._pipe_lib()  # load and configure the library here, before the worker threads use it
    _capi.synth_lib()

    def prepare(w):
        scans = scans_of(w)
        est = oracle_lib.OracleEstimator(p)
        for s in scans[:W]:
            est.register_scan(s)
        t0 = time.perf_counter()
        for s in scans[W:last]:
            est.register_scan(s)
        t_live = time.perf_counter() - t0
        ro = oracle_lib.OracleReplay(est.trace(), p)
        ro.run_host(0, W, scans)
        ro.reset_stats()
        return est, ro, scans, t_live

    with ThreadPoolExecutor(max_workers=n_workers) as ex:
        prepared = list(ex.map(prepare, range(n_workers)))
        if live is not None:
            live["value"] = round(sum((last - W) / pr[3] for pr in prepared), 4)
        t0 = time.perf_counter()
        list(ex.map(lambda pr: pr[1].run_host(W, last, pr[2]), prepared))
        dt = time.perf_counter() - t0
    return n_workers * (last - W) / dt, dt


def cpu_single_sequence(rows, cols, W, last, scans):
    """The reference's own threading: ONE sequence, parallel_for over keypoints on all cores."""
    import oracle_lib
    from form_b200 import _capi

    p = _capi.default_est_params(rows, cols, record_trace=1, gtsam_lm_schedule=1)
    est = oracle_lib.OracleEstimator(p)
    for s in scans[:last]:
        est.register_scan(s)
    ro = oracle_lib.OracleReplay(est.trace(), p)
    ro.run_host(0, W, scans)
    ro.reset_stats()
    t = ro.run_host(W, last, scans)
    return (last - W) / t


def reference_code_stage1(rows, cols, scans):
    """Extra CPU row (labelled, not the baseline): FORM's OWN extract() - the reference's
    extraction.tpp compiled unmodified into oracle/_ref/libformref.so against the API stand-ins of
    oracle/shim (so Eigen's arithmetic is a restatement and TBB is serial) - timed next to the
    restatement's extraction on the same scans, one thread each.  None when the library is absent."""
    import ctypes as C

    lib_path = os.path.join(ROOT, "oracle", "_ref", "libformref.so")
    if not os.path.exists(lib_path):
        return None
    import oracle_lib
    from form_b200 import _capi

    lib = C.CDLL(lib_path)
    psz = C.POINTER(C.c_size_t)
    lib.formref_extract.restype = C.c_int
    lib.formref_extract.argtypes = [C.POINTER(_capi.Params), C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p,
                                    C.c_size_t, psz, C.c_void_p, C.c_size_t, psz]
    params = _capi.default_params(rows, cols)
    n = rows * cols
    pl, pt = np.zeros(n, dtype=_capi.PLANAR_FEAT), np.zeros(n, dtype=_capi.POINT_FEAT)
    a, b = C.c_size_t(), C.c_size_t()
    t0 = time.perf_counter()
    for k, scan in enumerate(scans):
        if lib.formref_extract(C.byref(params), _capi.ptr(scan), n, k, _capi.ptr(pl), n, C.byref(a), _capi.ptr(pt), n,
                               C.byref(b)) != 0:
            return None
    t_ref = (time.perf_counter() - t0) / len(scans)
    o = oracle_lib.Oracle(params, threads=1)
    t0 = time.perf_counter()
    for k, scan in enumerate(scans):
        o.extract(scan, k)
    t_port = (time.perf_counter() - t0) / len(scans)
    return {"form_extract_ms_per_scan": round(1e3 * t_ref, 2), "restatement_extract_ms_per_scan": round(1e3 * t_port, 2),
            "scans": len(scans), "threads": 1,
            "what": "stage 1 only: FORM's own FeatureExtractor::extract (oracle/_ref, compiled from "
                    "/root/reference against the stand-ins of oracle/shim: restated Eigen arithmetic, serial TBB) "
                    "next to the restatement's extraction on the same scans - a check that the restatement is not "
                    "a slower baseline than the reference's code, not a baseline itself"}


def reference_code_pipeline(rows, cols, scans):
    """Extra CPU row (labelled, not the baseline): FORM's OWN Estimator::register_scan - form.cpp,
    constraints.cpp, extraction / map / matcher / factor / key-scanner sources compiled unmodified into
    oracle/_ref/libformref.so over the stand-ins of oracle/shim (restated Eigen arithmetic, serial TBB,
    GTSAM's optimiser restated) - next to the host logic over the restatement (reference LM schedule) on
    the same scans, one thread each, with the largest pose difference between the two.  None when the
    library is absent."""
    import ctypes as C

    lib_path = os.path.join(ROOT, "oracle", "_ref", "libformref.so")
    if not os.path.exists(lib_path):
        return None
    import oracle_lib
    from form_b200 import _capi

    lib = C.CDLL(lib_path)
    if not hasattr(lib, "formref_est_create"):
        return None
    psz = C.POINTER(C.c_size_t)
    lib.formref_est_create.restype = C.c_void_p
    lib.formref_est_create.argtypes = [C.POINTER(_capi.Params), C.c_double, C.c_double, C.c_int, C.c_int, C.c_int64,
                                       C.c_size_t, C.c_int64]
    lib.formref_est_destroy.argtypes = [C.c_void_p]
    lib.formref_est_register_scan.restype = C.c_int
    lib.formref_est_register_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, psz,
                                              C.c_void_p, C.c_size_t, psz]
    lib.formref_est_pose.argtypes = [C.c_void_p, C.c_void_p]
    p = _capi.default_est_params(rows, cols, num_threads=1, gtsam_lm_schedule=1)
    n = rows * cols
    h = lib.formref_est_create(C.byref(p.hot), p.new_pose_threshold, p.keyscan_match_ratio, p.max_num_rematches,
                               p.disable_smoothing, p.max_num_keyscans, p.max_num_recent_scans,
                               p.max_steps_unused_keyscan)
    ours = oracle_lib.OracleEstimator(p)
    pl, pt = np.zeros(n, dtype=_capi.PLANAR_FEAT), np.zeros(n, dtype=_capi.POINT_FEAT)
    a, b = C.c_size_t(), C.c_size_t()
    t_ref = t_port = worst = 0.0
    same_keypoints = True
    for scan in scans:
        t0 = time.perf_counter()
        rc = lib.formref_est_register_scan(h, _capi.ptr(scan), n, _capi.ptr(pl), n, C.byref(a), _capi.ptr(pt), n,
                                           C.byref(b))
        t_ref += time.perf_counter() - t0
        if rc != 0:
            lib.formref_est_destroy(h)
            return None
        t0 = time.perf_counter()
        kp, kq = ours.register_scan(scan)
        t_port += time.perf_counter() - t0
        same_keypoints = same_keypoints and kp.tobytes() == pl[: a.value].tobytes() and kq.tobytes() == pt[: b.value].tobytes()
        pr = np.zeros(1, dtype=_capi.POSE)
        lib.formref_est_pose(h, _capi.ptr(pr))
        po = ours.pose()
        worst = max(worst, float(np.linalg.norm(po["t"] - pr[0]["t"])), float(np.abs(po["R"] - pr[0]["R"]).max()))
    lib.formref_est_destroy(h)
    ours.close()
    return {"form_register_scan_ms_per_scan": round(1e3 * t_ref / len(scans), 2),
            "restatement_register_scan_ms_per_scan": round(1e3 * t_port / len(scans), 2),
            "scans": len(scans), "threads": 1, "keypoints_identical": bool(same_keypoints),
            "max_pose_difference": worst,
            "what": "the whole pipeline, smoother included: FORM's own Estimator::register_scan (oracle/_ref: form.cpp "
                    "and constraints.cpp compiled from /root/reference over stand-ins for Eigen / TBB / GTSAM) next to "
                    "this repository's host logic over the restatement, first scans of one sequence - a live check "
                    "that the two agree and that the restatement is not the slower CPU code, not a baseline itself"}


def optional_row(fn, *a):
    """The labelled extra rows must never take the bench line down with them."""
    try:
        return fn(*a)
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}


def cpu_baseline_multi(args, rows, cols, W, S, host_np):
    cores = host_cores()
    last = min(S, W + max(1, args.cpu_sample))
    n = last - W
    workers = min(cores, len(host_np))
    scans_of = lambda w: [host_np[w][k] for k in range(S)]  # noqa: E731
    live = {}
    value, dt = cpu_multi_sequence(rows, cols, W, last, scans_of, workers, 1, live)
    fused, _ = cpu_multi_sequence(rows, cols, W, last, scans_of, workers, 0)
    single = cpu_single_sequence(rows, cols, W, last, [host_np[0][k] for k in range(S)])
    return {"value": round(value, 4), "unit": "scans/s", "cores": workers, "kind": "port",
            "lm_schedule": "the reference's (GTSAM): one linearisation per LM iteration + one error "
                           "evaluation per trial step",
            "fused_schedule_value": round(fused, 4),
            "fused_schedule_note": "the same CPU job replaying the schedule our arm replays (every trial "
                                   "step linearised, accepted blocks reused): same iterates, more CPU work",
            "live_pipeline_value": live.get("value"),
            "live_pipeline_note": "the recording pass itself: the whole pipeline with the host smoother in "
                                  "the loop, one single-threaded sequence per host core",
            "sample": f"{workers} sequences x {n} scans (scans {W}..{last - 1}) after an untimed {W}-scan "
                      f"window warm-up: one single-threaded oracle replay per host core, {round(dt, 1)} s; "
                      f"oracle/ C++17 restatement, -O3 no -march",
            "ms_per_step": round(1e3 / value, 3),
            "single_sequence_reference_threading": {
                "value": round(single, 4), "unit": "scans/s", "cores": cores,
                "what": "ONE sequence, worker threads over keypoints where the reference uses TBB"},
            "reference_code_stage1": optional_row(reference_code_stage1, rows, cols, [host_np[0][k] for k in range(W, min(S, W + 4))]),
            "reference_code_pipeline": optional_row(reference_code_pipeline, rows, cols, [host_np[0][k] for k in range(min(S, 6))])}


def repo_libs_mapped():
    """Shared objects of this repository in the process's address space (/proc/self/maps)."""
    root = os.path.dirname(os.path.abspath(__file__))
    libs = set()
    try:
        with open("/proc/self/maps") as f:
            for line in f:
                path = line.split(None, 5)[-1].strip()
                if path.endswith(".so") and os.path.realpath(path).startswith(os.path.realpath(root) + os.sep):
                    libs.add(os.path.relpath(os.path.realpath(path), os.path.realpath(root)))
    except OSError:
        pass
    return sorted(libs)


def run_reference(args, rank, world):
    """The reference's own CPU path (oracle port: the reference cannot be built here) on the
    same multi-sequence job: one single-threaded sequence replay per host core."""
    if rank != 0:
        return None
    from form_b200 import synth

    rows, cols = synth.shape(args.sensor)
    W, K = args.preroll + args.warmup, args.steps  # same pre-roll + warm-up as our arm
    S = W + K
    cores = host_cores()
    workers = cores if args.sequences_per_gpu <= 0 else min(cores, args.sequences_per_gpu)
    last, n = S, K

    def scans_of(w):
        return [synth.scan(args.sensor, sequence_id(0, w), k, 1) for k in range(last)]

    value, dt = cpu_multi_sequence(rows, cols, W, last, scans_of, workers)
    n_points = rows * cols
    cpu = {"value": round(value, 4), "unit": "scans/s", "cores": workers, "kind": "port",
           "sample": f"{workers} sequences x {n} scans (scans {W}..{last - 1}) after an untimed {W}-scan "
                     f"warm-up, one single-threaded replay per host core, {round(dt, 1)} s"}
    return {
        "impl": "reference", "metric": METRIC,
        "value": round(value, 4), "unit": "scans/s", "n_gpus": world, "steps": n, "warmup": args.warmup,
        "ms_per_step": round(1e3 / value, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic", "mpoints_per_s": round(value * n_points / 1e6, 4),
        "config": {"workload": SENSOR_OF_WORKLOAD[args.sensor] + f"; {workers} independent sequences, one per host core",
                   "sensor": args.sensor, "rows": rows, "cols": cols, "scans_per_sequence": last,
                   "note": "FORM cannot be built as shipped here (Eigen3/GTSAM/oneTBB/tsl absent); this arm "
                           "is the oracle/ C++17 restatement of its hot path on the host cores - pinned to "
                           "FORM's own sources compiled over stand-ins (oracle/_ref), which run slower than "
                           "the restatement (reference_code_pipeline)"},
        "cpu_baseline": cpu,
        "e2e": {"value": round(value, 4), "unit": "scans/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        # the repository's shared objects this process has mapped: the oracle and the scan
        # generator, none of the product's (form_b200/lib/libformgpu.so, libformhost.so)
        "reference_code_pipeline": optional_row(
            reference_code_pipeline, rows, cols, [synth.scan(args.sensor, sequence_id(0, 0), k, 1) for k in range(6)]),
        "native_libs_mapped": repo_libs_mapped(),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="sequences", choices=["sequences", "sharded"],
                    help="sequences: independent sequences per GPU (the headline, weak scaling); sharded: "
                         "configs[4], ONE dense 128x2048 sequence point-sharded over the ranks (strong scaling)")
    ap.add_argument("--sensor", default="os0-128", choices=sorted(SENSOR_OF_WORKLOAD))
    ap.add_argument("--cpu-sample", type=int, default=20,
                    help="scans per sequence of the cpu_baseline row that --impl ours reports beside the GPU "
                         "value (--impl reference times --steps scans)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sequences-per-gpu", type=int, default=0,
                    help="independent sequences sharing one GPU (0 = 128 if host memory allows, else 64)")
    ap.add_argument("--only-value", action="store_true", help="development: only the device-resident leg")
    ap.add_argument("--only-e2e", action="store_true", help="development: only the host-buffer leg")
    ap.add_argument("--only-profile", action="store_true",
                    help="development: only the per-kernel-group CUDA-event times (us per scan)")
    ap.add_argument("--host-threads", type=int, default=0,
                    help="host threads driving the batches of a GPU (0 = one per batch, capped at the "
                         "rank's spare cores); a thread pipelines the batches it owns")
    ap.add_argument("--preroll", type=int, default=24,
                    help="untimed scans per sequence BEFORE the warm-up, so that the fixed-lag window has "
                         "reached its steady-state size whatever --warmup is")
    ap.add_argument("--emulate-cores", type=int, default=0,
                    help="development: restrict the timed legs to this many host cores (what a rank "
                         "gets on a box with few cores per GPU)")
    ap.add_argument("--batches-per-gpu", type=int, default=12,
                    help="the sequences of a GPU are split over this many concurrent batches (measured, 128 "
                         "sequences: 8 batches 3.6-8.7 k scans/s - one batch per host thread leaves a stream idle "
                         "whenever its thread is descheduled -, 12: 9.4-9.5 k, 16: 8.6-8.9 k, 32: 7.2 k)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the calls of the last timed scan returned (pair "
                         "counts, normal-equation blocks, error values, keypoints) for a fixed sample of "
                         "sequences as DIR/<name>.npy (float64, at most 64 MB), to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.mode != "sequences"):
        ap.error("--dump-outputs needs --impl ours --mode sequences")
    if args.dump_outputs and (args.only_value or args.only_e2e or args.only_profile):
        ap.error("--dump-outputs needs both timed legs: it cannot be combined with --only-value, --only-e2e "
                 "or --only-profile")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import __graft_entry__ as g

    # the reference arm maps the oracle and the scan generator only, never the product's libraries
    g.build(only_if_missing=True, load=args.impl != "reference")
    if args.impl == "reference":
        res = run_reference(args, rank, world)
    elif args.mode == "sharded":
        res = run_sharded(args, rank, world, local_rank)
    else:
        res = run_ours(args, rank, world, local_rank)
    if rank == 0 and res is not None:
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
