"""Batched submit (formgpu_batch_submit): the calls of several independent sequences share
one launch per kernel.  The kernel bodies are the single-sequence ones, so all index work
(keypoints, neighbour ids, pair counts, novel sets) must be BIT-identical to replaying each
sequence on its own context - and therefore to the oracle-checked single-sequence path;
normal-equation blocks agree to 1e-12 (summation order) and are run-to-run deterministic."""
import ctypes as C

import numpy as np
import pytest

from form_b200 import _capi, synth

pytestmark = pytest.mark.gpu


def _record(sensor, seq, n_scans, **overrides):
    from form_b200.pipeline import Estimator

    rows, cols = synth.shape(sensor)
    p = _capi.default_est_params(rows, cols, record_trace=1, **overrides)
    scans = [synth.scan(sensor, seq, k) for k in range(n_scans)]
    est = Estimator(p)
    for s in scans:
        est.register_scan(s)
    return est, scans, p


def test_batched_replay_is_bit_identical_to_single_contexts():
    import torch

    from form_b200.pipeline import BatchReplay, Replay

    n = 14
    runs = [_record("vlp-16", seq, n) for seq in (0, 3, 7)]
    p = runs[0][2]
    dev = [[torch.from_numpy(s.view(np.uint8)).cuda() for s in scans] for _, scans, _ in runs]
    torch.cuda.synchronize()
    ptrs = [[d.data_ptr() for d in seq] for seq in dev]
    singles = []
    for (est, scans, _), pp in zip(runs, ptrs):
        r = Replay(est.trace(), p)
        r.run_device(0, n, pp)
        singles.append(r.stats())
    br = BatchReplay([est.trace() for est, _, _ in runs], p)
    t, rounds = br.run(0, n, ptrs, on_device=True)
    assert rounds > 0 and br.launch_count() > 0
    def same(got, ref, s):
        for k in ref:
            if k == "checksum":
                # blocks are tolerance-class: a batched launch may split a pair over a different
                # number of CTAs than a single-sequence launch, which reorders the fp64 sums
                assert abs(got[k] - ref[k]) <= 1e-12 * abs(ref[k]), (s, k, got[k], ref[k])
            else:
                assert got[k] == ref[k], (s, k, got[k], ref[k])  # counts: bit-exact index work

    for s, ref in enumerate(singles):
        same(br.stats(s), ref, s)
    # far fewer launches than three separate contexts would need
    total = br.stats()
    assert total["scans"] == 3 * n
    # host-scan variant: scans uploaded and f64 keypoints written back inside the call
    bh = BatchReplay([est.trace() for est, _, _ in runs], p)
    host_ptrs = [[s.ctypes.data for s in scans] for _, scans, _ in runs]
    bh.run(0, n, host_ptrs, on_device=False)
    for s, ref in enumerate(singles):
        same(bh.stats(s), ref, s)
    # ... by default every next scan is uploaded ahead (formgpu_batch_prefetch_scan, alternating scan
    # buffers); with the prefetch off each EXTRACT request uploads its own scan: same results
    import os

    os.environ["FORM_REPLAY_PREFETCH"] = "0"
    try:
        bn = BatchReplay([est.trace() for est, _, _ in runs], p)
        bn.run(0, n, host_ptrs, on_device=False)
    finally:
        del os.environ["FORM_REPLAY_PREFETCH"]
    for s in range(3):
        assert bn.stats(s) == bh.stats(s)
    # run to run the batched path is deterministic (fixed partition, fixed reduction trees)
    b2 = BatchReplay([est.trace() for est, _, _ in runs], p)
    b2.run(0, n, ptrs, on_device=True)
    for s in range(3):
        assert b2.stats(s) == br.stats(s)


def test_captured_last_scan_is_what_its_calls_returned():
    """capture_last_scan (bench.py --dump-outputs): over a run of several scans, the records kept are
    those of its LAST scan only - keypoints as the live estimator got them, counts and blocks that
    add up to the work counters and checksum of a separate run of that one scan - and only for the
    sequences asked for."""
    import torch

    from form_b200.pipeline import BatchReplay, Estimator

    n = 8
    rows, cols = synth.shape("vlp-16")
    p = _capi.default_est_params(rows, cols, record_trace=1, gtsam_lm_schedule=1)
    runs = []
    for seq in (1, 4, 6):
        scans = [synth.scan("vlp-16", seq, k) for k in range(n)]
        est = Estimator(p)
        kp = [est.register_scan(s) for s in scans]
        runs.append((est, scans, kp[-1]))
    traces = [est.trace() for est, _, _ in runs]
    dev = [[torch.from_numpy(s.view(np.uint8)).cuda() for s in scans] for _, scans, _ in runs]
    torch.cuda.synchronize()
    got = {}
    for on_device, ptrs in ((True, [[d.data_ptr() for d in seq] for seq in dev]),
                            (False, [[s.ctypes.data for s in scans] for _, scans, _ in runs])):
        # the last scan alone, for its work counters
        one = BatchReplay(traces, p)
        one.run(0, n - 1, ptrs, on_device)
        one.reset_stats()
        one.run(n - 1, n, ptrs, on_device)
        # the same scan as the last of a three-scan run with capture on for sequences 0 and 1
        br = BatchReplay(traces, p)
        br.run(0, n - 3, ptrs, on_device)
        br.capture_last_scan(0)
        br.capture_last_scan(1)
        br.run(n - 3, n, ptrs, on_device)
        assert all(len(v) == 0 for v in br.captured(2).values())
        for s in range(2):
            c, st = br.captured(s), one.stats(s)
            kc = [int(v) for v in c["keypoint_counts"]]  # extract, then every commit
            assert kc[:2] == [st["planar_kp"], st["point_kp"]] and sum(kc[2::2]) == st["novel_planar"]
            assert int(c["counts"]["n_planar"].sum()) == st["assoc_planar"] > 0
            assert len(c["blocks"]) == st["lin_pairs"] > 0 and len(c["errors"]) == st["err_pairs"]
            cs = c["blocks"][:, 90].sum() + c["errors"].sum()
            assert abs(cs - st["checksum"]) <= 1e-12 * abs(st["checksum"])
            got[on_device, s] = c
        br.close()
        one.close()
    for s, (_, _, (pl, pt)) in enumerate(runs[:2]):
        assert len(got[True, s]["planar"]) == 0  # device-resident scans: keypoints stay on the GPU
        assert got[False, s]["planar"].tobytes() == pl.tobytes() and got[False, s]["point"].tobytes() == pt.tobytes()
        assert np.array_equal(got[False, s]["counts"], got[True, s]["counts"])
        assert np.allclose(got[False, s]["blocks"], got[True, s]["blocks"], rtol=1e-12, atol=0)


def test_batch_submit_extract_matches_oracle_and_reports_errors():
    import oracle_lib

    rows, cols = synth.shape("vlp-16")
    params = _capi.default_params(rows, cols)
    lib = _capi.gpu_lib()
    h = C.c_void_p()
    assert lib.formgpu_batch_create(C.byref(params), 0, None, 3, C.byref(h)) == 0
    try:
        assert lib.formgpu_batch_size(h) == 3
        cap_p = lib.formgpu_max_planar(lib.formgpu_batch_ctx(h, 0))
        cap_q = lib.formgpu_max_point(lib.formgpu_batch_ctx(h, 0))
        scans = [synth.scan("vlp-16", s, 1) for s in range(3)]
        planar = [np.zeros(cap_p, _capi.PLANAR_FEAT) for _ in range(3)]
        point = [np.zeros(cap_q, _capi.POINT_FEAT) for _ in range(3)]
        reqs = (_capi.Request * 3)()
        for s in range(3):
            reqs[s].sequence, reqs[s].op = s, _capi.OP_EXTRACT
            reqs[s].scan, reqs[s].n_points, reqs[s].scan_idx = scans[s].ctypes.data, rows * cols, 5 + s
            reqs[s].planar_out, reqs[s].planar_cap = planar[s].ctypes.data, cap_p
            reqs[s].point_out, reqs[s].point_cap = point[s].ctypes.data, cap_q
        assert lib.formgpu_batch_submit(h, reqs, 3) == 0
        ref = oracle_lib.Oracle(params)
        for s in range(3):
            rp, rq = ref.extract(scans[s], 5 + s)
            assert reqs[s].status == 0
            assert planar[s][: reqs[s].n_planar].tobytes() == rp.tobytes()
            assert point[s][: reqs[s].n_point].tobytes() == rq.tobytes()
        # one bad request does not stop the others
        reqs[1].n_points = 17
        rc = lib.formgpu_batch_submit(h, reqs, 3)
        assert rc == _capi.ERR_BAD_SCAN_SIZE
        assert [reqs[s].status for s in range(3)] == [0, _capi.ERR_BAD_SCAN_SIZE, 0]
        assert b"sequence 1" in lib.formgpu_batch_last_error(h)
        # two requests for the same sequence are refused
        reqs[1].n_points = rows * cols
        reqs[1].sequence = 0
        assert lib.formgpu_batch_submit(h, reqs, 3) == _capi.ERR_INVALID_ARG
    finally:
        lib.formgpu_batch_destroy(h)


def test_prefetched_scan_is_used_or_discarded():
    """formgpu_batch_prefetch_scan: the EXTRACT request that names the prefetched pointer takes the copy
    uploaded ahead (the scan buffers alternate); a request that names another scan discards it.  Either way
    the keypoints are those of the oracle for the scan the REQUEST names."""
    import oracle_lib

    rows, cols = synth.shape("vlp-16")
    params = _capi.default_params(rows, cols)
    lib = _capi.gpu_lib()
    h = C.c_void_p()
    assert lib.formgpu_batch_create(C.byref(params), 0, None, 1, C.byref(h)) == 0
    try:
        cap_p = lib.formgpu_max_planar(lib.formgpu_batch_ctx(h, 0))
        cap_q = lib.formgpu_max_point(lib.formgpu_batch_ctx(h, 0))
        scans = [synth.scan("vlp-16", 2, k) for k in range(4)]
        planar, point = np.zeros(cap_p, _capi.PLANAR_FEAT), np.zeros(cap_q, _capi.POINT_FEAT)
        ref = oracle_lib.Oracle(params)
        req = (_capi.Request * 1)()
        # (prefetched, requested): used, discarded, used again (other buffer), no prefetch at all
        for k, (pre, use) in enumerate([(0, 0), (1, 2), (3, 3), (None, 1)]):
            if pre is not None:
                assert lib.formgpu_batch_prefetch_scan(h, 0, scans[pre].ctypes.data, rows * cols) == 0
            req[0].sequence, req[0].op = 0, _capi.OP_EXTRACT
            req[0].scan, req[0].n_points, req[0].scan_idx = scans[use].ctypes.data, rows * cols, k
            req[0].planar_out, req[0].planar_cap = planar.ctypes.data, cap_p
            req[0].point_out, req[0].point_cap = point.ctypes.data, cap_q
            assert lib.formgpu_batch_submit(h, req, 1) == 0 and req[0].status == 0
            rp, rq = ref.extract(scans[use], k)
            assert planar[: req[0].n_planar].tobytes() == rp.tobytes(), (pre, use)
            assert point[: req[0].n_point].tobytes() == rq.tobytes(), (pre, use)
        assert lib.formgpu_batch_prefetch_scan(h, 0, scans[0].ctypes.data, 17) == _capi.ERR_BAD_SCAN_SIZE
        assert lib.formgpu_batch_prefetch_scan(h, 5, scans[0].ctypes.data, rows * cols) == _capi.ERR_INVALID_ARG
    finally:
        lib.formgpu_batch_destroy(h)


def test_batches_run_concurrently():
    import torch

    from form_b200.pipeline import BatchReplay, run_batches

    n = 8
    runs = [_record("vlp-16", seq, n) for seq in (1, 2)]
    p = runs[0][2]
    dev = [[torch.from_numpy(s.view(np.uint8)).cuda() for s in scans] for _, scans, _ in runs]
    torch.cuda.synchronize()
    ptrs = [[d.data_ptr() for d in seq] for seq in dev]
    traces = [est.trace() for est, _, _ in runs]
    a, b = BatchReplay(traces, p), BatchReplay(traces[::-1], p)
    t = run_batches([a, b], 0, n, [ptrs, ptrs[::-1]])
    assert t > 0
    assert a.stats(0) == b.stats(1) and a.stats(1) == b.stats(0)


def test_one_host_thread_pipelines_several_batches():
    """formgpu_batch_submit_async / formgpu_batch_wait: ONE host thread keeps a round in flight on
    each of its batches; results are those of the blocking submits."""
    import torch

    from form_b200.pipeline import BatchReplay, run_batches

    n = 8
    runs = [_record("vlp-16", seq, n) for seq in (1, 2, 6)]
    p = runs[0][2]
    dev = [[torch.from_numpy(s.view(np.uint8)).cuda() for s in scans] for _, scans, _ in runs]
    torch.cuda.synchronize()
    ptrs = [[d.data_ptr() for d in seq] for seq in dev]
    traces = [est.trace() for est, _, _ in runs]
    ref = BatchReplay(traces, p)
    ref.run(0, n, ptrs)
    reps = [BatchReplay([traces[i]], p) for i in range(3)]
    t = run_batches(reps, 0, n, [[ptrs[i]] for i in range(3)], threads=1)
    assert t > 0
    for i in range(3):
        got, want = reps[i].stats(0), ref.stats(i)
        assert {k: v for k, v in got.items() if k != "checksum"} == {k: v for k, v in want.items() if k != "checksum"}
        assert abs(got["checksum"] - want["checksum"]) <= 1e-12 * abs(want["checksum"])


def test_async_submit_state_and_failure_stamping():
    rows, cols = synth.shape("vlp-16")
    params = _capi.default_params(rows, cols)
    lib = _capi.gpu_lib()
    h = C.c_void_p()
    assert lib.formgpu_batch_create(C.byref(params), 0, None, 2, C.byref(h)) == 0
    try:
        scans = [synth.scan("vlp-16", s, 0) for s in range(2)]
        reqs = (_capi.Request * 2)()
        for s in range(2):
            reqs[s].sequence, reqs[s].op, reqs[s].flags = s, _capi.OP_EXTRACT, 0
            reqs[s].scan, reqs[s].n_points, reqs[s].scan_idx = scans[s].ctypes.data, rows * cols, s
        assert lib.formgpu_batch_done(h) == 1  # nothing in flight
        assert lib.formgpu_batch_submit_async(h, reqs, 2) == 0
        # a second submission before the wait is refused and does not disturb the first
        other = (_capi.Request * 1)()
        other[0].sequence, other[0].op = 0, _capi.OP_COMMIT
        assert lib.formgpu_batch_submit_async(h, other, 1) == _capi.ERR_STATE
        assert lib.formgpu_batch_wait(h) == 0
        assert lib.formgpu_batch_done(h) == 1
        assert reqs[0].n_planar > 0 and reqs[1].n_planar > 0
        assert lib.formgpu_batch_wait(h) == 0  # idempotent
        # a submission that aborts in its build phase stamps every request (ADVICE r1: a pooled
        # Estimator must not mistake an unprocessed request for a completed one)
        reqs[1].op = 99
        rc = lib.formgpu_batch_submit(h, reqs, 2)
        assert rc == _capi.ERR_INVALID_ARG
        assert [reqs[s].status for s in range(2)] == [rc, rc]
        assert lib.formgpu_batch_done(h) == 1
    finally:
        lib.formgpu_batch_destroy(h)


def test_pooled_live_estimators_match_standalone_estimators():
    """Four LIVE form::Estimators (host smoother in the loop, one thread each) behind the
    batching dispatcher: identical keypoints and control flow, poses equal to 1e-7, and far
    fewer submits than requests."""
    from concurrent.futures import ThreadPoolExecutor

    from form_b200.pipeline import Estimator, EstimatorPool

    sensor, n_scans, seqs = "vlp-16", 12, (0, 4, 5, 9)
    rows, cols = synth.shape(sensor)
    p = _capi.default_est_params(rows, cols)
    scans = {s: [synth.scan(sensor, s, k) for k in range(n_scans)] for s in seqs}
    # degenerate inputs inside a batch: one sequence sees a scan of pure dropouts (no keypoints:
    # Matcher::match returns early, matcher.hpp:72-74) while the others carry on
    scans[seqs[1]][5] = np.zeros_like(scans[seqs[1]][5])
    alone = {}
    for s in seqs:
        with Estimator(p) as e:
            kps = [e.register_scan(sc) for sc in scans[s]]
            alone[s] = (kps, e.pose(), e.stats(), e.window())
    with EstimatorPool(p, len(seqs)) as pool:
        def drive(i):
            e, s = pool.estimators[i], seqs[i]
            kps = [e.register_scan(sc) for sc in scans[s]]
            return kps, e.pose(), e.stats(), e.window()

        with ThreadPoolExecutor(len(seqs)) as ex:
            pooled = list(ex.map(drive, range(len(seqs))))
        st = pool.stats()
    for i, s in enumerate(seqs):
        kps, pose, stats, window = pooled[i]
        rk, rpose, rstats, rwindow = alone[s]
        for (pl, pt), (rpl, rpt) in zip(kps, rk):
            assert pl.tobytes() == rpl.tobytes() and pt.tobytes() == rpt.tobytes()
        assert stats == rstats, (stats, rstats)          # same ICP / LM iterations, same calls
        assert np.array_equal(window["scan"], rwindow["scan"])
        assert np.max(np.abs(pose["t"] - rpose["t"])) < 1e-7 and np.max(np.abs(pose["R"] - rpose["R"])) < 1e-7
    assert st["requests"] > st["submits"] > 0            # calls of different sequences shared submits
