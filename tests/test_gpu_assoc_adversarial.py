"""Every association kernel on the adversarial windows of assoc_scenes.py: exact ties across shift
ranks, scans and keypoints, coordinates on voxel faces, distances on the gates, bucket-size edges,
far poses, a sparse map and scan ids beyond 2^40.  Per scene and per configuration every call is
compared with the oracle (matches with dist^2 bits, pair counts, novel counts, stored keypoint
bytes) and with the independent brute-force rule R5 on the checked queries.

| configuration | association kernel |
|---|---|
| warp        | assoc_nn_kernel, one warp per query (the single-context default) |
| cells       | assoc_cells_kernel (FORMGPU_SINGLE_CELL_SEARCH=1) |
| batch       | assoc_cells_batch_kernel (raw formgpu_batch_* requests) |
| mixed       | one formgpu_batch_create_mixed submission per operation for scenes of widths 0.5, 0.8, 64 |

Stage 3 on the same windows: linearisation and error against the oracle at the association poses,
at poses drifted by 0.3 rad and 1 m from them, and far from the origin, with the pair-moment cache
and with FORMGPU_STREAM_LINEARIZE=1 (metric: _block_err)."""
import ctypes as C

import numpy as np
import pytest

import assoc_scenes as A
from form_b200 import _capi
from form_b200.context import Context
from helpers import scan_poses, unpack91

pytestmark = pytest.mark.gpu

SCENES = {s.name: s for s in A.all_scenes()}

CONFIGS = {
    "warp": {},
    "cells": {"FORMGPU_SINGLE_CELL_SEARCH": "1"},
    "batch": {},
}
ENV = ("FORMGPU_SINGLE_CELL_SEARCH", "FORMGPU_STREAM_LINEARIZE")


def _env(monkeypatch, cfg):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in cfg.items():
        monkeypatch.setenv(k, v)


class _Borrowed(Context):
    """The Context methods over a context owned by a batch (formgpu_batch_ctx): never destroyed here."""

    def __init__(self, handle, params):
        self._lib = _capi.gpu_lib()
        self._h = C.c_void_p(handle)
        self.params = params
        self.rows, self.cols = params.num_rows, params.num_columns
        self.max_planar = self._lib.formgpu_max_planar(self._h)
        self.max_point = self._lib.formgpu_max_point(self._h)

    def close(self):
        self._h = None


class Batch:
    """Raw formgpu_batch_* requests: every call of run_lockstep is one submission holding the next
    operation of every scene; matches and keypoints are read from the sequence's own context."""

    def __init__(self, params_list):
        self.lib = _capi.gpu_lib()
        self.params = (_capi.Params * len(params_list))(*params_list)
        self.h = C.c_void_p()
        assert self.lib.formgpu_batch_create_mixed(self.params, 0, None, len(params_list), C.byref(self.h)) == 0
        self.ctx = [_Borrowed(self.lib.formgpu_batch_ctx(self.h, i), params_list[i]) for i in range(len(params_list))]

    def close(self):
        for c in self.ctx:
            c.close()
        self.lib.formgpu_batch_destroy(self.h)

    def do_many(self, todo):
        reqs = (_capi.Request * len(todo))()
        keep = []
        for r, (i, op) in zip(reqs, todo):
            r.sequence = i
            c = self.ctx[i]
            if op[0] == "extract":
                pl, pt = np.zeros(c.max_planar, _capi.PLANAR_FEAT), np.zeros(c.max_point, _capi.POINT_FEAT)
                scan = np.ascontiguousarray(op[2])
                keep += [pl, pt, scan]
                r.op, r.scan, r.n_points, r.scan_idx = _capi.OP_EXTRACT, scan.ctypes.data, len(scan), op[1]
                r.planar_out, r.planar_cap, r.point_out, r.point_cap = pl.ctypes.data, len(pl), pt.ctypes.data, len(pt)
            elif op[0] == "rebuild":
                sp = scan_poses(list(op[1]), list(op[1].values()))
                keep.append(sp)
                r.op, r.poses, r.n_poses = _capi.OP_MAP_REBUILD, sp.ctypes.data, len(sp)
            elif op[0] == "associate":
                pk = np.ascontiguousarray(op[1])
                counts = np.zeros(c.params.max_window_scans, _capi.PAIR_COUNT)
                keep += [pk, counts]
                r.op, r.pose_k, r.counts_out, r.counts_cap = _capi.OP_ASSOCIATE, pk.ctypes.data, counts.ctypes.data, len(counts)
            elif op[0] == "commit":
                keep.append(None)
                r.op = _capi.OP_COMMIT
        rc = self.lib.formgpu_batch_submit(self.h, reqs, len(todo))
        assert rc == 0, (rc, self.lib.formgpu_batch_last_error(self.h))
        out, n = [], 0
        for r, (i, op) in zip(reqs, todo):
            assert r.status == 0
            c = self.ctx[i]
            if op[0] == "extract":
                pl, pt = keep[n], keep[n + 1]
                n += 3
                out.append((pl[: r.n_planar].copy(), pt[: r.n_point].copy()))
            elif op[0] == "rebuild":
                n += 1
                out.append(None)
            elif op[0] == "associate":
                counts = keep[n + 1]
                n += 2
                out.append((counts[: r.n_counts].copy(), c.matches(0), c.matches(1)))
            else:
                n += 1
                out.append(((r.n_planar, r.n_point), c.keypoints(0, op[1]), c.keypoints(1, op[1])))
        return out


def _check(scene, recs, label):
    """The records of a run against the oracle's and against the brute-force rule R5."""
    want, exp = A.oracle_run(scene)
    assert len(recs) == len(want)
    n_assoc = 0
    for n, (op, got, ref) in enumerate(zip(scene.ops, recs, want)):
        where = f"{label} {scene.name} op {n} ({op[0]})"
        if op[0] == "extract":
            assert got[0].tobytes() == ref[0].tobytes() and got[1].tobytes() == ref[1].tobytes(), where
        elif op[0] == "associate":
            e = exp[n_assoc]
            n_assoc += 1
            for t in (0, 1):
                m, rm = got[1 + t], ref[1 + t]
                assert len(m) == len(rm), where
                for f in ("found", "scan", "k"):
                    assert np.array_equal(m[f], rm[f]), (where, t, f, np.nonzero(m[f] != rm[f])[0][:8])
                assert np.array_equal(m["dist_sqrd"].view(np.uint64), rm["dist_sqrd"].view(np.uint64)), (where, t)
                ty = e["types"][t]
                bf, sel = ty["bf"], m[ty["idx"]]
                assert np.array_equal(sel["found"].astype(bool), bf["found"]), (where, t, "brute force")
                assert np.array_equal(sel["scan"], bf["scan"]) and np.array_equal(sel["k"], bf["k"]), (where, t)
                assert np.array_equal(sel["dist_sqrd"].view(np.uint64), bf["dist_sqrd"].view(np.uint64)), (where, t)
            assert got[0].tobytes() == ref[0].tobytes(), (where, "pair counts", got[0], ref[0])
        elif op[0] == "commit":
            assert tuple(got[0]) == tuple(ref[0]), (where, "novel keypoints", got[0], ref[0])
            assert got[1].tobytes() == ref[1].tobytes() and got[2].tobytes() == ref[2].tobytes(), where


@pytest.mark.parametrize("config", sorted(CONFIGS))
@pytest.mark.parametrize("name", sorted(SCENES))
def test_association_matches_oracle_and_brute_force(name, config, monkeypatch):
    _env(monkeypatch, CONFIGS[config])
    scene = SCENES[name]
    if config in ("warp", "cells"):
        with Context(scene.make_params()) as ctx:
            recs = A.run(scene, ctx)
    else:
        b = Batch([scene.make_params()])
        try:
            recs = A.run_lockstep([scene], b.do_many)[0]
        finally:
            b.close()
    _check(scene, recs, config)


@pytest.mark.parametrize("group", [("lattice_w0.5", "face_aligned", "huge_bucket", "large_ids"),
                                   ("gates", "synthetic_far", "sparse", "buckets_19", "far_w1.0")])
@pytest.mark.parametrize("config", ["batch"])
def test_one_mixed_launch(group, config, monkeypatch):
    """Scenes of different widths (0.5, 0.8, 64; 1.0, 0.8, 0.5) and sensor shapes in one
    formgpu_batch_create_mixed batch: every submission carries one operation of each, so one
    association launch searches maps of different widths."""
    _env(monkeypatch, CONFIGS[config])
    scenes = [SCENES[n] for n in group]
    b = Batch([s.make_params() for s in scenes])
    try:
        recs = A.run_lockstep(scenes, b.do_many)
    finally:
        b.close()
    for s, r in zip(scenes, recs):
        _check(s, r, f"mixed/{config}")


def _drifted(p, rng, rot, trans):
    """p moved by a rotation of exactly `rot` rad about a random axis and a translation of `trans` m."""
    ax = rng.normal(size=3)
    ax /= np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    dR = np.eye(3) + np.sin(rot) * K + (1 - np.cos(rot)) * K @ K
    d = rng.normal(size=3)
    return A.pose(p["R"].reshape(3, 3) @ dR, p["t"] + trans * d / np.linalg.norm(d))


H_TOL = 1e-9
UNIT = 2.0 ** -53


def _block_err(a91, b91, tol=H_TOL):
    """block_rel_err with a floor for directions a pair barely constrains.  Every Jacobian entry
    is computed through rotation matrices that are orthonormal only to about one unit roundoff u,
    so entry (a, b) of the block is determined only to about u * sqrt(G_max) * (|J_a| + |J_b|)
    (|J_a| = sqrt(G_aa)); the scale of an entry is therefore never taken below that floor divided
    by the tolerance.  For well-constrained rows sqrt(G_aa G_bb) is far above the floor and this is
    block_rel_err exactly; for a direction with G_aa ~ 0 (planes seen along one axis only) the
    entries are compared against the roundoff their inputs carry instead of against zero.
    Recomputed in exact rational arithmetic, such entries differ from the exact value by less than
    u * sqrt(G_max) * (|J_a| + |J_b|) on both the kernels' and the oracle's side."""
    A, B = unpack91(a91), unpack91(b91)
    s = np.sqrt(np.maximum(np.diag(B), 0.0))
    floor = (UNIT / tol) * s.max() * (s[:, None] + s[None, :])
    scale = np.maximum(np.outer(s, s), floor)
    scale[scale == 0] = 1.0
    return float(np.max(np.abs(A - B) / scale))


@pytest.mark.parametrize("stream", [False, True], ids=["moments", "stream"])
@pytest.mark.parametrize("name", ["lattice_w0.5", "duplicates", "gates", "face_aligned", "far_w0.5", "far_w1.0",
                                  "synthetic_far", "sparse"])
def test_stage3_on_adversarial_windows(name, stream, monkeypatch):
    """linearize / error of every pair of the current scan after each association, against the oracle
    in the same state: at the association poses, at poses drifted by 0.3 rad and 1 m, and (far
    scenes) thousands of metres from the origin."""
    import oracle_lib

    _env(monkeypatch, {"FORMGPU_STREAM_LINEARIZE": "1"} if stream else {})
    scene = SCENES[name]
    rng = np.random.default_rng(3)
    ref = oracle_lib.Oracle(scene.make_params())
    try:
        worst, n_pairs = 0.0, 0
        with Context(scene.make_params()) as ctx:
            rebuild, cur = {}, None
            for op in scene.ops:
                got, want = A.do(ctx, op), A.do(ref, op)
                if op[0] == "extract":
                    cur = op[1]
                elif op[0] == "rebuild":
                    rebuild = dict(op[1])
                elif op[0] == "associate" and len(want[0]):
                    assert got[0].tobytes() == want[0].tobytes()
                    at = {**rebuild, cur: op[1]}
                    pairs = np.zeros(len(want[0]), _capi.PAIR)
                    pairs["i"], pairs["j"] = want[0]["i"], cur
                    for poses in (at, {s: _drifted(p, rng, 0.3, 1.0) for s, p in at.items()},
                                  {s: _drifted(p, rng, 0.05, 0.2) for s, p in at.items()}):
                        sp = scan_poses(list(poses), list(poses.values()))
                        H, Hr = ctx.linearize(pairs, sp), ref.linearize(pairs, sp)
                        for a, b in zip(H, Hr):
                            worst = max(worst, _block_err(a, b))
                        e, er = ctx.error(pairs, sp), ref.error(pairs, sp)
                        assert np.allclose(e, er, rtol=1e-9, atol=1e-12), (name, e, er)
                        n_pairs += len(pairs)
    finally:
        ref.close()
    assert n_pairs > 0
    assert worst < H_TOL, (name, worst)
