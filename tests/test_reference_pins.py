"""Pins the oracle to the REFERENCE'S OWN CODE, all three stages of the hot path.

oracle/_ref/libformref.so is FORM's form/feature/extraction.tpp, features.hpp, utils.hpp,
form/mapping/map.tpp, form/optimization/matcher.hpp, form/feature/factor.{hpp,cpp} and
form/optimization/gtsam.hpp compiled UNMODIFIED from /root/reference (oracle/ref/Makefile)
against API stand-ins for the libraries this image lacks (oracle/shim: Eigen, GTSAM
Pose3/Values/noise-model/factor base classes, oneTBB, tsl::robin_map).  Every decision
FORM's own code takes - masks, dilation, thresholds, std::sort + greedy planar selection,
the extract_point stride/break quirks, neighbour gathering, the dropped-normal rule, voxel
keys, the strict-< bucket scans, the max_dist / min_dist_map gates, the world->local round
trip - is therefore exercised as the reference wrote it, and must agree with the oracle
restatement BIT FOR BIT (keypoints, match distances, pair counts, novel sets).  Stage 3 runs
the reference's PlanePoint / PointPoint::evaluateError, FeatureFactor::evaluateError,
FastIsotropic whitening and DenseFactor::linearize; residuals, Jacobians and the 13x13
augmented information blocks must agree with the restatement to 1e-12 (tolerance class:
the restatement reduces 7x7 moments instead of forming A^T A, so the bits differ).

Only Eigen's/GTSAM's internal arithmetic order is still a stated rule (SURVEY A.2), shared
by shim and oracle.  The library is prebuilt in this container (the reference tree does
not exist on the GPU box); these tests run wherever the library is present.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib
from form_b200 import _capi, synth
from helpers import block_rel_err, perturbed, scan_poses

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# FORM_REF_LIB: another build of the same sources (sanitizer runs)
REF_LIB = os.environ.get("FORM_REF_LIB") or os.path.join(ROOT, "oracle", "_ref", "libformref.so")

_vp, _sz, _u64, _i, _d = C.c_void_p, C.c_size_t, C.c_uint64, C.c_int, C.c_double
_psz = C.POINTER(C.c_size_t)
_SYMS = {
    "formref_extract": (_i, [C.POINTER(_capi.Params), _vp, _sz, _u64, _vp, _sz, _psz, _vp, _sz, _psz]),
    "formref_world_create": (_vp, [C.POINTER(_capi.Params)]),
    "formref_world_destroy": (None, [_vp]),
    "formref_compute_coords": (None, [_d, _d, _d, _d, _vp]),
    "formref_world_associate": (_i, [_vp, _vp, _sz, _u64, _vp, _sz, _vp, _sz] + [_vp] * 8),
    "formref_world_constraint_counts": (None, [_vp, _u64, _psz, _psz]),
    "formref_world_commit": (None, [_vp]),
    "formref_world_remove": (None, [_vp, _u64]),
    "formref_world_keypoints": (_sz, [_vp, _i, _u64, _vp, _sz]),
    "formref_world_linearize": (_i, [_vp, _u64, _u64, _vp, _vp, _d, _vp]),
    "formref_plane_point": (None, [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "formref_point_point": (None, [_vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "formref_linearize_raw": (_i, [_vp, _vp, _vp, _sz, _vp, _vp, _sz, _vp, _vp, _d, _vp]),
}
_ref = None


def ref():
    global _ref
    if _ref is None:
        if not os.path.exists(REF_LIB):
            import subprocess

            subprocess.call(["make", "-s", "-C", os.path.join(ROOT, "oracle", "ref")])
        if not os.path.exists(REF_LIB):
            pytest.skip("oracle/_ref/libformref.so is not built: it needs FORM's own sources (oracle/ref/Makefile, "
                        "REFERENCE=<FORM checkout>)")
        _ref = C.CDLL(REF_LIB)
        for name, (res, args) in _SYMS.items():
            fn = getattr(_ref, name)
            fn.restype, fn.argtypes = res, args
    return _ref


def ref_extract(params, scan, scan_idx):
    n = scan.shape[0]
    pl = np.zeros(n, dtype=_capi.PLANAR_FEAT)
    pt = np.zeros(n, dtype=_capi.POINT_FEAT)
    a, b = C.c_size_t(), C.c_size_t()
    rc = ref().formref_extract(C.byref(params), _capi.ptr(scan), n, scan_idx, _capi.ptr(pl), n, C.byref(a),
                               _capi.ptr(pt), n, C.byref(b))
    return rc, pl[: a.value].copy(), pt[: b.value].copy()


def random_scan(rng, rows, cols, dropout=0.03, near=0.02, far=0.01):
    """Organised scan of a wavy surface with dropouts, too-near and too-far returns; float
    noise makes exact curvature ties (where std::sort's order is unspecified) impossible."""
    az = np.tile(np.linspace(0, 2 * np.pi, cols, endpoint=False), rows)
    el = np.repeat(np.linspace(-0.35, 0.35, rows), cols)
    r = 7.0 + 1.5 * np.sin(3 * az + 0.3) + 0.8 * np.cos(7 * az) * np.cos(3 * el) + 0.02 * rng.standard_normal(rows * cols)
    u = rng.random(rows * cols)
    r = np.where(u < near, 0.5, r)
    r = np.where((u >= near) & (u < near + far), 150.0, r)
    scan = np.zeros(rows * cols, dtype=_capi.POINT4F)
    scan["x"] = (r * np.cos(el) * np.cos(az)).astype(np.float32)
    scan["y"] = (r * np.cos(el) * np.sin(az)).astype(np.float32)
    scan["z"] = (r * np.sin(el)).astype(np.float32)
    drop = rng.random(rows * cols) < dropout
    for f in ("x", "y", "z"):
        scan[f][drop] = 0.0
    return scan


def assert_same_features(params, scan, scan_idx):
    rc, rpl, rpt = ref_extract(params, scan, scan_idx)
    assert rc == 0
    o = oracle_lib.Oracle(params, threads=2)
    pl, pt = o.extract(scan, scan_idx)
    assert len(pl) == len(rpl) and len(pt) == len(rpt), (len(pl), len(rpl), len(pt), len(rpt))
    assert pt.tobytes() == rpt.tobytes(), "point keypoints differ from the reference"
    # positions, scan ids and order (rule R3 = planar_indices order) are exact
    for f in ("x", "y", "z", "pad", "npad", "scan"):
        assert np.array_equal(pl[f], rpl[f]), f
    # normals: the reference's neighbour gathering feeds the restated Eigen solver
    assert pl.tobytes() == rpl.tobytes(), "planar normals differ from the reference"
    return len(pl), len(pt)


@pytest.mark.parametrize("sensor,k", [("vlp-16", 0), ("vlp-16", 7), ("os1-64", 3)])
def test_extraction_matches_reference_on_synthetic_sensor_scans(sensor, k):
    rows, cols = synth.shape(sensor)
    params = _capi.default_params(rows, cols)
    n_pl, n_pt = assert_same_features(params, synth.scan(sensor, 0, k), k)
    assert n_pl > 100 and n_pt > 10


@pytest.mark.parametrize("overrides", [
    {},
    {"point_feats_per_sector": 0},
    {"neighbor_points": 3, "num_sectors": 5},          # sector remainder: 384 = 5 * 76 + 4
    {"planar_threshold": 0.05, "planar_feats_per_sector": 4},
    {"min_points": 20},                                # most normals dropped
    {"radius": 0.3, "min_norm_squared": 0.04},         # dropout zeros can become neighbours (A.3-7)
    {"point_feats_per_sector": 1},
])
def test_extraction_matches_reference_on_random_scans(overrides):
    rows, cols = 8, 384
    params = _capi.default_params(rows, cols, **overrides)
    rng = np.random.default_rng(17)
    total = 0
    for trial in range(4):
        n_pl, n_pt = assert_same_features(params, random_scan(rng, rows, cols), trial)
        total += n_pl + n_pt
    assert total > 0


def test_reference_rejects_wrong_scan_size_like_the_c_abi():
    params = _capi.default_params(8, 384)
    rc, _, _ = ref_extract(params, np.zeros(100, dtype=_capi.POINT4F), 0)
    assert rc == 2  # the reference throws (extraction.tpp:141-145) = FORMGPU_ERR_BAD_SCAN_SIZE


@pytest.mark.parametrize("p,w", [
    ((0.0, 0.0, 0.0), 0.8), ((-0.0, 0.79999, 0.8), 0.8), ((-1e-12, -0.8, -0.80000001), 0.8),
    ((1.6, 2.4000000000000004, 2.3999999999999995), 0.8), ((-37.123, 12.0, 99.99), 0.8),
    ((0.1, 0.2, 0.30000000000000004), 0.1),
])
def test_voxel_keys_match_reference(p, w):
    a, b = np.zeros(3, np.int32), np.zeros(3, np.int32)
    ref().formref_compute_coords(p[0], p[1], p[2], w, _capi.ptr(a))
    oracle_lib.lib().oracle_compute_coords(p[0], p[1], p[2], w, _capi.ptr(b))
    assert tuple(a) == tuple(b)


def test_voxel_keys_match_reference_at_faces():
    rng = np.random.default_rng(5)
    w = 0.8
    vals = [k * w for k in range(-40, 40)]
    vals = vals + [np.nextafter(v, np.inf) for v in vals] + [np.nextafter(v, -np.inf) for v in vals]
    vals = vals + list(rng.uniform(-50, 50, 200))
    for v in vals:
        a, b = np.zeros(3, np.int32), np.zeros(3, np.int32)
        ref().formref_compute_coords(v, -v, 0.5 * v, w, _capi.ptr(a))
        oracle_lib.lib().oracle_compute_coords(v, -v, 0.5 * v, w, _capi.ptr(b))
        assert tuple(a) == tuple(b), v


def _ref_associate(world, sp, cur_scan, pl, pt):
    out = [np.zeros(len(pl), _capi.PLANAR_FEAT), np.zeros(len(pl), _capi.PLANAR_FEAT), np.zeros(len(pl)),
           np.zeros(len(pl), np.uint8), np.zeros(len(pt), _capi.POINT_FEAT), np.zeros(len(pt), _capi.POINT_FEAT),
           np.zeros(len(pt)), np.zeros(len(pt), np.uint8)]
    rc = ref().formref_world_associate(world, _capi.ptr(sp), sp.shape[0], cur_scan, _capi.ptr(pl), len(pl),
                                       _capi.ptr(pt), len(pt), *[_capi.ptr(o) for o in out])
    assert rc == 0
    return out


@pytest.mark.parametrize("sensor,n_scans", [("vlp-16", 5), (None, 4)])
def test_association_commit_and_removal_match_reference(sensor, n_scans):
    """Matcher::match<0/1>, to_voxel_map, insert_matches and remove over a short sequence:
    per keypoint the matched scan, the bit pattern of dist^2 and the matched point; per pair
    the correspondence counts; per scan the stored keypoints."""
    rng = np.random.default_rng(11)
    if sensor:
        rows, cols = synth.shape(sensor)
        scans = [synth.scan(sensor, 0, k) for k in range(n_scans)]
        gt = [synth.gt_pose(0, k) for k in range(n_scans)]
    else:
        rows, cols = 8, 384
        scans = [random_scan(rng, rows, cols) for _ in range(n_scans)]
        ident = np.zeros((), dtype=_capi.POSE)
        ident["R"] = np.eye(3).reshape(9)
        gt = [ident] + [perturbed(ident, rng, 0.01, 0.05) for _ in range(n_scans - 1)]
    params = _capi.default_params(rows, cols)
    o = oracle_lib.Oracle(params, threads=2)
    world = ref().formref_world_create(C.byref(params))
    try:
        poses = {}
        for k, scan in enumerate(scans):
            pl, pt = o.extract(scan, k)
            poses[k] = gt[k] if k == 0 else perturbed(gt[k], rng, 0.002, 0.02)
            sp = scan_poses(list(poses), [poses[s] for s in poses])
            o.map_rebuild(sp)
            counts = o.associate(poses[k])
            r = _ref_associate(world, sp, k, pl, pt)
            for t, feats, (rq, rp, rd, rf) in ((0, pl, r[0:4]), (1, pt, r[4:8])):
                m = o.matches(t)
                assert len(m) == len(feats)
                assert rq.tobytes() == feats.tobytes()                      # match.query = *kp
                assert np.array_equal(rf, m["found"].astype(np.uint8))
                assert rd.tobytes() == m["dist_sqrd"].tobytes()             # dist^2 bit patterns
                found = m["found"] == 1
                assert np.array_equal(rp["scan"][found], m["scan"][found])  # matched scan
                # matched point: the reference hands back T_i^-1 (T_i p), the oracle names (scan, k)
                for s in np.unique(m["scan"][found]):
                    stored = o.keypoints(t, int(s))
                    sel = found & (m["scan"] == s)
                    for f in ("x", "y", "z"):
                        assert np.allclose(rp[f][sel], stored[f][m["k"][sel]], rtol=0, atol=1e-9)
            # correspondences appended per map scan (dist^2 < max_dist^2, matcher.hpp:103-111)
            by_scan = {int(c["i"]): (int(c["n_planar"]), int(c["n_point"])) for c in counts}
            for s in range(k):
                a, b = C.c_size_t(), C.c_size_t()
                ref().formref_world_constraint_counts(world, s, C.byref(a), C.byref(b))
                assert (a.value, b.value) == by_scan.get(s, (0, 0)), (k, s)
            o.commit_scan()
            ref().formref_world_commit(world)
            for t in (0, 1):
                stored = o.keypoints(t, k)
                buf = np.zeros(len(stored) + 8, dtype=stored.dtype)
                n = ref().formref_world_keypoints(world, t, k, _capi.ptr(buf), len(buf))
                assert n == len(stored)
                assert buf[:n].tobytes() == stored.tobytes()                # novel-keypoint sets
            if k == 2:  # marginalise scan 1 (form.cpp:111)
                o.remove_scans([1])
                ref().formref_world_remove(world, 1)
                del poses[1]
        assert sum(len(o.keypoints(0, k)) for k in poses) > 0
    finally:
        ref().formref_world_destroy(world)


# ------------------------------------------------------------------ stage 3
def _random_pose(rng, rot=0.6, trans=3.0):
    ident = np.zeros((), dtype=_capi.POSE)
    ident["R"] = np.eye(3).reshape(9)
    return perturbed(ident, rng, rot, trans)


def _random_correspondences(rng, n, m):
    p_i, p_j = rng.normal(size=(n, 3)) * 6, rng.normal(size=(n, 3)) * 6
    n_i = rng.normal(size=(n, 3))
    n_i /= np.linalg.norm(n_i, axis=1, keepdims=True)
    q_i, q_j = rng.normal(size=(m, 3)) * 6, rng.normal(size=(m, 3)) * 6
    return p_i, n_i, p_j, q_i, q_j


@pytest.mark.parametrize("n", [1, 7, 300])
def test_plane_point_and_point_point_match_reference(n):
    """PlanePoint / PointPoint::evaluateError (factor.cpp:30-128): residuals and both Jacobians."""
    rng = np.random.default_rng(100 + n)
    p_i, n_i, p_j, q_i, q_j = _random_correspondences(rng, n, n)
    Ti, Tj = _random_pose(rng), _random_pose(rng)
    a, b = np.array([Ti], dtype=_capi.POSE), np.array([Tj], dtype=_capi.POSE)
    r, H1, H2 = np.zeros(n), np.zeros((n, 6)), np.zeros((n, 6))
    ref().formref_plane_point(_capi.ptr(p_i), _capi.ptr(n_i), _capi.ptr(p_j), n, _capi.ptr(a), _capi.ptr(b),
                              _capi.ptr(r), _capi.ptr(H1), _capi.ptr(H2))
    o_r, o_H1, o_H2 = np.zeros(n), np.zeros((n, 6)), np.zeros((n, 6))
    oracle_lib.lib().oracle_plane_point(_capi.ptr(p_i), _capi.ptr(n_i), _capi.ptr(p_j), n, _capi.ptr(a),
                                        _capi.ptr(b), _capi.ptr(o_r), _capi.ptr(o_H1), _capi.ptr(o_H2))
    scale = 1.0 + np.abs(H1).max()
    assert np.abs(r - o_r).max() < 1e-12 * scale
    assert np.abs(H1 - o_H1).max() < 1e-12 * scale and np.abs(H2 - o_H2).max() < 1e-12 * scale
    assert np.abs(H1).max() > 0.1
    r, H1, H2 = np.zeros(3 * n), np.zeros((3 * n, 6)), np.zeros((3 * n, 6))
    ref().formref_point_point(_capi.ptr(q_i), _capi.ptr(q_j), n, _capi.ptr(a), _capi.ptr(b), _capi.ptr(r),
                              _capi.ptr(H1), _capi.ptr(H2))
    o_r, o_H1, o_H2 = np.zeros(3 * n), np.zeros((3 * n, 6)), np.zeros((3 * n, 6))
    oracle_lib.lib().oracle_point_point(_capi.ptr(q_i), _capi.ptr(q_j), n, _capi.ptr(a), _capi.ptr(b),
                                        _capi.ptr(o_r), _capi.ptr(o_H1), _capi.ptr(o_H2))
    scale = 1.0 + np.abs(H1).max()
    assert np.abs(r - o_r).max() < 1e-12 * scale
    assert np.abs(H1 - o_H1).max() < 1e-12 * scale and np.abs(H2 - o_H2).max() < 1e-12 * scale


@pytest.mark.parametrize("n,m", [(1, 0), (0, 1), (40, 9), (1001, 333)])
def test_dense_factor_linearize_matches_reference(n, m):
    """FeatureFactor + FastIsotropic + DenseFactor::linearize (factor.cpp:131-186,
    gtsam.hpp:67-140) vs the restatement's 91-double block."""
    rng = np.random.default_rng(7 * n + m)
    p_i, n_i, p_j, q_i, q_j = _random_correspondences(rng, n, m)
    Ti, Tj = _random_pose(rng), _random_pose(rng)
    a, b = np.array([Ti], dtype=_capi.POSE), np.array([Tj], dtype=_capi.POSE)
    got, want = np.zeros(91), np.zeros(91)
    rc = ref().formref_linearize_raw(_capi.ptr(p_i), _capi.ptr(n_i), _capi.ptr(p_j), n, _capi.ptr(q_i),
                                     _capi.ptr(q_j), m, _capi.ptr(a), _capi.ptr(b), 0.1, _capi.ptr(got))
    assert rc == 0
    oracle_lib.lib().oracle_linearize_raw(_capi.ptr(p_i), _capi.ptr(n_i), _capi.ptr(p_j), n, _capi.ptr(q_i),
                                          _capi.ptr(q_j), m, _capi.ptr(a), _capi.ptr(b), 0.1, _capi.ptr(want), None)
    assert np.abs(got).sum() > 0
    assert block_rel_err(got, want) < 1e-12


def test_whole_path_blocks_match_reference():
    """Stages 1 -> 2 -> 3 end to end: the reference's own matcher builds the correspondences
    of every pair (incl. its world->local round trip of the map point) and its own
    DenseFactor::linearize forms the block; the restatement must agree to 1e-9."""
    rng = np.random.default_rng(31)
    sensor, n_scans = "vlp-16", 4
    rows, cols = synth.shape(sensor)
    params = _capi.default_params(rows, cols)
    o = oracle_lib.Oracle(params, threads=2)
    world = ref().formref_world_create(C.byref(params))
    checked = 0
    try:
        poses = {}
        for k in range(n_scans):
            pl, pt = o.extract(synth.scan(sensor, 0, k), k)
            gt = synth.gt_pose(0, k)
            poses[k] = gt if k == 0 else perturbed(gt, rng, 0.002, 0.02)
            sp = scan_poses(list(poses), [poses[s] for s in poses])
            o.map_rebuild(sp)
            counts = o.associate(poses[k])
            _ref_associate(world, sp, k, pl, pt)
            if len(counts):
                pairs = np.zeros(len(counts), dtype=_capi.PAIR)
                pairs["i"] = counts["i"]
                pairs["j"] = k
                H = o.linearize(pairs, sp)
                for c, h in zip(counts, H):
                    got = np.zeros(91)
                    a = np.array([poses[int(c["i"])]], dtype=_capi.POSE)
                    b = np.array([poses[k]], dtype=_capi.POSE)
                    rc = ref().formref_world_linearize(world, int(c["i"]), k, _capi.ptr(a), _capi.ptr(b), params.sigma,
                                                       _capi.ptr(got))
                    assert rc == 0
                    assert block_rel_err(got, h) < 1e-9, (k, int(c["i"]))
                    checked += 1
            o.commit_scan()
            ref().formref_world_commit(world)
    finally:
        ref().formref_world_destroy(world)
    assert checked >= 3
