"""Every stage-1 kernel configuration on the adversarial scans of extract_scenes.py: range gates and
the w lane, neighbour radius equalities, curvature ties and threshold equalities, closest-point
ties and the pruning margin, degenerate covariances and FLT_MIN in the eigen solver, sector,
capacity and shape edges.  Per scene and configuration the result is compared with the oracle
and, for the pick positions, with the numpy restatement, so that a wrong oracle cannot hide a
wrong kernel.

| configuration | kernels |
|---|---|
| single    | extract_select_kernel (512 threads), extract_normals_kernel (warp per pick, closest_in_row_pruned), extract_pack_kernel: masks, curvature bits, picks, keep flags, closest prev / next and keypoint bytes |
| few       | extract_select_batch_kernel at 512 threads, extract_normals_batch_kernel (FORMGPU_MANY_ROWS_MIN=1000000) |
| many      | select at 192 threads, extract_normals_rows_kernel (thread per pick, closest_in_row_thread, neighbor_counts_thread) |
| select32 / select64 | many-row select with one or two warps per CTA, so one warp walks many sectors (FORMGPU_SELECT_THREADS, read once per process: run in a child process) |
| mixed     | one formgpu_batch_create_mixed submission holding scenes of different shapes and parameters |

Batched configurations compare per-request counts and keypoint bytes."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__":  # the child process of test_narrow_select_ctas
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402
import pytest  # noqa: E402

import extract_scenes as E  # noqa: E402
from form_b200.context import Context  # noqa: E402
from test_gpu_assoc_adversarial import Batch  # noqa: E402

pytestmark = pytest.mark.gpu

SCENES = {s.name: s for s in E.all_scenes()}
SCAN_IDX = 7
MANY_ROWS = {"few": "1000000", "many": "1"}


def _oracle(scene):
    import oracle_lib

    o = oracle_lib.Oracle(scene.params)
    try:
        pl, pt = o.extract(scene.scan, SCAN_IDX)
        return pl, pt, o.extract_debug()
    finally:
        o.close()


def _check_keypoints(scene, pl, pt, label):
    """Keypoint bytes against the oracle, keypoint positions against the numpy restatement."""
    rpl, rpt, _ = _oracle(scene)
    assert (len(pl), len(pt)) == (len(rpl), len(rpt)), (label, "counts", len(pl), len(pt), len(rpl), len(rpt))
    assert pl.tobytes() == rpl.tobytes(), (label, "planar keypoints (normals included)")
    assert pt.tobytes() == rpt.tobytes(), (label, "point keypoints")
    R = E.restate(scene)
    s4 = R["s4"].astype(np.float64)
    kept = R["picks"][R["keep"]]
    got = np.stack([pl["x"], pl["y"], pl["z"]], axis=1)
    assert np.array_equal(got, s4[kept, :3]), (label, "planar pick positions vs restatement")
    got = np.stack([pt["x"], pt["y"], pt["z"]], axis=1)
    assert np.array_equal(got, s4[R["qpicks"], :3]), (label, "point pick positions vs restatement")


def _batch_extract(scenes):
    b = Batch([s.params for s in scenes])
    try:
        return b.do_many([(i, ("extract", SCAN_IDX, s.scan)) for i, s in enumerate(scenes)])
    finally:
        b.close()


@pytest.mark.parametrize("name", sorted(SCENES))
def test_single_context_matches_oracle(name):
    scene = SCENES[name]
    _, _, rd = _oracle(scene)
    with Context(scene.params) as ctx:
        pl, pt = ctx.extract(scene.scan, SCAN_IDX)
        d = ctx.extract_debug()
    for k in ("valid", "point_valid"):
        assert np.array_equal(d[k], rd[k]), k
    assert np.array_equal(d["curvature"].view(np.uint32), rd["curvature"].view(np.uint32)), "curvature bits"
    for k in ("planar_indices", "planar_keep", "closest_prev", "closest_next", "point_indices"):
        assert np.array_equal(d[k], rd[k]), (k, np.nonzero(d[k] != rd[k])[0][:8] if len(d[k]) == len(rd[k]) else
                                             (len(d[k]), len(rd[k])))
    R = E.restate(scene)
    assert np.array_equal(d["planar_indices"], R["picks"]) and np.array_equal(d["point_indices"], R["qpicks"])
    assert np.array_equal(d["closest_prev"], R["cprev"]) and np.array_equal(d["closest_next"], R["cnext"])
    _check_keypoints(scene, pl, pt, "single")


@pytest.mark.parametrize("config", sorted(MANY_ROWS))
@pytest.mark.parametrize("name", sorted(SCENES))
def test_batched_matches_oracle(name, config, monkeypatch):
    monkeypatch.setenv("FORMGPU_MANY_ROWS_MIN", MANY_ROWS[config])  # read by formgpu_batch_create
    scene = SCENES[name]
    (pl, pt), = _batch_extract([scene])
    _check_keypoints(scene, pl, pt, config)


MIXED = [("range_gates", "radius_np16", "shape_3x4096", "m20_flt_min", "sectors_pps1_max", "shape_1x33_np5"),
         ("closest_ties", "shape_2x3_np1", "unused_lengths_pfps1", "cov_zero", "far_ulps", "planar_cap_zero")]


@pytest.mark.parametrize("config", sorted(MANY_ROWS))
@pytest.mark.parametrize("group", range(len(MIXED)))
def test_one_mixed_launch(group, config, monkeypatch):
    """Scenes of different shapes (1..3 rows, 3..4096 columns) and parameters (np 1..16, 1..64
    sectors) in one submission: CTAs past a smaller item's rows leave at once."""
    monkeypatch.setenv("FORMGPU_MANY_ROWS_MIN", MANY_ROWS[config])
    scenes = [SCENES[n] for n in MIXED[group]]
    for s, (pl, pt) in zip(scenes, _batch_extract(scenes)):
        _check_keypoints(s, pl, pt, f"mixed/{config} {s.name}")


def _child(threads):
    """Every scene through the many-row kernels with `threads` select threads (run as a process of
    its own: the select width is read once per process)."""
    assert os.environ.get("FORMGPU_SELECT_THREADS") == str(threads)
    for s in SCENES.values():
        (pl, pt), = _batch_extract([s])
        _check_keypoints(s, pl, pt, f"select{threads} {s.name}")


@pytest.mark.parametrize("threads", [32, 64])
def test_narrow_select_ctas(threads):
    env = dict(os.environ, FORMGPU_SELECT_THREADS=str(threads), FORMGPU_MANY_ROWS_MIN="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(threads)], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]


if __name__ == "__main__":
    _child(int(sys.argv[1]))
