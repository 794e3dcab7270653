"""Adversarial windows for stage 2 (map rebuild, nearest-neighbour association, commit) and an
independent restatement of rule R5.  TEST INFRASTRUCTURE, not collected by pytest.

The synthetic LiDAR scenes of the other tests are smooth surfaces near the origin: they almost never
put two candidates at exactly the same squared distance, a coordinate on a voxel face, a distance on
a gate, or a bucket on a size edge of the kernels' data layout.  The scenes here do that on purpose:

* rooms whose every point lies on a dyadic lattice (step w / 4), seen from lattice poses with exact
  90-degree rotations, so keypoints, stored points and queries are lattice points and squared
  distances tie exactly across shift ranks, scans and keypoint indices;
* windows whose stored scans coincide exactly after the rebuild (committed far apart, rebuilt at one
  pose), with scan ids beyond 2^40;
* a non-dyadic width (w = 0.8) with world coordinates placed on fl(k w) and one ulp either side;
* queries exactly max_dist_matching and min_dist_map away from their neighbours;
* poses far from the origin, a sparse map, and buckets of 15 / 16 / 17 / 64 / 65 and > 65535 points.

A scene is a list of operations (extract, rebuild, associate, commit); `run` plays it on anything
with the methods of form_b200.context.Context (the CPU oracle has the same ones).  The poses are
chosen here, not by a smoother, so every call is reproducible from the scene alone.

`brute_force_r5` is the check that does not depend on the oracle's search: a vectorised numpy scan
of the 27 voxels around each query with the reference's arithmetic (IEEE division for the voxel
key, the 4-lane squared norm) and the arg-min of (dist^2, shift rank, scan id, k) over the full
64-bit scan id."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from form_b200 import _capi, synth
from helpers import scan_poses
from np_restatement import SHIFTS, transform

DBL_MAX = np.finfo(np.float64).max
ROWS, COLS = 16, 256  # shape of the lattice scans


# ---------------------------------------------------------------------------------------------
# poses
# ---------------------------------------------------------------------------------------------
def pose(R=None, t=(0.0, 0.0, 0.0)):
    out = np.zeros((), dtype=_capi.POSE)
    out["R"] = (np.eye(3) if R is None else np.asarray(R, dtype=np.float64)).reshape(9)
    out["t"] = np.asarray(t, dtype=np.float64)
    return out


def rotz(quarter: int) -> np.ndarray:
    """Exact rotation by quarter * 90 degrees about z (integer entries)."""
    c, s = [(1, 0), (0, 1), (-1, 0), (0, -1)][quarter % 4]
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], dtype=np.float64)


def compose(a, b):
    """a * b (apply b, then a)."""
    Ra, Rb = a["R"].reshape(3, 3), b["R"].reshape(3, 3)
    return pose(Ra @ Rb, Ra @ b["t"] + a["t"])


def translated(p, d):
    return pose(p["R"].reshape(3, 3), p["t"] + np.asarray(d, dtype=np.float64))


# ---------------------------------------------------------------------------------------------
# lattice rooms
# ---------------------------------------------------------------------------------------------
def _walk(a: int, pillars=((-20, 3, 2), (-4, 2, 3), (10, 4, 1))) -> np.ndarray:
    """Lattice points (units of the step) along the walls of a square room of half-size a: the
    first wall carries pillars (x position, depth into the room, width)."""
    pts = []
    x, y = -a, -a

    def go(dx, dy, n):
        nonlocal x, y
        for _ in range(n):
            x += dx
            y += dy
            pts.append((x, y))

    for px, depth, width in pillars:
        go(1, 0, px - x)
        go(0, 1, depth)
        go(1, 0, width)
        go(0, -1, depth)
    go(1, 0, a - x)
    go(0, 1, 2 * a)
    go(-1, 0, 2 * a)
    go(0, -1, 2 * a)
    return np.array(pts, dtype=np.int64)


def room_world(phase: int = 0, zphase: int = 0, zstep: int = 2, dup_rows=(), a: int = 32) -> np.ndarray:
    """(ROWS*COLS, 3) integer lattice coordinates of one scan of the room: row r at height
    (r - 5) * zstep + zphase, its columns walking the walls from `phase`; the top quarter of the rows
    walks an inset wall (a ledge).  Rows listed in dup_rows repeat the row below (identical points
    inside one scan)."""
    low, high = _walk(a), _walk(a - 2, pillars=((-10, 2, 2),))
    out = np.zeros((ROWS, COLS, 3), dtype=np.int64)
    for r in range(ROWS):
        src = r - 1 if r in dup_rows else r
        w = high if src >= 3 * ROWS // 4 else low
        idx = (phase + np.arange(COLS)) % len(w)
        out[r, :, :2] = w[idx]
        out[r, :, 2] = (src - 5) * zstep + zphase
    return out.reshape(-1, 3)


def organised(points_sensor: np.ndarray) -> np.ndarray:
    """(n, 3) float64 sensor-frame points (exact in float32) -> POINT4F scan; rows of zeros stay
    missing returns."""
    f = points_sensor.astype(np.float32)
    assert np.array_equal(f.astype(np.float64), points_sensor), "scan points must be exact in float32"
    scan = np.zeros(len(f), dtype=_capi.POINT4F)
    scan["x"], scan["y"], scan["z"] = f[:, 0], f[:, 1], f[:, 2]
    return scan


def room_scan(step: float, sensor, **kw) -> np.ndarray:
    """The room seen from `sensor` (a pose with an exact rotation and a lattice translation)."""
    P = room_world(**kw).astype(np.float64) * step
    R = sensor["R"].reshape(3, 3)
    p = (P - sensor["t"]) @ R  # R^T (P - t), exact: integer rotation, lattice values
    n2 = np.sum(p * p, axis=1)
    assert np.all((n2 >= 1.0) & (n2 <= 1e4)), "every point within the valid range of its sensor"
    return organised(p)


# ---------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------
@dataclass
class Scene:
    name: str
    params: dict                               # formgpu_params overrides (rows / cols included)
    ops: list = field(default_factory=list)    # ("extract", id, scan) / ("rebuild", {id: pose}) /
                                               # ("associate", pose) / ("commit", id)
    sample: int | None = None                  # queries checked by brute force (None: all)

    @property
    def width(self) -> float:
        return float(self.params["max_dist_matching"])

    def make_params(self) -> _capi.Params:
        p = dict(self.params)
        rows, cols = p.pop("num_rows", ROWS), p.pop("num_columns", COLS)
        return _capi.default_params(rows, cols, **p)

    def step(self, scan_id, scan, rebuild: dict, assoc: list, commit=True):
        self.ops.append(("extract", scan_id, scan))
        self.ops.append(("rebuild", dict(rebuild)))
        for p in assoc:
            self.ops.append(("associate", p))
        if commit:
            self.ops.append(("commit", scan_id))


def _sensor(quarter, t_units, step):
    return pose(rotz(quarter), np.asarray(t_units, dtype=np.float64) * step)


def lattice(w: float, cell_centre: bool = False, offset=(0.0, 0.0, 0.0), name=None) -> Scene:
    """Six scans of the lattice room with step w / 4 from exact poses (90-degree rotations, lattice
    translations), sampling it with different row and column phases: every association query ties
    across shift ranks, scans and keypoints.  `cell_centre` adds a second association per scan at
    the pose shifted by w / 8 on every axis (queries at cell centres).  `offset` translates the whole
    window (far from the origin); it must be exact."""
    s = w / 4
    sc = Scene(name or f"lattice_w{w}", dict(max_dist_matching=w, min_dist_map=min(0.1, s / 2)))
    sensors = [(0, (0, 0, 0), 0, 0), (1, (4, -3, 0), 0, 1), (2, (-5, 2, 1), 3, 0), (3, (2, 6, -1), 1, 1),
               (0, (-3, -4, 0), 2, 0), (2, (6, 1, 1), 0, 1)]
    done = {}
    for i, (q, tu, ph, zph) in enumerate(sensors):
        sensor = _sensor(q, tu, s)
        scan = room_scan(s, sensor, phase=ph, zphase=zph)
        world = translated(sensor, offset)
        assoc = [world]
        if cell_centre:
            assoc = [translated(world, (s / 2, s / 2, s / 2)), world]
        sc.step(10 + i, scan, {**done, 10 + i: world}, assoc)
        done[10 + i] = world
    return sc


def duplicates(ids=(1, 2, 3, 4), shift_one=False, dup_rows=(), name="duplicates") -> Scene:
    """Each scan (the same room scan, so the same keypoints) is committed at a distant pose, where
    nothing matches and every keypoint is stored; the last rebuild puts all of them at one pose, so
    stored points coincide exactly across scans and the ties go to the lower scan id, then k.
    shift_one: the second scan is rebuilt one cell (w / 4) off.  dup_rows: rows repeated inside the
    scan (ties on k inside one scan)."""
    w = 0.5
    s = w / 4
    sc = Scene(name, dict(max_dist_matching=w, min_dist_map=0.1))
    scan = room_scan(s, pose(), dup_rows=dup_rows)
    done = {}
    for n, i in enumerate(ids):
        far = pose(t=(1000.0 * (n + 1), -2000.0, 500.0))
        sc.step(i, scan, {**done, i: far}, [far])
        done[i] = far
    aligned = {i: pose() for i in ids}
    if shift_one:
        aligned[ids[1]] = pose(t=(s, 0.0, 0.0))
    cur = ids[-1] + 7 if ids[-1] < 2**63 else 6
    q_scan = room_scan(s, pose(rotz(1), (0.0, 0.0, s)), phase=1, zphase=1)
    sc.step(cur, q_scan, {**aligned, cur: pose(rotz(1), (0.0, 0.0, s))},
            [pose(rotz(1), (0.0, 0.0, s)), pose()])
    return sc


def large_ids() -> Scene:
    """The duplicates scene with scan ids that need all 64 bits, mixed with small ones: 1 and
    2^40 + 1 (and 5 and 2^63 + 5) differ only above bit 40."""
    return duplicates(ids=(3, 2**40 + 1, 1, 2**63 + 5, 2**40, 5), name="large_ids")


def face_target(w: float, k: int, ulps: int) -> float:
    """fl(k w) moved by `ulps` units in the last place."""
    v = float(np.float64(k) * w)
    for _ in range(abs(ulps)):
        v = float(np.nextafter(v, np.inf if ulps > 0 else -np.inf))
    return v


def fast_path_fails(v: float, w: float) -> bool:
    """floor(v * fl(1 / w)) != floor(v / w): the voxel key's fast path alone would be wrong."""
    return bool(np.floor(v * (1.0 / w)) != np.floor(v / w))


def failing_k(w: float, ks) -> int:
    """The first k for which one of fl(k w), one ulp below, one ulp above fails the fast path."""
    for k in ks:
        if any(fast_path_fails(face_target(w, k, d), w) for d in (-1, 0, 1)):
            return k
    raise AssertionError("no k in range")


def _place(x: float, target: float) -> float:
    """t with fl(x + t) == target (x + t is the last operation of the transform at R = I)."""
    t = target - x
    for _ in range(64):
        got = x + t
        if got == target:
            return t
        t = float(np.nextafter(t, np.inf if got < target else -np.inf))
    raise AssertionError("no translation puts the coordinate on the target")


def face_aligned() -> Scene:
    """w = 0.8 (fl(1 / w) inexact).  Per rebuild and per association the translations put the
    wall x = +a s, the wall y = +a s and the height of row 7 of the scan exactly on fl(k w) or one
    ulp either side, with k chosen where the voxel key's fast path disagrees with the division for
    one of the three (k < 0 on the y axis).  Every stored scan gets a new choice at every rebuild."""
    w, s, a = 0.8, 0.125, 32
    sc = Scene("face_aligned", dict(max_dist_matching=w, min_dist_map=0.1))
    kx, ky, kz = failing_k(w, range(300, 400)), failing_k(w, range(-300, -400, -1)), failing_k(w, range(40, 140))
    wall, row_z = a * s, (7 - 5) * 2 * s

    def at(v):
        dx, dy, dz = v % 3 - 1, (v // 3) % 3 - 1, (v // 9) % 3 - 1
        return pose(t=(_place(wall, face_target(w, kx, dx)), _place(wall, face_target(w, ky, dy)),
                       _place(row_z, face_target(w, kz, dz))))

    done = []
    for i in range(5):
        scan = room_scan(s, pose(), phase=3 * i, zphase=0)
        rebuild = {j: at(7 * i + 5 * n) for n, j in enumerate(done)}
        cur = at(11 * i + 4)
        rebuild[30 + i] = cur
        sc.step(30 + i, scan, rebuild, [at(11 * i + 13), at(11 * i + 22), cur])
        done.append(30 + i)
    # exact ties across a face whose voxel only the division gets right: the query scan's wall
    # x = +a s on such a v, two stored scans' walls one lattice step either side (v -+ s, exact), so
    # the winner is whichever of the two lies in the query's own voxel
    v = next(c for c in (face_target(w, k, d) for k in range(300, 400) for d in (-1, 0, 1))
             if fast_path_fails(c, w))
    ty, tz = _place(wall, face_target(w, ky, 0)), _place(row_z, face_target(w, kz, 0))
    side = {35: pose(t=(_place(wall, v - s), ty, tz)), 36: pose(t=(_place(wall, v + s), ty, tz))}
    for sid, p in side.items():
        sc.step(sid, room_scan(s, pose()), {**{j: at(j) for j in done}, **side}, [pose(t=(5000.0, 0.0, 0.0))])
        done.append(sid)
    q = pose(t=(_place(wall, v), ty, tz))
    sc.step(37, room_scan(s, pose(), phase=1), {**{j: pose(t=(5000.0 + 50.0 * j, 0.0, 0.0)) for j in done[:5]}, **side, 37: q}, [q])
    return sc


def gates() -> Scene:
    """max_dist_matching = 1, min_dist_map = 0.25, lattice step 0.25: the query scan is associated
    at its pose moved by exactly 1 and exactly 0.25 across the walls and between the rows, so many
    queries are exactly max_dist_matching (not a pair) or min_dist_map (not novel) from their nearest
    neighbour."""
    s = 0.25
    sc = Scene("gates", dict(max_dist_matching=1.0, min_dist_map=0.25))
    s0 = _sensor(0, (0, 0, 0), s)
    sc.step(40, room_scan(s, s0), {40: s0}, [s0])
    s1 = _sensor(1, (3, -2, 0), s)
    moves = [(1.0, 0, 0), (0, -1.0, 0), (0.25, 0, 0), (0, 0, 0.25), (0, 0, 1.0), (0, 0, 0)]
    sc.step(41, room_scan(s, s1, phase=5), {40: s0, 41: s1}, [translated(s1, m) for m in moves])
    s2 = _sensor(3, (-2, 1, 0), s)
    sc.step(42, room_scan(s, s2, phase=9, zphase=1), {40: s0, 41: s1, 42: s2},
            [translated(s2, m) for m in [(0, 0, 0.25), (-1.0, 0, 0), (0, 0, 0)]])
    return sc


def far(w: float, offset) -> Scene:
    """The lattice scene (with the cell-centre associations) translated far from the origin."""
    return lattice(w, cell_centre=True, offset=offset, name=f"far_w{w}")


def synthetic_far(n_scans: int = 4) -> Scene:
    """Synthetic VLP-16 scans whose ground-truth trajectory is moved by a generic rotation and
    |t| = 2e4 m; associations at perturbed poses (the smoother's job in the pipeline)."""
    from helpers import perturbed

    rows, cols = synth.shape("vlp-16")
    sc = Scene("synthetic_far", dict(num_rows=rows, num_columns=cols, max_dist_matching=0.8, min_dist_map=0.1))
    ax = np.array([0.3, -0.5, 0.8]) / np.linalg.norm([0.3, -0.5, 0.8])
    th = 0.9
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    G = pose(np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K, (12000.0, -15000.5, 5000.25))
    rng = np.random.default_rng(7)
    done = {}
    for k in range(n_scans):
        true = compose(G, synth.gt_pose(0, k))
        cur = perturbed(true, rng, 0.0005, 0.005)
        assoc = [perturbed(true, rng, 0.002, 0.03), perturbed(true, rng, 0.001, 0.01)]
        sc.step(k, synth.scan("vlp-16", 0, k), {**done, k: cur}, assoc)
        done[k] = assoc[-1]
    return sc


def sparse() -> Scene:
    """A map of a few dozen points (three small patches of one scan) against a full room scan:
    most queries have no neighbour at all (found = 0, dist^2 = DBL_MAX); near the patches the
    query's own voxel is often empty and its neighbour lies in a diagonal voxel."""
    w = 0.5
    s = w / 4
    sc = Scene("sparse", dict(max_dist_matching=w, min_dist_map=0.1))
    full = room_scan(s, pose()).reshape(ROWS, COLS)
    patchy = np.zeros_like(full)
    for r0, c0 in [(4, 20), (8, 100), (11, 190)]:
        patchy[r0:r0 + 3, c0:c0 + 16] = full[r0:r0 + 3, c0:c0 + 16]
    sc.step(50, patchy.reshape(-1), {50: pose()}, [pose()])
    q = _sensor(2, (3, 3, 1), s)
    sc.step(51, room_scan(s, q, phase=2, zphase=1), {50: pose(), 51: q},
            [translated(q, (s / 2, -s / 2, s / 2)), translated(q, (0.3, 0.2, 0.1)), q])
    return sc


BUCKET_SEED = 19  # lattice offsets of the rebuild in `buckets` (a seed whose map has every edge size)


def buckets(seed: int = BUCKET_SEED, n_scans: int = 28) -> Scene:
    """The same room scan committed n_scans times at distant poses (every keypoint stored), then
    rebuilt at small lattice offsets: voxel buckets are sums of the scans' shares and take every
    size, among them 15 / 16 / 17 (kCellMin, the smallest cell-ordered bucket) and 64 / 65 (the
    largest bucket a warp keeps in registers while it orders it)."""
    w = 0.5
    s = w / 4
    sc = Scene(f"buckets_{seed}", dict(max_dist_matching=w, min_dist_map=0.1))
    scan = room_scan(s, pose())
    rng = np.random.default_rng(seed)
    done = {}
    for i in range(n_scans):
        far_pose = pose(t=(-3000.0 * (i + 1), 700.0, 0.0))
        sc.step(100 + i, scan, {**done, 100 + i: far_pose}, [far_pose])
        done[100 + i] = far_pose
    rebuild = {i: pose(t=rng.integers(-1, 2, size=3) * s) for i in done}
    q = _sensor(1, (1, 1, 0), s)
    sc.step(200, room_scan(s, q, phase=4, zphase=1), {**rebuild, 200: q},
            [translated(q, (s / 2, s / 2, s / 2)), q])
    return sc


def huge_bucket(n_scans: int = 5) -> Scene:
    """Five OS0-128 synthetic scans committed at distant poses, then rebuilt at t = (32, 32, 32)
    with max_dist_matching = 64: one voxel holds far more than kCellMax = 65535 points, so it gets
    no cell table and every search in it scans the whole bucket.  Checked on a fixed sample of the
    queries."""
    rows, cols = synth.shape("os0-128")
    sc = Scene("huge_bucket", dict(num_rows=rows, num_columns=cols, max_dist_matching=64.0, min_dist_map=0.1),
               sample=2000)
    done = {}
    for k in range(n_scans):
        far_pose = pose(t=(5000.0 * (k + 1), 0.0, 0.0))
        sc.step(80 + k, synth.scan("os0-128", 0, k), {**done, 80 + k: far_pose}, [far_pose])
        done[80 + k] = far_pose
    centre = pose(t=(32.0, 32.0, 32.0))
    sc.step(80 + n_scans, synth.scan("os0-128", 0, n_scans), {**{i: centre for i in done}, 80 + n_scans: centre},
            [centre], commit=True)
    return sc


def all_scenes() -> list:
    return [lattice(0.5, cell_centre=True), lattice(1.0), duplicates(), duplicates(shift_one=True, name="dup_shift"),
            duplicates(dup_rows=(6, 9), name="dup_rows"), large_ids(), face_aligned(), gates(),
            far(0.5, (2.0**16, -2.0**14, 2.0**12)), far(1.0, (-2.0**15, 2.0**13, -2.0**16)), synthetic_far(),
            sparse(), buckets(), huge_bucket()]


# ---------------------------------------------------------------------------------------------
# playing a scene
# ---------------------------------------------------------------------------------------------
def do(backend, op):
    """One operation on a Context / Oracle; the result carries what the parity checks compare."""
    if op[0] == "extract":
        return backend.extract(op[2], op[1])
    if op[0] == "rebuild":
        backend.map_rebuild(scan_poses(list(op[1]), list(op[1].values())))
        return None
    if op[0] == "associate":
        counts = backend.associate(op[1])
        return counts, backend.matches(0), backend.matches(1)
    if op[0] == "commit":
        added = backend.commit_scan()
        return added, backend.keypoints(0, op[1]), backend.keypoints(1, op[1])
    raise ValueError(op[0])


def run(scene: Scene, backend) -> list:
    return [do(backend, op) for op in scene.ops]


def run_lockstep(scenes: list, do_many) -> list:
    """Plays several scenes side by side: do_many([(i, op), ...]) runs the next operation of every
    scene that still has one (one batched submission) and returns their results in that order."""
    recs = [[] for _ in scenes]
    for n in range(max(len(s.ops) for s in scenes)):
        todo = [(i, s.ops[n]) for i, s in enumerate(scenes) if n < len(s.ops)]
        for (i, _), r in zip(todo, do_many(todo)):
            recs[i].append(r)
    return recs


# ---------------------------------------------------------------------------------------------
# the independent rule R5
# ---------------------------------------------------------------------------------------------
_B = 1 << 20


def _code(keys: np.ndarray) -> np.ndarray:
    assert np.all(np.abs(keys) < _B - 2), "voxel keys outside the packed range of the brute force"
    k = keys + _B
    return (k[..., 0] << 42) | (k[..., 1] << 21) | k[..., 2]


def brute_force_r5(world_pts, scan_ids, ks, queries, w: float, max_pairs: int = 4_000_000) -> dict:
    """VoxelMap::find_closest for every query by exhaustive search of the 27 voxels around it:
    voxel keys floor(p / w) with an IEEE division, dist^2 = (d0^2 + d2^2) + (d1^2 + 0), arg-min of
    (dist^2, shift rank, scan id (all 64 bits), k).  Also reports the ties that rule R5 decides.
    Returns arrays over the queries: found, scan, k, dist_sqrd (DBL_MAX when nothing is found),
    rank, and the tie classes (tie_rank: tied candidates in different shift ranks; tie_scan: same
    rank, different scans; tie_k: same scan; tie_hi40: tied scans equal in their low 40 bits)."""
    world_pts = np.asarray(world_pts, dtype=np.float64).reshape(-1, 3)
    queries = np.asarray(queries, dtype=np.float64).reshape(-1, 3)
    scan_ids = np.asarray(scan_ids, dtype=np.uint64)
    ks = np.asarray(ks, dtype=np.uint32)
    m = len(queries)
    out = dict(found=np.zeros(m, bool), scan=np.zeros(m, np.uint64), k=np.zeros(m, np.uint32),
               dist_sqrd=np.full(m, DBL_MAX), rank=np.full(m, -1), tie_rank=np.zeros(m, bool),
               tie_scan=np.zeros(m, bool), tie_k=np.zeros(m, bool), tie_hi40=np.zeros(m, bool))
    if m == 0 or len(world_pts) == 0:
        return out
    codes = _code(np.floor(world_pts / w).astype(np.int64))
    order = np.argsort(codes, kind="stable")
    codes, wp, sc, kk = codes[order], world_pts[order], scan_ids[order], ks[order]
    qkeys = np.floor(queries / w).astype(np.int64)
    qc = _code(qkeys[:, None, :] + SHIFTS[None, :, :])            # (m, 27)
    lo = np.searchsorted(codes, qc, side="left")
    cnt = np.searchsorted(codes, qc, side="right") - lo
    per_q = cnt.sum(axis=1)
    start = 0
    while start < m:
        cum = np.cumsum(per_q[start:])
        stop = start + max(1, int(np.searchsorted(cum, max_pairs, side="right")))
        _chunk(out, start, min(stop, m), lo, cnt, per_q, codes, wp, sc, kk, queries)
        start = stop
    return out


def _chunk(out, a, b, lo, cnt, per_q, codes, wp, sc, kk, queries):
    c = cnt[a:b].reshape(-1)
    total = int(c.sum())
    if total == 0:
        return
    q_of = np.repeat(np.arange(a, b), per_q[a:b])
    rank_of = np.repeat(np.tile(np.arange(27), b - a), c)
    first = np.repeat(lo[a:b].reshape(-1), c)
    within = np.arange(total) - np.repeat(np.cumsum(c) - c, c)
    cand = first + within
    d = wp[cand] - queries[q_of]
    d2 = (d[:, 0] * d[:, 0] + d[:, 2] * d[:, 2]) + (d[:, 1] * d[:, 1] + 0.0)
    has = per_q[a:b] > 0
    starts = np.concatenate([[0], np.cumsum(per_q[a:b])[:-1]])[has]
    best = np.full(b - a, np.inf)
    best[has] = np.minimum.reduceat(d2, starts)
    tied = d2 == best[q_of - a]
    tq, tr, ts, tk = q_of[tied], rank_of[tied], sc[cand[tied]], kk[cand[tied]]
    o = np.lexsort((tk, ts, tr, tq))
    tq, tr, ts, tk = tq[o], tr[o], ts[o], tk[o]
    head = np.ones(len(tq), bool)
    head[1:] = tq[1:] != tq[:-1]
    wq = tq[head]
    out["found"][wq] = True
    out["dist_sqrd"][wq] = best[wq - a]
    out["rank"][wq] = tr[head]
    out["scan"][wq] = ts[head]
    out["k"][wq] = tk[head]
    # tie classes: compare every tied candidate with its query's winner
    wi = np.cumsum(head) - 1
    w_r, w_s = tr[head][wi], ts[head][wi]
    other = ~head
    np.logical_or.at(out["tie_rank"], tq[other & (tr != w_r)], True)
    same_r = other & (tr == w_r)
    np.logical_or.at(out["tie_scan"], tq[same_r & (ts != w_s)], True)
    np.logical_or.at(out["tie_k"], tq[same_r & (ts == w_s)], True)
    lo40 = np.uint64((1 << 40) - 1)
    np.logical_or.at(out["tie_hi40"], tq[same_r & (ts != w_s) & ((ts & lo40) == (w_s & lo40))], True)


# ---------------------------------------------------------------------------------------------
# what every association of a scene must return, from the oracle's stored keypoints
# ---------------------------------------------------------------------------------------------
def _xyz(kp) -> np.ndarray:
    return np.stack([kp["x"], kp["y"], kp["z"]], axis=1) if len(kp) else np.zeros((0, 3))


def _world(p, kp):
    return transform(p["R"], p["t"], _xyz(kp)) if len(kp) else np.zeros((0, 3))


def sample_of(n: int, sample: int | None, seed: int = 0) -> np.ndarray:
    if sample is None or n <= sample:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=sample, replace=False))


def expectations(scene: Scene, recs: list) -> list:
    """For every associate operation of the scene, from the records of a run (the oracle's): per
    type the brute-force result on the checked queries (all, or the scene's fixed sample), their
    indices, the map's bucket sizes and world coordinates, and the numpy gates (pair counts by
    scan id, novel count)."""
    w = scene.width
    p = scene.make_params()
    max2, min2 = p.max_dist_matching * p.max_dist_matching, p.min_dist_map * p.min_dist_map
    stored, cur_kp, maps, out = {}, None, None, []
    for op, r in zip(scene.ops, recs):
        if op[0] == "extract":
            cur_kp = r
        elif op[0] == "commit":
            stored[op[1]] = (r[1], r[2])
        elif op[0] == "rebuild":
            maps = []
            for t in (0, 1):
                pts, ids, ks = [np.zeros((0, 3))], [np.zeros(0, np.uint64)], [np.zeros(0, np.uint32)]
                for sid, ps in op[1].items():
                    if sid in stored and len(stored[sid][t]):
                        kp = stored[sid][t]
                        pts.append(_world(ps, kp))
                        ids.append(np.full(len(kp), sid, dtype=np.uint64))
                        ks.append(np.arange(len(kp), dtype=np.uint32))
                maps.append((np.concatenate(pts), np.concatenate(ids), np.concatenate(ks)))
        elif op[0] == "associate":
            e = dict(types=[])
            for t in (0, 1):
                q = _world(op[1], cur_kp[t])
                idx = sample_of(len(q), scene.sample, seed=t)
                bf = brute_force_r5(*maps[t], q[idx], w)
                keys = np.floor(maps[t][0] / w).astype(np.int64)
                _, sizes = np.unique(keys, axis=0, return_counts=True) if len(keys) else (None, np.zeros(0, int))
                own = set(map(tuple, keys)) if len(keys) else set()
                qk = np.floor(q[idx] / w).astype(np.int64)
                own_empty = np.array([tuple(v) not in own for v in qk], dtype=bool)
                e["types"].append(dict(idx=idx, bf=bf, sizes=sizes, map_xyz=maps[t][0], query_xyz=q[idx],
                                       own_empty=own_empty, n_query=len(q)))
            out.append(e)
            # numpy gates over all queries (possible only when nothing is sampled)
            if scene.sample is None:
                counts = {}
                novel = []
                for t in (0, 1):
                    bf = e["types"][t]["bf"]
                    pair = bf["found"] & (bf["dist_sqrd"] < max2)
                    for sid, n in zip(*np.unique(bf["scan"][pair], return_counts=True)):
                        counts.setdefault(int(sid), [0, 0])[t] = int(n)
                    novel.append(int(np.count_nonzero(bf["dist_sqrd"] > min2)))
                e["counts"], e["novel"] = counts, novel
    return out


_CACHE: dict = {}


def oracle_run(scene: Scene):
    """The oracle's records of a scene and their brute-force expectations, computed once per
    process (shared by the CPU and the GPU tests of one session)."""
    if scene.name not in _CACHE:
        import oracle_lib

        ref = oracle_lib.Oracle(scene.make_params())
        try:
            recs = run(scene, ref)
        finally:
            ref.close()
        _CACHE[scene.name] = (recs, expectations(scene, recs))
    return _CACHE[scene.name]
