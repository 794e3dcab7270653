"""Adversarial organised scans for stage 1 (extract.cu: select, normals and pack kernels).

Every scene is a `Scene(name, params, scan, reach)` built deterministically from dyadic (or
otherwise exactly representable) float32 values, and aimed at one comparison of the extraction:
a range gate, the neighbour radius, the planar threshold, a curvature or closest-point tie, the
pruning margin of the adjacent-row search, the eigen solver's branches, or a sector / capacity /
shape edge.  `reach(R)` asserts, on the numpy restatement of np_restatement.py (`restate`), that
the scene really lands on its edge; test_extract_scenes_cpu.py calls it for every scene.

Conventions.  The background of most scenes is a "zig-zag" wall: x alternates between 8 and 9
from column to column, so every background column has curvature (2 ceil(np/2))^2 >= 4 and never
passes the default planar threshold; a "segment" stamped at column c (`stamp`) is symmetric about
c (p - d_k at c - k, p + d_k at c + k), so the curvature at c is exactly 0 and c is the first
candidate of its sector.  Adjacent rows are usually copies shifted by 1/2 in z, so the closest
adjacent-row point of a pick is its own column.

Edges an organised scan cannot reach (nothing tests them):
- The QL iteration cap (`iter > 90`): the implicit symmetric QL step on a 3x3 tridiagonal matrix
  deflates in a handful of iterations for every finite input (Eigen's cap exists for the n x n
  case); no covariance of at most 49 points reaches it.
- A nonzero box bound that the (1 - 1e-5) margin leaves unchanged: that needs a subnormal bound,
  a pick and an adjacent-row chunk closer than 2^-63 in every lane without touching.  The bound 0
  (coincident points) is reached (`closest_seed_zero`), and it is what tells `<=` from `<` in the
  pruning test.  For a normal bound the margin keeps every chunk whose points could tie with the
  seed (their dist^2 is within a few ulp of the bound, far inside 1e-5), so there `<=` and `<`
  give the same answer.
- Which chunk seeds the fallback search when two boxes tie: the seed only orders the evaluation,
  the pruning after it is conservative and the (dist^2, column) minimum does not depend on the
  order in which chunks are evaluated (`closest_fallback` builds the tie; the answer is fixed).
- Column cols-1 as a closest point: edge columns are never valid (find_closest only considers
  valid points), so the last candidate column is cols-np-1 (`closest_ties`).
"""
from __future__ import annotations

import dataclasses
from typing import Callable

import numpy as np

import np_restatement as npr
from form_b200 import _capi

F32 = np.float32
FLT_MIN = float(np.finfo(np.float32).tiny)  # 2^-126


@dataclasses.dataclass
class Scene:
    name: str
    params: _capi.Params
    scan: np.ndarray            # POINT4F, rows * cols
    reach: Callable[[dict], None]
    edge: str = ""

    @property
    def rows(self):
        return self.params.num_rows

    @property
    def cols(self):
        return self.params.num_columns

    def s4(self):
        return np.stack([self.scan["x"], self.scan["y"], self.scan["z"], self.scan["w"]], axis=1)


def to_scan(P):
    P = np.ascontiguousarray(P, dtype=F32).reshape(-1, 4)
    scan = np.zeros(len(P), dtype=_capi.POINT4F)
    for i, f in enumerate("xyzw"):
        scan[f] = P[:, i]
    return scan


def params(rows, cols, **kw):
    return _capi.default_params(rows, cols, **kw)


def sqn(d):
    """sqnorm4 of one 4-vector in float32, Eigen's packet order."""
    return float(npr.sqnorm4_f32(np.asarray(d, F32)[None, :])[0])


def ulp_up(x):
    return float(np.nextafter(F32(x), F32(np.inf)))


def ulp_down(x):
    return float(np.nextafter(F32(x), F32(-np.inf)))


def split_yw(target, y_candidates=None):
    """A difference vector (0, y, 0, w) whose float32 sqnorm4 is exactly `target` (y a coarse
    dyadic, so that p.y + y stays exact; w is free because p.w = 0)."""
    for y in y_candidates or [k / 64 for k in range(63, 0, -1)]:
        y2 = F32(y) * F32(y)
        rest = float(target) - float(y2)
        if rest < 0:
            continue
        w0 = F32(np.sqrt(rest))
        for k in range(-4, 5):
            w = F32(w0)
            for _ in range(abs(k)):
                w = np.nextafter(w, F32(np.inf) if k > 0 else F32(-np.inf))
            d = np.array([0.0, y, 0.0, w], F32)
            if sqn(d) == float(F32(target)):
                return d
    raise AssertionError(f"no (y, w) split of {target!r}")


def zigzag(rows, cols, x0=8.0, dz=0.5, step=1 / 16):
    c = np.arange(cols)
    P = np.zeros((rows, cols, 4), F32)
    P[..., 0] = x0 + (c % 2)
    P[..., 1] = (c - cols // 2) * step
    P[..., 2] = (np.arange(rows) * dz)[:, None]
    return P


def wall(rows, cols, x0=8.0, dz=0.5, step=1 / 16):
    """A straight wall: every valid column has curvature exactly 0."""
    P = zigzag(rows, cols, x0, dz, step)
    P[..., 0] = x0
    return P


def stamp(P, r, c, offsets):
    """Symmetric segment centred on (r, c): p + d_k at c + k, p - d_k at c - k (k = 1..len)."""
    p = P[r, c].copy()
    p[0] = 8.0
    P[r, c] = p
    for k, d in enumerate(offsets, start=1):
        d = np.asarray(d, F32)
        P[r, c + k] = p + d
        P[r, c - k] = p - d
        assert np.array_equal((P[r, c + k] - p).astype(F32), d) and np.array_equal((p - P[r, c - k]).astype(F32), d)
    # guards: the first column past each end sticks out by 2 m, so that no column next to the
    # centre sees a straight window (its curvature would tie with the centre's 0 at a lower column)
    L = len(offsets)
    if c + L + 1 < P.shape[1]:
        P[r, c + L + 1, 0] = 10.0
    if c - L - 1 >= 0:
        P[r, c - L - 1, 0] = 10.0


# --------------------------------------------------------------------------------------------
# the numpy restatement of one scene
# --------------------------------------------------------------------------------------------
def restate(scene):
    """Everything the reach assertions and the CPU comparison need, from np_restatement only."""
    p = scene.params
    rows, cols, np_ = p.num_rows, p.num_columns, p.neighbor_points
    s4 = scene.s4()
    valid, pvalid = npr.masks(s4, rows, cols, np_, p.min_norm_squared, p.max_norm_squared)
    curv = npr.curvature(s4, rows, cols, np_, valid)
    picks, used = npr.planar_picks(curv, valid, rows, cols, np_, p.num_sectors, p.planar_threshold,
                                   p.planar_feats_per_sector)
    qpicks = npr.point_picks(used, valid, pvalid, rows, cols, np_, p.num_sectors, p.point_feats_per_sector)
    r2 = p.radius * p.radius
    cprev, cnext, keep, nbrs, count = [], [], [], [], []
    for idx in picks.tolist():
        row = idx // cols
        cp = npr.closest_in_row(s4, valid, s4[idx], (row - 1) * cols, row * cols) if row > 0 else -1
        cn = npr.closest_in_row(s4, valid, s4[idx], (row + 1) * cols, (row + 2) * cols) if row < rows - 1 else -1
        nb = npr.neighbor_list(s4, idx, np_, r2)
        for c in (cp, cn):
            if c >= 0:
                nb = nb + [s4[c]] + npr.neighbor_list(s4, c, np_, r2)
        cprev.append(cp)
        cnext.append(cn)
        nbrs.append(nb)
        count.append(len(nb))
        keep.append((cp >= 0 or cn >= 0) and len(nb) >= p.min_points)
    return dict(s4=s4, valid=valid, pvalid=pvalid, curv=curv, picks=picks, used=used, qpicks=qpicks,
                cprev=np.array(cprev, np.int32), cnext=np.array(cnext, np.int32), keep=np.array(keep, bool),
                nbrs=nbrs, count=np.array(count, int), rows=rows, cols=cols, np=np_, params=p)


def candidate_ties(R):
    """Does any sector hold two planar candidates (valid, below the threshold) of equal curvature?"""
    p = R["params"]
    cv = R["curv"].reshape(R["rows"], R["cols"])
    ok = R["valid"].reshape(R["rows"], R["cols"]) & (cv.astype(np.float64) < p.planar_threshold)
    for a, b in npr.sectors(R["cols"], p.num_sectors):
        for r in range(R["rows"]):
            v = cv[r, a:b][ok[r, a:b]]
            if len(np.unique(v)) < len(v):
                return True
    return False


def cov_f32(s4, idx, nbrs):
    """compute_normal's covariance in float32 in the oracle's order: (c00, c10, c11, c20, c21, c22)."""
    p = s4[idx].astype(F32)
    nf = F32(len(nbrs))
    c = [F32(0)] * 6
    for q in nbrs:
        a0, a1, a2 = ((q[0] - p[0]) / nf, (q[1] - p[1]) / nf, (q[2] - p[2]) / nf)
        a0, a1, a2 = F32(a0), F32(a1), F32(a2)
        c = [F32(c[0] + a0 * a0), F32(c[1] + a1 * a0), F32(c[2] + a1 * a1), F32(c[3] + a2 * a0),
             F32(c[4] + a2 * a1), F32(c[5] + a2 * a2)]
    return c


def v1norm2(c):
    """The solver's (m20 / scale)^2 in float32 (0 scale -> 1)."""
    scale = max(abs(x) for x in c)
    if scale == 0:
        scale = F32(1)
    m20 = F32(c[3] / F32(scale))
    return F32(m20 * m20), F32(scale)


def pick_pos(R, r, c):
    """Position of the planar pick (r, c) in the pick list, asserting it was picked."""
    where = np.nonzero(R["picks"] == r * R["cols"] + c)[0]
    assert len(where) == 1, f"({r}, {c}) is not a planar pick"
    return int(where[0])


def d2row(R, idx, row):
    """float32 dist^2 from point idx to every valid point of `row` (inf where invalid)."""
    cols = R["cols"]
    seg = R["s4"][row * cols:(row + 1) * cols]
    d = npr.sqnorm4_f32(seg - R["s4"][idx][None, :])
    return np.where(R["valid"][row * cols:(row + 1) * cols], d, np.inf)


# --------------------------------------------------------------------------------------------
# scenes
# --------------------------------------------------------------------------------------------
def range_gates():
    """sqnorm4 exactly on min_norm_squared / max_norm_squared and one float ulp either side, in
    interior and edge columns; points whose w lane alone puts them inside / outside the gate."""
    rows, cols, np_ = 3, 96, 5
    P = wall(rows, cols, x0=8.0)
    lo = [np.array([1, 0, 0, 0], F32), split_yw(ulp_down(1.0)), split_yw(ulp_up(1.0))]
    hi = [np.array([100, 0, 0, 0], F32), np.array([96, 28, 0, 0], F32),          # 9216 + 784 = 1e4
          np.array([100, 0, 0, 2 ** -5], F32),                                   # w alone: 1e4 + 2^-10
          np.array([0.5, 0.5, 0.5, 0.5], F32)]                                   # w alone: 0.75 -> 1
    below_hi = split_yw(ulp_down(1e4), [96.0, 99.0, 99.5, 99.75, 98.0])
    assert [sqn(d) for d in lo] == [1.0, ulp_down(1.0), ulp_up(1.0)]
    assert [sqn(d) for d in hi] == [1e4, 1e4, ulp_up(1e4), 1.0] and sqn(below_hi) == ulp_down(1e4)
    # row 1: interior gate points, 12 columns apart (each out-of-range one dilates +-np)
    pts = lo + hi + [below_hi]
    for i, q in enumerate(pts):
        P[1, 8 + 10 * i] = q
    # row 0 and 2: edge columns only (never dilate: the closed form's clamps)
    for r in (0, 2):
        for c in range(np_):
            P[r, c] = lo[1] if c % 2 else hi[2]
            P[r, cols - 1 - c] = hi[2] if c % 2 else lo[1]
        P[r, np_] = lo[0]
        P[r, cols - np_ - 1] = hi[0]

    def reach(R):
        sq = npr.sqnorm4_f32(R["s4"]).astype(np.float64)
        for r, c, want in [(1, 8, 1.0), (1, 18, ulp_down(1.0)), (1, 28, ulp_up(1.0)), (1, 38, 1e4),
                           (1, 48, 1e4), (1, 58, ulp_up(1e4)), (1, 68, 1.0), (1, 78, ulp_down(1e4)),
                           (0, 5, 1.0), (0, cols - 6, 1e4), (0, 1, ulp_down(1.0)), (0, 0, ulp_up(1e4))]:
            assert sq[r * cols + c] == want, (r, c)
        pv = R["pvalid"].reshape(rows, cols)
        assert pv[1, 8] and not pv[1, 18] and pv[1, 28] and pv[1, 38] and pv[1, 48] and not pv[1, 58]
        assert pv[1, 68] and pv[1, 78]
        xyz = R["s4"][1 * cols + 68].copy()
        xyz[3] = 0
        assert sqn(xyz) < 1.0                        # the w lane alone makes (1, 68) range-valid
        v = R["valid"].reshape(rows, cols)
        assert v[0, np_:2 * np_ + 1].all() and v[0, cols - 2 * np_ - 1:cols - np_].all()  # edges dilate nothing
        assert not v[1, 18 - np_:18 + np_ + 1].any() and not v[1, 58 - np_:58 + np_ + 1].any()

    return Scene("range_gates", params(rows, cols), to_scan(P), reach, "r2 on the range gates")


def w_closest():
    """The w lane alone decides the closest adjacent-row point: the pick's own-azimuth chunk holds
    the xyz-nearest point (large w), a point of another chunk is farther in xyz but nearer in 4
    lanes, so its xyz box bound is far below the seed's 4-lane distance."""
    rows, cols = 3, 128
    P = zigzag(rows, cols)
    P[..., 3] = ((np.arange(cols) % 5) * 0.125)[None, :]
    c = 50
    stamp(P, 1, c, [(0, k / 16, 0, 0) for k in range(1, 6)])
    p = P[1, c]
    for r in (0, 2):
        P[r, :, 0] += 4.0                   # the rest of the adjacent rows is far
        P[r, c] = p + np.array([0, 0, 0.125, 3.0], F32)       # own chunk: xyz 1/64, 4-lane 9 + 1/64
        P[r, 100] = p + np.array([0, 0.5, 0.5, 0.0], F32)      # chunk 3: xyz 1/2, 4-lane 1/2

    def reach(R):
        k = pick_pos(R, 1, c)
        assert R["cprev"][k] == 100 and R["cnext"][k] == 2 * cols + 100
        idx = cols + c
        own = np.array([d2row(R, idx, r)[c] for r in (0, 2)])
        far = np.array([d2row(R, idx, r)[100] for r in (0, 2)])
        xyz = [sqn(np.r_[R["s4"][r * cols + c][:3] - R["s4"][idx][:3], 0]) for r in (0, 2)]
        assert np.all(far < own) and np.all(np.array(xyz) < far)
        assert R["valid"][c] and R["valid"][100]

    return Scene("w_closest", params(rows, cols), to_scan(P), reach, "w lane decides find_closest")


def _radius_offsets(np_, j, inside_ulp=False):
    """Row offsets whose first miss (dist^2 == radius^2 = 1) is at k = j; j > np_: no miss.
    inside_ulp: offset j sits one float ulp inside the radius instead (then the miss is at j + 1)."""
    out = []
    for k in range(1, np_ + 1):
        if k < j:
            out.append(np.array([0, k / 64, 0, 0], F32))
        elif k == j:
            out.append(split_yw(ulp_down(1.0)) if inside_ulp else np.array([0, 1, 0, 0], F32))
        else:
            out.append(np.array([0, 1 + k / 16, 0, 0], F32))
    return out


def radius_scene(np_, js, cols, **kw):
    """One segment per first-miss offset j (and j one ulp inside) in every row; adjacent rows are
    copies shifted by 1/2 in z, so prev / next neighbour counts see the same radius equalities."""
    rows = kw.pop("rows", 3)
    P = zigzag(1, cols)[0]
    P = np.repeat(P[None], rows, 0)
    P[..., 2] = (np.arange(rows) * 0.5)[:, None]
    centres = []
    c = np_ + 2 + (np_ % 2)
    for j in js:
        for ulp in (False, True):
            if ulp and j > np_:
                continue
            c += (c % 2)
            assert c + 2 * np_ + 2 < cols - np_
            for r in range(rows):
                stamp(P, r, c, _radius_offsets(np_, j, ulp))
            centres.append((c, j, ulp))
            c += 2 * np_ + 4
    return P, centres


def radius_eq(np_, js, cols, name, **kw):
    rows = kw.get("rows", 3)
    P, centres = radius_scene(np_, js, cols, **dict(kw))
    prm = params(rows, cols, neighbor_points=np_, num_sectors=1, planar_feats_per_sector=200, **{
        k: v for k, v in kw.items() if k != "rows"})

    def reach(R):
        r2 = R["params"].radius ** 2
        for (c, j, ulp) in centres:
            pick_pos(R, rows // 2, c)
            idx = (rows // 2) * cols + c
            n_plus = len(npr.neighbor_list(R["s4"], idx, np_, r2)) // 2
            want = min(j - 1 + (1 if ulp else 0), np_)
            assert n_plus == want, (c, j, ulp, n_plus)
            if j <= np_:
                d = sqn(R["s4"][idx + j] - R["s4"][idx])
                assert d == (ulp_down(1.0) if ulp else 1.0)

    return Scene(name, prm, to_scan(P), reach, "neighbour dist^2 on the radius")


def min_points_scene(met):
    """Neighbour count exactly min_points (kept) and min_points - 1 (dropped): picks with first miss
    j = 2 have 2 + 2 * 3 = 8 neighbours in the middle row and 2 + 3 = 5 in the first / last row."""
    mp = 8 if met else 9
    rows, cols = 3, 96
    P, centres = radius_scene(5, [2], cols)

    def reach(R):
        for (c, j, ulp) in centres:
            if ulp:
                continue
            k = pick_pos(R, 1, c)
            assert R["count"][k] == 8 and R["keep"][k] == met
            k0 = pick_pos(R, 0, c)
            assert R["count"][k0] == 5 and not R["keep"][k0]

    return Scene(f"min_points_{'met' if met else 'short'}",
                 params(rows, cols, min_points=mp, num_sectors=1), to_scan(P), reach, "n == min_points")


def one_adjacent_row():
    """rows = 2: every pick has exactly one adjacent row (prev for row 1, next for row 0); for
    j = 2 the neighbour count 2 + (1 + 2) lands on min_points = 5 exactly."""
    rows, cols = 2, 96
    P, centres = radius_scene(5, [2, 3], cols, rows=2)

    def reach(R):
        for (c, j, ulp) in centres:
            for r in (0, 1):
                k = pick_pos(R, r, c)
                assert (R["cprev"][k] >= 0) != (R["cnext"][k] >= 0)
                if j == 2 and not ulp:
                    assert R["count"][k] == 5 and R["keep"][k]

    return Scene("one_adjacent_row", params(rows, cols, num_sectors=2), to_scan(P), reach, "rows = 2")


def curv_threshold():
    """Centre curvatures 0.25 - 1 ulp, 0.25 and 0.25 + 1 ulp with planar_threshold = 0.25: the z
    asymmetry e = z(c+1) + z(c+2) of the segment is 0.5 - 2^-27, 0.5 or 0.5 + 2^-26."""
    rows, cols = 3, 128
    P = zigzag(rows, cols)
    P[..., 2] = 0.0
    P[0, :, 2], P[2, :, 2] = -0.5, 0.5
    base = [(0, k / 16, 0, 0) for k in range(1, 6)]
    centres = {}
    for c, (e1, e2), want in [(20, (0.5, -2.0 ** -26), ulp_down(0.25)), (50, (0.5, 0.0), 0.25),
                              (80, (0.5, 2.0 ** -26), ulp_up(0.25)), (110, (0.25, 0.0), 0.0625)]:
        for r in range(rows):
            stamp(P, r, c, base)
            P[r, c + 1, 2] += F32(e1)
            P[r, c + 2, 2] += F32(e2)
        centres[c] = want

    def reach(R):
        for c, want in centres.items():
            assert float(R["curv"][cols + c]) == want, (c, R["curv"][cols + c], want)
            picked = np.any(R["picks"] == cols + c)
            assert picked == (want < 0.25), c

    return Scene("curv_threshold", params(rows, cols, planar_threshold=0.25), to_scan(P), reach,
                 "curvature on the planar threshold")


def curv_ties(name="curv_ties", rows=3, cols=200, **kw):
    """Curvature from a period-7 z pattern on a straight wall: exact ties across sectors, across
    32-candidate walk steps and inside one step within np columns of each other."""
    P = wall(rows, cols)
    c = np.arange(cols)
    P[..., 2] += (((c * c) % 7) / 64.0)[None, :].astype(F32)
    prm = params(rows, cols, **kw)

    def reach(R):
        cv = R["curv"].reshape(rows, cols)[1]
        vals, cnt = np.unique(cv[R["valid"].reshape(rows, cols)[1]], return_counts=True)
        assert cnt.max() >= 32 and len(vals) < 10          # many exact ties
        tied = np.nonzero(cv == vals[cnt.argmax()])[0]
        assert np.any(np.diff(tied) < R["np"])               # tied columns inside one suppression window
        assert len(R["picks"]) > 0

    return Scene(name, prm, to_scan(P), reach, "exact curvature ties")


def curv_zero(name, rows, cols, check=None, **kw):
    """A straight wall (curvature exactly 0 at every valid column): every column ties, so the
    greedy walk takes sector starts, every np columns, and the per-sector cap decides."""
    P = wall(rows, cols, step=1 / 32 if cols > 1024 else 1 / 16)
    prm = params(rows, cols, **kw)

    def reach(R):
        v = R["valid"]
        assert np.all(R["curv"][v] == 0)
        if check:
            check(R)

    return Scene(name, prm, to_scan(P), reach, "all-zero curvature, sector / cap edges")


def _sector_of(R, cols_idx):
    p = R["params"]
    pps = p.num_columns // p.num_sectors
    return np.minimum(cols_idx // pps, p.num_sectors - 1)


def sectors():
    out = []

    def rem(R):      # remainder columns go to the last sector; a pick on a sector's last column
        cols, p = R["cols"], R["params"]
        pps = cols // p.num_sectors
        assert cols % p.num_sectors and (cols - (p.num_sectors - 1) * pps) > pps
        pc = R["picks"] % cols
        assert np.any((pc + 1) % pps == 0)
    out.append(curv_zero("sectors_remainder", 2, 70, rem, num_sectors=6))

    def narrow(R):   # pps < np: one pick suppresses columns of later sectors
        pc = np.sort(R["picks"][R["picks"] < R["cols"]])
        pps = R["cols"] // R["params"].num_sectors
        assert pps < R["np"] and np.all(np.diff(pc) >= R["np"])
        assert len(np.unique(_sector_of(R, pc))) < R["params"].num_sectors - 2
    out.append(curv_zero("sectors_narrow", 2, 64, narrow, num_sectors=24))

    def pps1(R):
        assert R["cols"] // R["params"].num_sectors == 1 and R["params"].num_sectors == 64
    out.append(curv_zero("sectors_pps1_max", 2, 64, pps1, num_sectors=64, neighbor_points=3))
    def max_rem(R):  # 64 sectors of 2 columns, the last one of 4
        assert R["params"].num_sectors == 64 and R["cols"] - 63 * (R["cols"] // 64) == 4
    out.append(curv_zero("sectors_max_remainder", 2, 130, max_rem, num_sectors=64))

    # point picks only (planar threshold 0): a narrow sector's mask is changed only by the point
    # pick of an earlier sector
    def pts(R):
        assert len(R["picks"]) == 0
        q = np.sort(R["qpicks"][R["qpicks"] < R["cols"]])
        assert np.all(np.diff(q) >= R["np"])
        s = _sector_of(R, q)
        # some sector got no pick of its own: every candidate was suppressed from the left
        assert len(np.unique(s)) < R["params"].num_sectors
    out.append(curv_zero("sectors_points_cascade", 2, 64, pts, num_sectors=16, planar_threshold=0.0,
                         point_feats_per_sector=1))
    return out


def capacity():
    out = []

    def zero_cap(R):   # planar_feats_per_sector = 0: the reference's '>' still allows one pick
        per = np.bincount(_sector_of(R, R["picks"] % R["cols"]) + R["params"].num_sectors * (R["picks"] // R["cols"]))
        assert per.max() == 1 and len(R["picks"]) == R["rows"] * R["params"].num_sectors
    out.append(curv_zero("planar_cap_zero", 3, 96, zero_cap, planar_feats_per_sector=0))

    def full(R):       # every column of the middle sector picked: the speculative list is full
        p = R["params"]
        pps = R["cols"] // p.num_sectors
        longest = R["cols"] - (p.num_sectors - 1) * pps
        spec_cap = (longest + R["np"] - 1) // R["np"] + 1
        pc = R["picks"][R["picks"] < R["cols"]]
        n_mid = int(np.sum(_sector_of(R, pc) == 1))
        assert n_mid == spec_cap - 1 == pps // R["np"], (n_mid, spec_cap)
    out.append(curv_zero("planar_spec_full_np1", 3, 96, full, num_sectors=3, neighbor_points=1,
                         planar_feats_per_sector=100))
    out.append(curv_zero("planar_spec_full_np2", 3, 96, full, num_sectors=3, neighbor_points=2,
                         planar_feats_per_sector=100))

    def cap51(R):
        pc = R["picks"][R["picks"] < R["cols"]]
        assert np.bincount(_sector_of(R, pc)).max() == R["params"].planar_feats_per_sector + 1
    out.append(curv_zero("planar_cap_hit_4096", 2, 4096, cap51))

    # unused-list lengths around k * pfps and 31 / 32 / 33: sector s keeps U_s range-valid columns
    for pfps, Us in ((3, (5, 6, 7, 8, 9, 10)), (1, (31, 32, 33, 2, 3, 1)), (4, (31, 32, 33, 7, 8, 9))):
        out.append(_unused_lengths(pfps, Us))
    return out


def _unused_lengths(pfps, Us):
    """Point walks on sectors whose unused lists have exactly the given lengths (planar picks off,
    every other column of the sector's tail out of the range gate - point validity does not dilate)."""
    S, pps = len(Us), 48
    cols = S * pps
    rows = 2
    P = wall(rows, cols)
    for s, U in enumerate(Us):
        a = s * pps
        lo = max(a, 5)
        keep = list(range(lo, lo + U))
        for c in range(a, a + pps):
            if c not in keep:
                P[:, c] = (0, 0, 0, 0)
    prm = params(rows, cols, num_sectors=S, planar_threshold=0.0, point_feats_per_sector=pfps)

    def reach(R):
        pv = R["pvalid"].reshape(rows, cols)[0]
        got = [int(pv[s * pps:(s + 1) * pps].sum()) for s in range(S)]
        assert got == list(Us), got
        assert len(R["qpicks"]) > 0

    return Scene(f"unused_lengths_pfps{pfps}", prm, to_scan(P), reach, "phase-B boundary of the point walk")


def closest_ties():
    """Adjacent-row points at bit-identical dist^2 from a pick: in the pick's own chunk, in a lower
    chunk at the same lane (the in-lane c < bc rule), on both sides of the seed chunk, at columns
    31 / 32, at the last valid column cols - np - 1, and a four-way tie."""
    rows, cols, np_ = 3, 256, 5
    P = zigzag(rows, cols)
    P[0, :, 0] += 32.0
    P[2, :, 0] += 32.0                               # the rest of the adjacent rows is far
    d, h = 1 / 64, 1 / 32
    A = [np.array(v, F32) for v in ((0, d, h, 0), (0, -d, h, 0), (0, h, d, 0), (0, -h, d, 0))]
    # (pick column, adjacent row, columns of its tie points)
    plan = [
        (70, 0, [68, 72]),                  # same chunk
        (110, 0, [78, 110]),                # lower chunk at the seed column's lane
        (150, 0, [118, 182]),               # both sides of the seed chunk, none in it
        (190, 0, [31, 32]),                 # columns 31 / 32
        (230, 0, [200, cols - np_ - 1]),    # the last valid column
        (20, 2, [14, 40, 104, 170]),        # four-way tie over four chunks
    ]
    # row 2 mirrors the row-0 ties (z offset negated)
    plan += [(c, 2, cc) for c, r, cc in plan if r == 0]
    for c in sorted({c for c, _, _ in plan}):
        stamp(P, 1, c, [(0, k / 16, 0, 0) for k in range(1, 6)])
    for c, r, cc in plan:
        p = P[1, c]
        for col, a in zip(cc, A):
            P[r, col] = p + a * np.array([1, 1, 1 if r == 0 else -1, 1], F32)

    def reach(R):
        for c, r, cc in plan:
            k = pick_pos(R, 1, c)
            dd = d2row(R, cols + c, r)
            assert list(np.nonzero(dd == dd.min())[0]) == sorted(cc), (c, r)
            assert (R["cprev"] if r == 0 else R["cnext"])[k] == r * cols + min(cc)

    return Scene("closest_ties", params(rows, cols, num_sectors=2), to_scan(P), reach, "find_closest ties")


def closest_seed_zero():
    """dist^2 == 0: the pick coincides with two adjacent-row points, one in its own chunk and one in
    a lower chunk.  The lower chunk's box bound is 0 == the seed, and (1 - 1e-5) * 0 == 0, so only a
    '<=' pruning test evaluates it; rule R2 then takes the lower column.  Only the lower copy has
    different in-radius neighbours (spanning the plane z = const with the pick's row, where the
    seed-chunk copy's span x = const), so the choice also shows in the normal, which is what the
    batched runs compare."""
    rows, cols = 3, 160
    P = zigzag(rows, cols)
    P[0, :, 0] += 32.0
    P[2, :, 0] += 32.0
    cs = [(100, 40), (140, 12), (60, 28)]
    for c, lower in cs:
        stamp(P, 1, c, [(0, k / 16, 0, 0) for k in range(1, 6)])
        for r in (0, 2):
            P[r, c] = P[1, c]
            P[r, lower] = P[1, c]
            for k in (1, 2):
                # the lower copy spans the plane z = p.z with the own row, the seed-chunk copy x = p.x
                P[r, lower + k] = P[1, c] + np.array([k / 16, 0, 0, 0], F32)
                P[r, lower - k] = P[1, c] - np.array([k / 16, 0, 0, 0], F32)
                P[r, c + k] = P[1, c] + np.array([0, 0, k / 16, 0], F32)
                P[r, c - k] = P[1, c] - np.array([0, 0, k / 16, 0], F32)

    def reach(R):
        for c, lower in cs:
            k = pick_pos(R, 1, c)
            assert (c >> 5) != (lower >> 5)
            assert R["cprev"][k] == lower and R["cnext"][k] == 2 * cols + lower
            assert d2row(R, cols + c, 0)[c] == 0.0
            assert R["count"][k] == 2 * (1 + 4) + 10, R["count"][k]   # own row 10, each adjacent row 1 + 4
            p = R["params"]
            ok, n, _ = npr.normal_f64(R["s4"], R["valid"], cols + c, rows, cols, p.neighbor_points, p.radius,
                                      p.min_points)
            assert ok and abs(n[2]) > 0.999, n

    return Scene("closest_seed_zero", params(rows, cols, num_sectors=1), to_scan(P), reach,
                 "box bound == seed == 0")


def closest_fallback():
    """No valid adjacent-row point at the pick's azimuth: the seed is the chunk of least box
    distance, here a tie between the chunks on either side (the lower one must be taken).  Row 2
    has no valid point at all."""
    rows, cols, np_ = 3, 160, 5
    P = zigzag(rows, cols)
    P[0, :, 1] += F32(1 / 32)                   # half a column step: the boxes tie exactly
    P[0, :, 2] = 0.125
    w = 2
    c = 32 * w + 16
    stamp(P, 1, c, [(0, k / 16, 0, 0) for k in range(1, 6)])
    P[1, :, 2] = 0.0
    P[0, 32 * w:32 * w + 32] = 0.0                # out of range -> the whole chunk (and +-np) invalid
    P[2] = 0.0

    def reach(R):
        k = pick_pos(R, 1, c)
        v0 = R["valid"].reshape(rows, cols)[0]
        assert not v0[32 * w:32 * w + 32].any() and not R["valid"].reshape(rows, cols)[2].any()
        assert R["cnext"][k] == -1
        p = R["s4"][cols + c]
        box = []
        for ww in (w - 1, w + 1):
            sel = np.nonzero(v0[32 * ww:32 * ww + 32])[0] + 32 * ww
            q = R["s4"][sel, :3]
            lo, hi = q.min(0), q.max(0)
            dd = np.maximum(np.maximum(lo - p[:3], p[:3] - hi), 0).astype(F32)
            box.append(F32(F32(dd[0] * dd[0] + dd[1] * dd[1]) + dd[2] * dd[2]))
        assert box[0] == box[1], box
        assert R["cprev"][k] == 32 * w - np_ - 1

    return Scene("closest_fallback", params(rows, cols, num_sectors=1), to_scan(P), reach,
                 "fallback seed, box tie; no valid row")


def far_ulps():
    """Picks 64-72 m out whose adjacent-row candidates sit a few ulp apart (groups of 6 columns at
    nearly one position, some straddling a 32-column chunk border): the float dist^2 of the
    reference and the box bound round most differently here."""
    rows, cols = 3, 192
    rng = np.random.default_rng(12)
    P = wall(rows, cols, x0=64.0)
    P[..., 2] = 0.0
    for r in (0, 2):
        g = (np.arange(cols) // 6) * 6 + 3
        P[r, :, 1] = (g - cols // 2) / 16
        P[r, :, 2] = F32(2.0 ** -10 if r == 0 else -2.0 ** -10)
        for lane in (0, 1):
            ulp = np.spacing(P[r, :, lane]).astype(F32)
            P[r, :, lane] = (P[r, :, lane] + rng.integers(-3, 4, cols) * ulp).astype(F32)

    def reach(R):
        assert len(R["picks"]) > 10
        close = 0
        for k, idx in enumerate(R["picks"].tolist()):
            if idx // cols != 1:
                continue
            dd = np.sort(d2row(R, idx, 0))
            if np.isfinite(dd[1]) and dd[1] - dd[0] <= 8 * np.spacing(F32(dd[0])):
                close += 1
        assert close >= 3, close

    return Scene("far_ulps", params(rows, cols, num_sectors=2), to_scan(P), reach, "ulp-level candidates far out")


def degenerate_covariances():
    """compute_normal on rank-0 / rank-1 / repeated-eigenvalue / isotropic covariances."""
    out = []
    # zero covariance: every point of every row is the same point
    P = np.zeros((3, 32, 4), F32)
    P[...] = (8, 1, 0.5, 0)

    def zero(R):
        assert len(R["picks"]) > 0 and R["keep"].all()
        assert all(max(abs(x) for x in cov_f32(R["s4"], i, nb)) == 0 for i, nb in zip(R["picks"], R["nbrs"]))
        assert np.all(R["cprev"][R["cprev"] >= 0] % 32 == 5)        # dist^2 0 everywhere: lowest valid column
    out.append(Scene("cov_zero", params(3, 32, num_sectors=2), to_scan(P), zero, "scale == 0"))

    # rank 1: every point on one line (adjacent rows shifted half a step along it)
    P = wall(3, 64)
    P[..., 2] = 0.0
    P[0, :, 1] += F32(1 / 32)
    P[2, :, 1] -= F32(1 / 32)

    def rank1(R):
        assert R["keep"].any()
        for i, nb in zip(R["picks"], R["nbrs"]):
            c = cov_f32(R["s4"], i, nb)
            assert c[0] == c[1] == c[3] == c[4] == c[5] == 0 and c[2] > 0
    out.append(Scene("cov_rank1", params(3, 64), to_scan(P), rank1, "collinear neighbours"))

    # repeated in-plane eigenvalue (np = 1): own row +-s along y, adjacent rows +-s in z
    s = 0.25
    P = zigzag(3, 48)
    P[..., 0] = 8.0
    P[..., 1] = ((np.arange(48) - 24) * s)[None, :]
    P[..., 2] = np.array([-s, 0, s], F32)[:, None]

    def repeated(R):
        k = pick_pos(R, 1, 20)
        c = cov_f32(R["s4"], R["picks"][k], R["nbrs"][k])
        assert c[2] == c[5] > 0 and c[0] == c[1] == c[3] == c[4] == 0, c
    out.append(Scene("cov_repeated", params(3, 48, neighbor_points=1, num_sectors=1), to_scan(P), repeated,
                     "repeated in-plane eigenvalue, m20 == 0"))

    # isotropic (np = 2): own row +-s, +-2s along y; adjacent rows hold p + (s, 0, s) and
    # p + (s, 0, -s) at the pick's column and, with w = 1/4 (farther in 4 lanes, the same in xyz),
    # at +-1 and +-2 columns: diag(10 s^2) / n^2 in exact arithmetic
    P = zigzag(3, 64)
    cs = [20, 40]
    for c in cs:
        stamp(P, 1, c, [(0, s, 0, 0), (0, 2 * s, 0, 0)])
        p = P[1, c]
        for r, sg in ((0, 1), (2, -1)):
            P[r, c - 2:c + 3] = p + np.array([s, 0, sg * s, 0.25], F32)
            P[r, c] = p + np.array([s, 0, sg * s, 0], F32)

    def iso(R):
        for c in cs:
            k = pick_pos(R, 1, c)
            A = np.array(R["nbrs"][k], np.float64)[:, :3] - R["s4"][cols_iso + c][:3]
            w = np.linalg.eigvalsh(A.T @ A)
            assert len(R["nbrs"][k]) == 14 and np.ptp(w) == 0.0, w
    cols_iso = 64
    out.append(Scene("cov_isotropic", params(3, 64, neighbor_points=2, num_sectors=1), to_scan(P), iso,
                     "three equal eigenvalues"))
    return out


def m20_flt_min():
    """(m20 / scale)^2 below, exactly at and above FLT_MIN = 2^-126, and subnormal z offsets.
    np = 1, rows = 3: n = 8 neighbours, own row +-1/2 along x, adjacent rows +-1/4 in y; one own-row
    neighbour carries z = 3 * 2^-e, so c20 = 3 * 2^-e * 2^-7, scale = c00 = 6 * 2^-8 and m20 = 2^-e
    exactly: e = 63 puts v1norm2 on FLT_MIN, 62 above, 64 below; 1e-30 and the subnormal 2^-140
    are further below."""
    rows, cols = 3, 64
    P = np.zeros((rows, cols, 4), F32)
    P[..., 0] = (4.0 + np.arange(cols) * 0.5)[None, :]
    P[..., 1] = np.array([0.25, 0.0, -0.25], F32)[:, None]
    bumps = {10: 3 * 2.0 ** -62, 20: 3 * 2.0 ** -63, 30: 3 * 2.0 ** -64, 40: 1e-30, 50: 2.0 ** -140}
    for c, e in bumps.items():
        P[1, c + 1, 2] = F32(e)

    def reach(R):
        got = {}
        for k, idx in enumerate(R["picks"].tolist()):
            if idx // cols == 1 and idx % cols in bumps:
                c = cov_f32(R["s4"], idx, R["nbrs"][k])
                got[idx % cols] = float(v1norm2(c)[0])
                assert R["count"][k] == 8
        assert got[10] > FLT_MIN and got[20] == FLT_MIN and got[30] < FLT_MIN and 0 < got[30], got
        assert got[40] < FLT_MIN
        assert 0 < R["s4"][cols + 51][2] < FLT_MIN          # a subnormal coordinate of a valid point
        assert R["valid"][cols + 51]

    return Scene("m20_flt_min", params(rows, cols, neighbor_points=1, num_sectors=1, planar_feats_per_sector=100),
                 to_scan(P), reach, "v1norm2 vs FLT_MIN; subnormal coordinates")


def shapes():
    out = []
    for rows, cols, np_ in ((3, 11, 5), (2, 31, 5), (3, 32, 5), (1, 33, 5), (3, 65, 5), (2, 3, 1), (3, 33, 16)):
        def check(R, rows=rows, cols=cols, np_=np_):
            assert R["rows"] == rows and R["cols"] == cols
            assert R["valid"].reshape(rows, cols)[:, np_:cols - np_].any()
        out.append(_bumpy(f"shape_{rows}x{cols}_np{np_}", rows, cols, check, neighbor_points=np_,
                          num_sectors=1 if cols < 40 else 2))
    out.append(_bumpy("shape_3x4096", 3, 4096, None, num_sectors=6))
    return out


def _bumpy(name, rows, cols, check=None, **kw):
    """A wall with a period-7 z pattern at gentle amplitude: many exact curvature ties, planar picks
    that keep their normals."""
    P = wall(rows, cols, step=1 / 32 if cols > 1024 else 1 / 16)
    c = np.arange(cols)
    P[..., 2] += (((c * c) % 7) / 256.0)[None, :].astype(F32)
    prm = params(rows, cols, **kw)

    def reach(R):
        assert R["valid"].any()
        if check:
            check(R)

    return Scene(name, prm, to_scan(P), reach, "shape edge")


def all_scenes():
    out = [range_gates(), w_closest(),
           radius_eq(1, [1, 2], 64, "radius_np1"),
           radius_eq(5, [1, 2, 3, 4, 5, 6], 256, "radius_np5"),
           radius_eq(16, [1, 2, 8, 15, 16, 17], 512, "radius_np16"),
           min_points_scene(True), min_points_scene(False), one_adjacent_row(),
           curv_threshold(), curv_ties(), curv_ties("curv_ties_sectors", 3, 400, num_sectors=5),
           closest_ties(), closest_seed_zero(), closest_fallback(), far_ulps(), m20_flt_min()]
    out += degenerate_covariances() + sectors() + capacity() + shapes()
    names = [s.name for s in out]
    assert len(names) == len(set(names)), names
    return out
