"""The adversarial stage-2 windows of assoc_scenes.py on the CPU: (1) every scene reaches the edge it
exists for - exact ties decided by shift rank, by scan id (also between ids equal in their low 40
bits) and by k, coordinates on which the voxel key's fast path would be wrong, distances exactly on
the two gates, bucket sizes on the kernels' layout edges, queries without a neighbour - so a later
edit of a scene cannot silently lose its purpose; (2) the oracle's matches, pair counts and novel
counts equal the independent numpy restatement of rule R5 on every checked query."""
import numpy as np
import pytest

import assoc_scenes as A

SCENES = {s.name: s for s in A.all_scenes()}


def _stats(name):
    sc = SCENES[name]
    _, exp = A.oracle_run(sc)
    p = sc.make_params()
    max2, min2 = p.max_dist_matching ** 2, p.min_dist_map ** 2
    st = dict(tie_rank=0, tie_scan=0, tie_k=0, tie_hi40=0, no_neighbour=0, eq_max=0, eq_min=0,
              fast_path=0, face_tie=0, empty_own=0, sizes=set())
    for e in exp:
        for ty in e["types"]:
            bf = ty["bf"]
            for k in ("tie_rank", "tie_scan", "tie_k", "tie_hi40"):
                st[k] += int(bf[k].sum())
            st["no_neighbour"] += int((~bf["found"]).sum())
            st["eq_max"] += int((bf["found"] & (bf["dist_sqrd"] == max2)).sum())
            st["eq_min"] += int((bf["found"] & (bf["dist_sqrd"] == min2)).sum())
            st["empty_own"] += int((ty["own_empty"] & bf["found"]).sum())
            w = sc.width
            for v in (ty["map_xyz"].reshape(-1), ty["query_xyz"].reshape(-1)):
                st["fast_path"] += int(np.count_nonzero(np.floor(v * (1.0 / w)) != np.floor(v / w)))
            q = ty["query_xyz"]
            off = np.any(np.floor(q * (1.0 / w)) != np.floor(q / w), axis=1)
            st["face_tie"] += int(np.count_nonzero(off & bf["tie_rank"]))
            st["sizes"] |= set(int(n) for n in ty["sizes"])
    return st


COVERAGE = {
    # scene: what it must reach (minimum counts; "sizes": bucket sizes that must occur)
    "lattice_w0.5": dict(tie_rank=500, tie_scan=500, tie_k=100, no_neighbour=1),
    "lattice_w1.0": dict(tie_rank=200, tie_k=100),
    "duplicates": dict(tie_scan=1000, tie_rank=100, tie_k=100),
    "dup_shift": dict(tie_scan=1000, tie_rank=100),
    "dup_rows": dict(tie_k=300, tie_scan=1000),
    "large_ids": dict(tie_scan=1000, tie_hi40=1000),
    # face_tie: queries whose voxel only the division gets right, with an exact tie across shift ranks
    "face_aligned": dict(fast_path=100, face_tie=100),
    "gates": dict(eq_max=100, eq_min=100, tie_rank=100),
    "far_w0.5": dict(tie_rank=500, tie_scan=500),
    "far_w1.0": dict(tie_rank=500, tie_scan=500),
    "sparse": dict(no_neighbour=1000, empty_own=5),
    "buckets_19": dict(sizes={15, 16, 17, 64, 65}),
    "huge_bucket": dict(max_size=65536),
}


@pytest.mark.parametrize("name", sorted(COVERAGE))
def test_scene_reaches_its_edge(name):
    st = _stats(name)
    for key, want in COVERAGE[name].items():
        if key == "sizes":
            assert want <= st["sizes"], (name, sorted(want - st["sizes"]))
        elif key == "max_size":
            assert max(st["sizes"]) >= want, (name, max(st["sizes"]))
        else:
            assert st[key] >= want, (name, key, st[key], want)


def test_sparse_map_is_sparse():
    _, exp = A.oracle_run(SCENES["sparse"])
    assert 0 < len(exp[-1]["types"][0]["map_xyz"]) + len(exp[-1]["types"][1]["map_xyz"]) < 100


@pytest.mark.parametrize("name", sorted(SCENES))
def test_oracle_matches_independent_r5(name):
    """Matches (found, scan, k, dist^2 bits) on every checked query; pair counts by scan id and the
    novel count against the numpy gates (dist^2 < max^2 pairs, dist^2 > min^2 novel)."""
    sc = SCENES[name]
    recs, exp = A.oracle_run(sc)
    assoc = [r for op, r in zip(sc.ops, recs) if op[0] == "associate"]
    commits = {i: r for i, (op, r) in enumerate(zip(sc.ops, recs)) if op[0] == "commit"}
    assert len(assoc) == len(exp)
    for n, ((counts, m0, m1), e) in enumerate(zip(assoc, exp)):
        for t, m in enumerate((m0, m1)):
            ty = e["types"][t]
            bf, idx = ty["bf"], ty["idx"]
            assert len(m) == ty["n_query"]
            got = m[idx]
            where = f"{name} association {n} type {t}"
            assert np.array_equal(got["found"].astype(bool), bf["found"]), where
            assert np.array_equal(got["scan"], bf["scan"]), where
            assert np.array_equal(got["k"], bf["k"]), where
            assert np.array_equal(got["dist_sqrd"].view(np.uint64), bf["dist_sqrd"].view(np.uint64)), where
        # pair counts of every type that had queries: the numpy gate (dist^2 < max^2) over the
        # brute force (every query) or, for sampled scenes, over the oracle's own matches (checked
        # against the brute force on the sample above)
        max2 = sc.make_params().max_dist_matching ** 2
        got_counts = {int(c["i"]): (int(c["n_planar"]), int(c["n_point"])) for c in counts}
        for t, m in enumerate((m0, m1)):
            if not len(m):
                continue  # Matcher::match returns early: the type's counts are stale
            if "counts" in e:
                want = {i: c[t] for i, c in e["counts"].items() if c[t]}
            else:
                pair = m["found"].astype(bool) & (m["dist_sqrd"] < max2)
                want = {int(i): int(k) for i, k in zip(*np.unique(m["scan"][pair], return_counts=True))}
            got = {i: c[t] for i, c in got_counts.items() if c[t]}
            assert got == want, (name, n, t)
    # the commit after the last association of a scan adds the numpy novel count
    last = None
    for i, op in enumerate(sc.ops):
        if op[0] == "associate":
            last = sum(1 for o in sc.ops[: i + 1] if o[0] == "associate") - 1
        elif op[0] == "commit" and "novel" in exp[last]:
            assert tuple(commits[i][0]) == tuple(exp[last]["novel"]), (name, i)
