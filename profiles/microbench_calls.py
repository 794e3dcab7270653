"""Wall-clock cost of single hot-path calls (linearize / associate / extract) on a warm
context, to separate launch + latency floors from kernel work.  Run on a GPU box."""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from form_b200 import _capi, synth  # noqa: E402
from form_b200.context import Context  # noqa: E402
from helpers import gt, perturbed, scan_poses  # noqa: E402


def main():
    sensor = "os0-128"
    rows, cols = synth.shape(sensor)
    params = _capi.default_params(rows, cols)
    rng = np.random.default_rng(0)
    n_scans = int(os.environ.get("N_SCANS", "12"))
    with Context(params) as ctx:
        est = {}
        for k in range(n_scans):
            scan = synth.scan(sensor, 0, k)
            ctx.extract(scan, k)
            est[k] = perturbed(gt(0, k), rng, 0.0005, 0.005)
            poses = scan_poses(list(range(k + 1)), [est[s] for s in range(k + 1)])
            ctx.map_rebuild(poses)
            counts = ctx.associate(est[k])
            ctx.commit_scan()
        k = n_scans - 1
        pairs = np.zeros(len(counts), dtype=_capi.PAIR)
        pairs["i"], pairs["j"] = counts["i"], k
        allpairs = np.array([(i, j) for j in range(n_scans) for i in range(j)], dtype=_capi.PAIR)
        ncorr = int(counts["n_planar"].sum() + counts["n_point"].sum())

        def timeit(fn, n=300):
            fn()
            ctx.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            return (time.perf_counter() - t0) / n * 1e6

        print(f"pairs of current scan: {len(pairs)}, correspondences {ncorr}; window pairs {len(allpairs)}")
        print(f"linearize(cur scan)  {timeit(lambda: ctx.linearize(pairs, poses)):7.2f} us")
        print(f"linearize(window)    {timeit(lambda: ctx.linearize(allpairs, poses), 100):7.2f} us")
        print(f"error(cur scan)      {timeit(lambda: ctx.error(pairs, poses)):7.2f} us")
        print(f"associate            {timeit(lambda: ctx.associate(est[k]), 100):7.2f} us")
        print(f"map_rebuild          {timeit(lambda: ctx.map_rebuild(poses), 100):7.2f} us")
        scan = synth.scan(sensor, 0, k)
        print(f"extract (host bufs)  {timeit(lambda: ctx.extract(scan, k), 50):7.2f} us")
        print(f"synchronize (empty)  {timeit(lambda: ctx.synchronize()):7.2f} us")


if __name__ == "__main__":
    main()
