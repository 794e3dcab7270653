"""Workload for compute-sanitizer (profiles/sanitize.sh): a batched replay of three short VLP-16
sequences (every batched kernel incl. the ticketed moment merge and the cached evaluation)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def main():
    from form_b200 import _capi, synth
    from form_b200.pipeline import BatchReplay, Estimator

    sensor, n = "vlp-16", 6
    rows, cols = synth.shape(sensor)
    p = _capi.default_est_params(rows, cols, record_trace=1, max_num_recent_scans=3)
    runs = []
    for seq in (0, 1, 2):
        scans = [synth.scan(sensor, seq, k) for k in range(n)]
        est = Estimator(p)
        for s in scans:
            est.register_scan(s)
        runs.append((est, scans))
    host_ptrs = [[s.ctypes.data for s in scans] for _, scans in runs]
    br = BatchReplay([est.trace() for est, _ in runs], p)
    br.run(0, n, host_ptrs, on_device=False)
    st = br.stats()
    assert st["scans"] == 3 * n and st["lin_pairs"] > 0
    br.close()
    print("probe ok")


if __name__ == "__main__":
    main()
