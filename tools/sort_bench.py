"""Time the LSD one-sweep pass (k_onesweep) and its digit histogram (k_radix_hist) on one packed sort.

usage: python tools/sort_bench.py [rows, default 1e8]

The run is built from a column of `rows` uniform keys below `rows` and sorted with the MSD route turned off
(QCE_MSD=0), so every one of its digits takes a one-sweep pass.  Prints one JSON line: ms per pass, the pass's
rate over its 16 B per tuple, and k_radix_hist's ms per sort, each from the launch profile of three sorts after two
warm-up sorts.  `ok` also checks a 300001-tuple sort against numpy's stable argsort."""
import json
import os
import sys

os.environ["QCE_MSD"] = "0"  # read by the engine at its first sort
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import qce_b200  # noqa: E402

n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
e = qce_b200.Engine()
rng = np.random.default_rng(1)
col = rng.integers(0, n, n, dtype=np.uint64)
e.upload_column(0, 0, col)
small = rng.integers(0, 1 << 27, 300001, dtype=np.uint64)
t = e.tuples_from_host(small, np.arange(len(small), dtype=np.uint64))
e.sort_tuples(t)
k, p = e.tuples_to_host(t)
o = np.argsort(small, kind="stable")
ok = bool((k == small[o]).all() and (p == o.astype(np.uint64)).all())
e.tuples_free(t)
for _ in range(2):
    t = e.build_tuples(0, 0)
    e.sort_tuples(t)
    e.tuples_free(t)
e.profile(True)
for _ in range(3):
    t = e.build_tuples(0, 0)
    e.sort_tuples(t)
    ok = ok and e.is_sorted(t)
    e.tuples_free(t)
prof = e.profile_read()
e.profile(False)
ms = prof["onesweep_k"]["ms"] / prof["onesweep_k"]["launches"]
print(json.dumps({"rows": n, "ok": ok, "passes_per_sort": prof["onesweep_k"]["launches"] // 3, "ms_per_pass": ms,
                  "GBps": 16.0 * n / ms / 1e6, "hist_ms": prof["radix_hist"]["ms"] / 3}))
