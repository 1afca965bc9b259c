"""Time the tuple sort and one query on runs above 2^30 tuples (the ground between the MSD route's limit and the
reference's int limit of 2^31 - 1 tuples).

usage: python tools/big_run_bench.py [out.json]

  * the packed sort of a whole base column at 2^30 + 1 and 2^31 - 1 rows, uniform 32-bit keys (4 one-sweep passes);
  * the wide (key >= 2^32, key / row-id) sort at 2^30 + 1 rows, 40-bit keys (5 passes);
  * the end-to-end 2-way join of tests/test_gpu_big_runs.py through qce_host_run_batch (1.2 G rows, 1.1 G past the
    filter), checked against its closed form.

Every shape is run once as warm-up, then REPS times.  Sort times are device events: the engine's launch profile
(qce_profile_json) around each kernel of the sort, summed; `wall_ms` is a host clock around qce_sort_tuples and a
device synchronise.  Rates count 16 B per tuple per pass (24 B wide) over the one-sweep passes' time, and are also
given as a fraction of the 6544 GB/s copy rate DESIGN.md uses as the bandwidth roof.  Inputs are far larger than L2.
Prints one JSON object (and writes it to out.json when given), with the card's name and power limit."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import qce_b200  # noqa: E402
from tests import test_gpu_big_runs as big  # noqa: E402

REPS = 3
ROOF_GBPS = 6544.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def time_sort(e, kind, n):
    big.upload(e, torch, 70, 0, n, big.gen_t(torch, kind))
    per_pass_bytes = 24 if kind == "wide" else 16
    tag = "onesweep_kv" if kind == "wide" else "onesweep_k"
    rows = []
    for rep in range(REPS + 1):  # the first is the warm-up
        t = e.build_tuples(70, 0)
        e.sync()
        e.profile(True)
        t0 = time.perf_counter()
        e.sort_tuples(t)
        e.sync()
        wall = (time.perf_counter() - t0) * 1e3
        prof = e.profile_read()
        e.profile(False)
        if rep == 0:
            ok = e.is_sorted(t)
        e.tuples_free(t)
        if rep:
            kern = {k: v for k, v in prof.items() if not k.startswith("gap_before:")}
            rows.append({"wall_ms": wall, "kernel_ms": sum(v["ms"] for v in kern.values()),
                         "onesweep_ms": prof[tag]["ms"], "passes": prof[tag]["launches"],
                         "hist_ms": prof["radix_hist"]["ms"]})
    e.drop_relations()
    best = sorted(rows, key=lambda r: r["onesweep_ms"])[len(rows) // 2]  # the median rep
    gbps = per_pass_bytes * n * best["passes"] / best["onesweep_ms"] / 1e6
    return {"case": "%s_sort" % kind, "n": n, "sorted": ok, **best, "onesweep_ms_per_pass": best["onesweep_ms"] / best["passes"],
            "onesweep_GBps": gbps, "onesweep_frac_of_roof": gbps / ROOF_GBPS,
            "reps_onesweep_ms": [r["onesweep_ms"] for r in rows]}


def time_e2e():
    """in a fresh process: the Rig holds its own engine"""
    code = r"""
import json, sys, time
sys.path.insert(0, %r)
import torch, bench
from tests import test_gpu_big_runs as big
rig = bench.Rig(torch, None, 0, 1, 0)
cols = big.e2e_columns(torch)
for (rel, col), (rows, fn) in cols.items():
    rig.upload_fn(rel, col, rows, lambda b, c, fn=fn: big.dev_column(torch, c, lambda i: fn(i + b)))
torch.cuda.empty_cache()
q, want = big.E2E_QUERIES[0], big.e2e_expected(torch, cols)[0]
torch.cuda.empty_cache()
ms = []
for rep in range(%d + 1):
    t0 = time.perf_counter()
    got = rig.run(q)
    ms.append((time.perf_counter() - t0) * 1e3)
    assert got == want, (got, want)
print(json.dumps({"case": "e2e_join", "query": q.strip(), "rows": big.E2E_N0, "past_filter": big.E2E_N0 - big.E2E_C - 1,
                  "first_ms": ms[0], "reps_ms": ms[1:], "ms": sorted(ms[1:])[len(ms[1:]) // 2]}))
""" % (ROOT, REPS)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200)
    if p.returncode != 0:
        raise RuntimeError(p.stderr[-3000:])
    return json.loads(p.stdout.strip().splitlines()[-1])


def main():
    out = {"card": card(), "roof_GBps": ROOF_GBPS, "reps": REPS, "results": []}
    e = qce_b200.Engine()
    for kind, n in (("u32", big.N30 + 1), ("u32", big.N31), ("wide", big.N30 + 1)):
        out["results"].append(time_sort(e, kind, n))
        print(json.dumps(out["results"][-1]), flush=True)
    del e
    out["results"].append(time_e2e())
    print(json.dumps(out))
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
