"""Wide-key join over N ranks: the config-2 query (filter + equi-join + 3 checksums) with join keys
offset by 2^40, every relation row-sharded (QCE_REPLICATE_BYTES=0), against the same query on keys
below 2^32 and, optionally, another build of the project (e.g. the commit before the wide exchange,
which gathers wide joins on rank 0).

Each arm runs the driver binary twice on the same relation files: once loading only, once loading and
running the query `--steps` times; (difference / steps) is the time of one query step, host clock
around a run that ends with its results printed.  Tuples received per rank come from the engine's
QCE_TRACE join lines (builds that print them).  Every arm's stdout is checked against the FK->PK
closed forms of the workload.

  python tools/wide_join_scale.py --ranks 1 2 4 8 --rows 10000000 --steps 5 [--other-build DIR] --out profiles/x.json
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import workload as wl  # noqa: E402

OFF = 1 << 40
TRACE = re.compile(r"\[qce\] join rank (\d+)/(\d+): route=(\w+) keys=(\w+) width=(\d+) recv R=(\d+)/(\d+) S=(\d+)/(\d+)")
QUERY = "0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2\n"


def gen_db(n, offset, seed=1):
    """FK->PK: R0.c1 uniform over R1's keys, R1.c1 a permutation (every FK matches once)"""
    rng = np.random.default_rng(seed)
    pk = rng.permutation(n).astype(np.uint64)
    fk = rng.integers(0, n, n, dtype=np.uint64)
    f0 = rng.integers(0, 10 ** 6, n, dtype=np.uint64)
    f1 = rng.integers(0, 10 ** 6, n, dtype=np.uint64)
    r0 = [np.arange(n, dtype=np.uint64), fk + np.uint64(offset), f0]
    r1 = [np.arange(n, dtype=np.uint64), pk + np.uint64(offset), f1]
    return [r0, r1]


def closed_form(db):
    """what the query prints, from the FK->PK structure (no join needed)"""
    r0, r1 = db
    keep = r0[2] > 500000
    pos = np.empty(len(r1[1]), dtype=np.int64)
    pos[(r1[1] - r1[1].min()).astype(np.int64)] = np.arange(len(r1[1]))
    m = pos[(r0[1][keep] - r1[1].min()).astype(np.int64)]
    sums = [int(r0[0][keep].sum(dtype=np.uint64)), int(r1[0][m].sum(dtype=np.uint64)), int(r1[2][m].sum(dtype=np.uint64))]
    return " ".join(str(s) if int(keep.sum()) else "NULL" for s in sums) + " \n"


def run(binary, paths, text, env):
    t = time.perf_counter()
    p = subprocess.run([binary], input=("".join(x + "\n" for x in paths) + "Done\n" + text).encode(),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env, timeout=3600)
    return time.perf_counter() - t, p.stdout.decode(), p.stderr.decode(), p.returncode


def arm(binary, paths, ranks, steps, want):
    env = dict(os.environ, QCE_GPUS=str(ranks), QCE_REPLICATE_BYTES="0", QCE_TRACE="1", QCE_COMM_TIMEOUT_S="600")
    t_load, _, _, rc0 = run(binary, paths, "", env)
    t_all, out, err, rc = run(binary, paths, QUERY * steps, env)
    res = {"rc": rc, "ms_per_step": 1e3 * (t_all - t_load) / steps if rc == 0 and rc0 == 0 else None,
           "load_s": round(t_load, 2), "correct": rc == 0 and out == want * steps}
    joins = [m.groups() for m in TRACE.finditer(err)]
    if joins:
        last = joins[-ranks:]
        res["route"] = sorted({j[2] for j in last})
        res["keys"] = sorted({j[3] for j in last})
        res["recv_per_rank"] = [[int(j[5]), int(j[7])] for j in sorted(last, key=lambda j: int(j[0]))]
        res["total_per_side"] = [int(last[0][6]), int(last[0][8])]
    if rc != 0:
        res["stderr_tail"] = err[-600:]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--rows", type=int, default=10_000_000, help="rows per relation per rank")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--other-build", default=None, help="package directory of another build to run as well")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    this = os.path.join(ROOT, "query-compiler-executor_b200", "build", "queries")
    builds = {"this": this}
    if args.other_build:
        builds["other"] = os.path.join(args.other_build, "build", "queries")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         stderr=subprocess.DEVNULL).stdout.decode().strip()
    report = {"gpu": smi, "rows_per_rank": args.rows, "steps": args.steps, "query": QUERY.strip(), "runs": []}
    for ranks in args.ranks:
        n = ranks * args.rows
        for keys, offset in (("wide", OFF), ("packed", 0)):
            db = gen_db(n, offset)
            want = closed_form(db)
            d = tempfile.mkdtemp()
            paths = wl.write_db(d, db)
            del db
            for name, binary in builds.items():
                r = arm(binary, paths, ranks, args.steps, want)
                r.update({"ranks": ranks, "keys": keys, "build": name})
                report["runs"].append(r)
                print(json.dumps(r), flush=True)
            subprocess.run(["rm", "-rf", d])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(report, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
