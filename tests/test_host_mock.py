"""CPU: the C host operator layer (parser, arranger, the join-kind state machine,
update_mid_results, print_sums -- query-compiler-executor_b200/src/*.c) linked against
tests/c/mock_engine.c, a plain-C stand-in for the C-ABI calls it makes.  This is how the
host logic is held to the reference's recorded outputs WITHOUT a GPU, and fuzzed under
ASan/UBSan.  The mock is test infrastructure: the product never links it (the same host
objects against libqce_b200.so are tested on the GPU in tests/test_gpu_queries.py)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import qce_oracle as orc
from oracle import workload as wl
from tests.helpers import PKG, ROOT, load_db, load_json, run_queries_bin

OUT = os.path.join(ROOT, "tests", "c", "build")
SOURCES = [os.path.join(PKG, "main", "queries_driver.c"), os.path.join(ROOT, "tests", "c", "mock_engine.c")] + \
    sorted(os.path.join(PKG, "src", f) for f in os.listdir(os.path.join(PKG, "src")) if f.endswith(".c"))
# a header change rebuilds the mocks too
HEADERS = [os.path.join(ROOT, "include", "qce_b200.h")] + \
    sorted(os.path.join(PKG, "src", f) for f in os.listdir(os.path.join(PKG, "src")) if f.endswith(".h"))


def _build(name, flags):
    os.makedirs(OUT, exist_ok=True)
    exe = os.path.join(OUT, name)
    newest = max(os.path.getmtime(s) for s in SOURCES + HEADERS)
    if not os.path.exists(exe) or os.path.getmtime(exe) < newest:
        subprocess.run(["gcc", "-g", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(PKG, "src"),
                        "-o", exe] + flags + SOURCES + ["-lpthread"], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return exe


@pytest.fixture(scope="module")
def mock_bin():
    return _build("queries_mock", ["-O1"])


@pytest.fixture(scope="module")
def asan_bin():
    return _build("queries_mock_asan", ["-O1", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"])


def _paths(db):
    return wl.write_db(tempfile.mkdtemp(), db)


@pytest.mark.parametrize("db_name,batch", [("ops_db.npz", "ops.json"), ("small_db.npz", "small_batch.json"),
                                           ("edge_db.npz", "edge.json")])
def test_host_layer_reproduces_recorded_reference_stdout(mock_bin, db_name, batch):
    """Every PDQ query the reference's stdout was recorded for: PDQ-T must match byte for byte,
    PDQ-D must match or be refused; queries on which the reference aborts must abort the same
    way with the same partial stdout."""
    paths = _paths(load_db(db_name))
    recs = load_json(batch)
    good = [r for r in recs if r["class"] == "PDQ-T"]
    out, err, rc = run_queries_bin(mock_bin, paths, "".join(r["query"] + "\n" for r in good))
    assert rc == 0, err
    assert out == "".join(r["stdout"] for r in good)
    for r in recs:
        if r["class"] == "PDQ-D":
            o, e, _ = run_queries_bin(mock_bin, paths, r["query"] + "\n")
            assert o == r["stdout"] or (o == "" and "refused" in e), (r, o, e)
        elif r["class"] == "CRASH":
            o, e, rc = run_queries_bin(mock_bin, paths, r["query"] + "\n")
            assert o == r["stdout"], (r, o, e)   # whatever the reference printed before it died


@pytest.mark.parametrize("seed", [21, 22, 23])
def test_host_layer_matches_oracle_on_fresh_workloads(mock_bin, seed):
    """Fresh seeded databases and query mixes: host layer + mock == the numpy restatement of
    the reference's state machine (both stable-sorted, so even tie-dependent queries agree)."""
    db = wl.gen_small_db(seed=seed, scale=0.01)
    paths = _paths(db)
    checked = 0
    for q in wl.gen_queries(db, 60, seed=seed, max_joins=3):
        try:
            want = orc.run_batch(db, q + "\n")
        except Exception:   # the reference aborts / the oracle refuses: covered by the golden CRASH cases
            continue
        o, e, rc = run_queries_bin(mock_bin, paths, q + "\n")
        refused = o == "" and "refused" in e
        assert o == want or refused, (q, o, want, e[-300:])
        checked += 1
    assert checked >= 40


def test_host_layer_is_clean_under_asan_ubsan(asan_bin):
    """Well-formed, hazardous and malformed query lines through the sanitizer build: the
    process may refuse or mirror a reference abort, but never touches memory it does not own."""
    rng = np.random.default_rng(5)
    db = wl.gen_small_db(seed=9, scale=0.005)
    paths = _paths(db)
    lines = wl.gen_queries(db, 120, seed=9, max_joins=4)
    lines += ["0 1|0.1=1.1&0.2<20&1.2<20|0.0 1.0", "0|0.1=0.2|0.0", "0 0|0.1=1.1&0.2<20&1.2<20|0.0 1.0", "0|0.2<100&0.1=0.2|0.0",
              "0 1 2 3|0.1=1.1&1.2=2.1&2.2=3.1|0.0 1.0 2.0 3.0", "0 1|0.1=1.1|0.0 1.0 2.0", "0 1|0.9=1.9|0.0", "13 12|0.1=1.1&0.0>3|1.0",
              "0 1|0.1=1.1&0.2|0.0", "9|9|9", "0 1|0.1<5&0.1>7&0.1=3|0.1", "0 1 0|0.1=1.1&1.2=2.1&0.2=2.1|0.0"]
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")   # per-query state is freed; the driver exits without freeing globals
    for i in range(0, len(lines), 4):
        text = "".join(p + "\n" for p in paths) + "Done\n" + "".join(l + "\n" for l in lines[i:i + 4])
        p = subprocess.run([asan_bin], input=text.encode(), stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env, timeout=120)
        err = p.stderr.decode()
        assert "AddressSanitizer" not in err and "runtime error" not in err, (lines[i:i + 4], err[-2000:])


@pytest.mark.parametrize("elide", ["1", "0"])
def test_host_layer_hands_every_handle_back(mock_bin, elide):
    """Every row-id column and tuple run the host layer receives goes back to the engine by the end of the batch
    (the mock counts them).  A predicate with both sides on one binding (0.1=0.2) used to orphan one row-id column
    per query in install_results -- on the GPU that was 112 MB of arena per step of config 3."""
    db = wl.gen_small_db(seed=4, scale=0.01)
    paths = _paths(db)
    lines = wl.gen_queries(db, 60, seed=4, max_joins=3)
    lines += ["0|0.1=0.2|0.0", "0 1|0.1=1.0&0.1=0.2|0.0 1.1", "0 1 2|0.1=0.2&0.1=1.0&1.1=2.0&0.2<100000|0.0 1.0 2.0",
              "0|0.2<100&0.1=0.2|0.0", "0 1|0.1=1.1&0.2<20&1.2<20|0.0 1.0"]
    env = {"QCE_MOCK_BALANCE": "1", "QCE_ELIDE": elide}
    clean = 0
    batches = [lines[i:i + 5] for i in range(0, 60, 5)] + [[l] for l in lines[60:]]
    for batch in batches:  # small batches: a query that mirrors a reference abort ends its process
        o, e, rc = run_queries_bin(mock_bin, paths, "".join(l + "\n" for l in batch), env=env)
        if rc != 0:
            continue
        report = [l for l in e.splitlines() if l.startswith("mock engine:")]
        assert report == ["mock engine: 0 row-id columns and 0 tuple runs were never freed"], (batch, report)
        clean += 1
    assert clean >= 10
