"""CPU: the numpy oracle against the reference on fresh random queries and the C2 twin: against the stdout
recorded in tests/golden/twins.json (tests/golden/make_golden.py) always, and against the live reference
binary on top where it is built (oracle/_ref, only where the reference's sources were available)."""
import tempfile

from oracle import qce_oracle as orc
from oracle import workload as wl
from tests.helpers import load_json


def test_random_queries_against_live_reference():
    db = wl.gen_small_db(seed=99, scale=0.002)
    recs = load_json("twins.json")["random_small"]
    queries = wl.gen_queries(db, 30, seed=123)
    assert [r["query"] for r in recs] == queries
    n_checked = 0
    for rec in recs:
        if rec["class"] in ("TIE", "CRASH"):
            continue  # tie-dependent or crashing in the reference: undefined, excluded
        assert orc.run_batch(db, rec["query"] + "\n") == rec["stdout"], rec["query"]
        n_checked += 1
    assert n_checked >= 20
    if wl.have_reference():
        paths = wl.write_db(tempfile.mkdtemp(), db)
        n_checked = 0
        for q in queries:
            cls, ref = wl.classify(paths, db, q + "\n", timeout=60)
            if cls in ("PDQ-T", "PDQ-D"):
                assert orc.run_batch(db, q + "\n") == ref, q
                n_checked += 1
        assert n_checked >= 20


def test_c2_scaled_twin_against_live_reference():
    db = wl.gen_pair_db(20000, 20000, filt_domain=1000)
    q = "0 1|0.1=1.1&0.2>500|0.0 1.0 1.2\n"
    rec = load_json("twins.json")["c2_twin"]
    assert rec["text"] == q
    assert orc.run_batch(db, q) == rec["stdout"]
    if wl.have_reference():
        ref, _, rc = wl.run_reference(wl.write_db(tempfile.mkdtemp(), db), q)
        assert rc == 0 and ref == rec["stdout"]
