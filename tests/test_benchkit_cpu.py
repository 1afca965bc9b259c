"""CPU: the bench's synthetic workloads (tools/benchkit.py) and their INDEPENDENT checkers on scaled twins,
held to the reference's stdout recorded in tests/golden/twins.json (tests/golden/make_golden.py), as is the
numpy oracle, and to the compiled reference (oracle/_ref/queries) on top where it is built.  bench.py trusts
these checkers at sizes no CPU run can reach (10^9 rows); here the same index-map / closed-form code must
reproduce the reference's stdout byte for byte where the reference can run -- which also shows the
generated queries sit inside the parity-defined query class (SURVEY.md 8c)."""
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import qce_oracle as orc
from oracle import workload as wl
from tests.helpers import load_json
from tools import benchkit as bk


@pytest.fixture(autouse=True)
def _cpu_device():
    old, bk.DEVICE = bk.DEVICE, "cpu"
    yield
    bk.DEVICE = old


def _db(w):
    return [[w.column_np(r, c) for c in range(len(w.relations[r][1]))] for r in range(len(w.relations))]


def _expected(name, db, text):
    """the stdout recorded for twin `name` (its stdin text must be the one recorded); the oracle must print
    it, and so must the compiled reference wherever oracle/_ref/queries is built"""
    rec = load_json("twins.json")[name]
    assert text == rec["text"]
    want = rec["stdout"]
    assert orc.run_batch(db, text) == want
    if wl.have_reference():
        out, err, rc = wl.run_reference(wl.write_db(tempfile.mkdtemp(), db), text)
        assert rc == 0, err
        assert out == want
    return want


def test_hash_is_the_same_function_in_numpy_and_torch():
    i = np.arange(0, 5000, dtype=np.uint64) * np.uint64(977) + np.uint64(3)
    for seed in (0, 1, 7, 5003):
        a = bk.mix_np(i, seed)
        b = bk.mix_t(torch, torch.from_numpy(i.view(np.int64)), seed).numpy().view(np.uint64)
        np.testing.assert_array_equal(a, b)
    w = bk.c3_workload(4096)
    for r in range(4):
        for c in range(4):
            np.testing.assert_array_equal(w.column_np(r, c), w.column_t(torch, r, c, 0, 4096).numpy().view(np.uint64))
    assert sorted(w.column_np(2, 0).tolist()) == list(range(4096))  # the primary keys are a permutation


def test_c3_checker_equals_the_reference():
    w = bk.c3_workload(40_000)
    out = _expected("benchkit_c3", _db(w), w.text(0))
    # the checker evaluated in two row windows, as the ranks of a sharded run do
    p1, s1 = bk.c3_check(torch, w, 0, 16_384)
    p2, s2 = bk.c3_check(torch, w, 16_384, 40_000 - 16_384)
    assert out == bk.format_line(p1 + p2, [(a + b) & bk.M64 for a, b in zip(s1, s2)])


def test_c4_checker_equals_the_reference():
    w = bk.c4_workload(60_000)
    out = _expected("benchkit_c4", _db(w), w.text(0))
    pairs, sums = bk.c4_check(torch, w, 0, w.rows(0))
    assert out == bk.format_line(pairs, sums)
    # Zipf(1.2): the heaviest key really is heavy
    z = w.z("np", np.arange(60_000, dtype=np.uint64))
    assert np.bincount(z.astype(np.int64)).max() > 0.1 * 60_000


def test_c5_batch_checker_equals_the_reference():
    w = bk.c5_workload(scale=1.0 / 10000, nqueries=120)
    out = _expected("benchkit_c5", _db(w), w.text(0))
    want = ""
    for k in range(len(w.queries)):
        first, pairs, sums = bk.c5_check_query(torch, w, k, 0, w.rows(w.plans[k][0][0]))
        if first is not None:
            want += "%d\n" % first
        want += bk.format_line(pairs, sums)
    assert out == want


def test_c2_closed_form_equals_the_reference():
    n = 200_000
    db = wl.gen_pair_db(n, n)
    out = _expected("benchkit_c2", db, "0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2\n")
    t = [[torch.from_numpy(c.view(np.int64)) for c in rel] for rel in db]
    lhs, pairs, sums = bk.c2_check(torch, None, t[0][1], t[0][2], t[0][0], t[1][1], t[1][0], t[1][2], n, 500000)
    assert out == bk.format_line(pairs, sums)
