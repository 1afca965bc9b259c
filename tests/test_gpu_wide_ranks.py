"""GPU: joins on keys >= 2^32 over several ranks (QCE_GPUS=n, every relation row-sharded) are
exchanged by key range like packed ones -- binned by key - (smallest key) over the width of the key
range -- instead of being gathered on rank 0.  The binaries' stdout must equal the oracle's byte for
byte, and the engine's QCE_TRACE lines must show every wide join taking the exchange on every rank."""
import os
import re
import tempfile

import numpy as np
import pytest

from oracle import qce_oracle as orc
from oracle import workload as wl
from tests.helpers import QUERIES_BIN, REFMAIN_BIN, run_queries_bin

pytestmark = pytest.mark.gpu
U64 = np.uint64
OFF = U64(1 << 40)
TOP = (1 << 64) - 1
SHARD_ALL = {"QCE_REPLICATE_BYTES": 0, "QCE_COMM_TIMEOUT_S": 120, "QCE_TRACE": 1}
TRACE = re.compile(r"\[qce\] join rank (\d+)/(\d+): route=(\w+) keys=(\w+) width=(\d+) recv R=(\d+)/(\d+) S=(\d+)/(\d+)")


def _run(db, q, world, elide=1, binary=QUERIES_BIN, timeout=900):
    paths = wl.write_db(tempfile.mkdtemp(), db)
    out, err, rc = run_queries_bin(binary, paths, q, env=dict(SHARD_ALL, QCE_GPUS=world, QCE_ELIDE=elide), timeout=timeout)
    assert rc == 0, err[-3000:]
    assert out == orc.run_batch(db, q)
    joins = [tuple(int(x) if x.isdigit() else x for x in m.groups()) for m in TRACE.finditer(err)]
    wide = [j for j in joins if j[3] == "wide"]
    assert wide, "no wide join reported"
    assert all(j[2] == "exchange" for j in wide), wide
    assert {j[0] for j in wide} == set(range(world)) and all(j[1] == world for j in wide)
    return wide


def _wide_join_db(n=300_000, seed=5):
    """the shape of test_wide_keys_join: a 50k-value domain in [2^40, 2^62)"""
    rng = np.random.default_rng(seed)
    dom = rng.integers(1 << 40, 1 << 62, 50_000, dtype=np.uint64)
    return [[np.arange(n, dtype=U64), dom[rng.integers(0, len(dom), n)], rng.integers(0, 1000, n, dtype=np.uint64)]
            for _ in range(2)]


def _c2_wide_db(n=3_000_000):
    db = wl.gen_pair_db(n, n)
    for r in db:
        r[1] = r[1] + OFF
    return db


def _ends_db(n=200_000, seed=11):
    """keys over the whole of [0, 2^64 - 1], both ends present on both sides"""
    rng = np.random.default_rng(seed)
    dom = rng.integers(0, TOP, 40_000, dtype=np.uint64, endpoint=True)
    dom[:2] = [0, TOP]
    db = []
    for _ in range(2):
        c1 = dom[rng.integers(0, len(dom), n)]
        c1[:4] = [0, TOP, 0, TOP]
        db.append([np.arange(n, dtype=U64), c1, rng.integers(0, 1000, n, dtype=np.uint64)])
    return db


def _zipf_wide_db(n=300_000):
    db = wl.gen_zipf_db(n, seed=4)
    db[0][1] = db[0][1] + OFF   # Zipf FK side
    db[1][0] = db[1][0] + OFF   # the PK it refers to
    return db


def _mixed_db(n=300_000, seed=13):
    """R0's join column below 2^32, R1's partly above (the packed side is widened)"""
    rng = np.random.default_rng(seed)
    dom = rng.integers(0, 1 << 31, 50_000, dtype=np.uint64)
    c0 = dom[rng.integers(0, len(dom), n)]
    c1 = dom[rng.integers(0, len(dom), n)]
    big = rng.random(n) < 0.2
    c1[big] = OFF + rng.integers(0, 1 << 20, int(big.sum()), dtype=np.uint64)
    return [[np.arange(n, dtype=U64), c0, rng.integers(0, 1000, n, dtype=np.uint64)],
            [np.arange(n, dtype=U64), c1, rng.integers(0, 1000, n, dtype=np.uint64)]]


def _chain_db(n=100_000, seed=17):
    rng = np.random.default_rng(seed)
    dom = OFF + rng.integers(0, 1 << 30, 50_000, dtype=np.uint64)
    return [[np.arange(n, dtype=U64), dom[rng.integers(0, len(dom), n)], rng.integers(0, 1000, n, dtype=np.uint64)]
            for _ in range(3)]


@pytest.mark.parametrize("elide", [1, 0])
@pytest.mark.parametrize("world", [2, 3])
def test_wide_joins_row_sharded(world, elide):
    _run(_wide_join_db(), "0 1|0.1=1.1&0.2<500|0.0 1.0 0.1\n", world, elide)
    wide = _run(_c2_wide_db(), "0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2\n", world, elide)
    if world == 3:   # a balanced key-range share; the rank-0 route gives one rank everything
        for j in wide:
            assert j[5] <= 0.45 * j[6] and j[7] <= 0.45 * j[8], j
    _run(_ends_db(), "0 1|0.1=1.1|0.0 1.0 0.1\n", world, elide)
    _run(_zipf_wide_db(), "0 1 2|0.1=1.0&1.1=2.0|0.0 1.2 2.1\n", world, elide)
    _run(_mixed_db(), "0 1|0.1=1.1|0.0 1.0 1.1\n", world, elide)
    _run(_chain_db(), "0 1 2|0.1=1.1&1.1=2.1|0.0 1.0 2.0 1.1\n", world, elide)


def test_wide_c2_eight_ranks():
    wide = _run(_c2_wide_db(), "0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2\n", 8)
    for j in wide:
        assert j[5] <= 0.2 * j[6] and j[7] <= 0.2 * j[8], j


def test_reference_main_wide_sharded():
    """The reference's own main/queries_main.c, linked against this library, on a wide-key join over 2 ranks."""
    if not os.path.exists(REFMAIN_BIN):
        pytest.skip("build/queries_refmain is built only where the reference's main/queries_main.c is (make REF=<its checkout>)")
    _run(_wide_join_db(), "0 1|0.1=1.1&0.2<500|0.0 1.0 0.1\n", 2, binary=REFMAIN_BIN)
