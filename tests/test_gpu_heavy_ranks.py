"""GPU: joins whose exchange cuts inside a heavy key (qce_split_plan, k_push_split), through the
same binaries as tests/test_gpu_ranks.py with every relation row-sharded over QCE_GPUS ranks (the
ranks may share one B200).  Every case is held to the oracle byte for byte, and the QCE_TRACE join
lines show which route each join took and what every rank received."""
import os
import re
import tempfile

import numpy as np
import pytest

from oracle import qce_oracle as orc
from oracle import workload as wl
from tests.helpers import QUERIES_BIN, REFMAIN_BIN, run_queries_bin

pytestmark = pytest.mark.gpu

TRACE = re.compile(r"\[qce\] join rank (\d+)/(\d+): route=(\w+) keys=(\w+) width=(\d+) recv R=(\d+)/(\d+) S=(\d+)/(\d+)"
                   r" split=(\d+) levels=(\d+)")
C4 = "0 1 2|0.1=1.0&1.1=2.0|0.0 1.2 2.1\n"


def _run(db, q, world, elide=1, binary=QUERIES_BIN):
    paths = wl.write_db(tempfile.mkdtemp(), db)
    env = {"QCE_REPLICATE_BYTES": 0, "QCE_COMM_TIMEOUT_S": 120, "QCE_GPUS": world, "QCE_ELIDE": elide, "QCE_TRACE": 1}
    out, err, rc = run_queries_bin(binary, paths, q, env=env, timeout=900)
    assert rc == 0, err[-2000:]
    assert out == orc.run_batch(db, q)
    joins = {}   # rank -> its join lines in order
    for m in TRACE.finditer(err):
        joins.setdefault(int(m.group(1)), []).append([m.group(3)] + [int(x) for x in m.groups()[4:]])
    assert sorted(joins) == list(range(world)), err[-2000:]
    return [[joins[r][j] for r in range(world)] for j in range(len(joins[0]))]


def _balanced(join, world):
    """every rank's R + S received within 10 % of its share, plus one inner copy per split rank"""
    total = join[0][3] + join[0][5]   # R and S tuples over all ranks
    for route, width, r, rt, s, st, split, levels in join:
        assert r + s <= 1.10 * total / world + world, (r + s, total / world, join)


@pytest.mark.parametrize("elide", [1, 0])
@pytest.mark.parametrize("world", [3, 8])
def test_zipf_c4(world, elide):
    """Config 4's shape: Zipf(1.2) FK side, heavy on the outer side of both joins.  The parent's bin
    cuts leave the first join at 1.44 of a share at 8 ranks."""
    joins = _run(wl.gen_zipf_db(3_000_000), C4, world, elide)
    first = joins[0]
    _balanced(first, world)
    if world == 8:
        assert first[0][7] >= 1   # refined below the top-8-bit bins


@pytest.mark.parametrize("world", [3, 8])
def test_one_key_on_most_of_r(world):
    """One key on 60 % of R: its outer tuples are sliced over several ranks."""
    db = wl.gen_pair_db(2_000_000, 2_000_000)
    db[0][1][: 1_200_000] = 777_777
    joins = _run(db, "0 1|0.1=1.1|0.0 1.2\n", world)
    _balanced(joins[0], world)
    if world == 8:
        assert joins[0][0][6] >= 1
        assert sum(1 for j in joins[0] if j[2] >= 100_000) >= 3


@pytest.mark.parametrize("elide", [1, 0])
def test_heavy_pk_row_repeats_through_the_chain(elide):
    """60 % of R0.c1 on one PK value: both joins split, and the second join's outer side repeats one row
    id on 60 % of its tuples (the faithful re-join then deduplicates pairs across ranks)."""
    db = wl.gen_zipf_db(1_000_000)
    db[0][1][: 600_000] = db[1][0][12345]
    joins = _run(db, C4, 8, elide)
    assert joins[0][0][6] >= 1 and joins[1][0][6] >= 1


def test_key_heavy_on_both_sides():
    """300 K outer and 200 inner tuples of one key (60 M pairs): the inner group goes to every rank of
    the key's span."""
    n = 1_000_000
    rng = np.random.default_rng(11)
    r = rng.integers(0, 1 << 24, n, dtype=np.uint64)
    r[: 300_000] = 4_242_424
    s = rng.integers(0, 1 << 24, n, dtype=np.uint64)
    s[: 200] = 4_242_424
    db = [[np.arange(n, dtype=np.uint64), r], [np.arange(n, dtype=np.uint64), s]]
    joins = _run(db, "0 1|0.1=1.1|0.0 1.0\n", 8)
    assert joins[0][0][6] >= 1
    assert sum(1 for j in joins[0] if j[4] >= 200) >= 2   # the 200 inner tuples on several ranks


def test_inner_only_heavy_key_stays_whole():
    """A key heavy only on the inner side (one outer tuple) is never split: its outer tuple's match count
    stays on one rank."""
    n = 500_000
    rng = np.random.default_rng(12)
    s = rng.integers(0, n, n, dtype=np.uint64)
    s[: n // 2] = 4321
    db = [[np.arange(n, dtype=np.uint64), rng.integers(0, 1000, n, dtype=np.uint64)],
          [np.arange(n, dtype=np.uint64), s]]
    joins = _run(db, "0 1|0.0=1.1|0.1 1.0\n", 2)
    assert all(j[6] == 0 for j in joins[0])


def test_split_output_joined_again_then_self_join():
    """A split join's output column joined again on the same column, then a predicate with both sides on
    one binding (scan_join)."""
    db = wl.gen_zipf_db(1_000_000)
    db[0][1][: 500_000] = db[1][0][7]
    _run(db, "0 1 2|0.1=1.0&1.0=2.0&1.1=1.1|0.0 1.2 2.1\n", 8)


def test_uniform_c2_keeps_the_bin_cuts():
    """The uniform C2 twin: within 10 % on the bin cuts, so no refinement and nothing split."""
    db = wl.gen_pair_db(3_000_000, 3_000_000)
    joins = _run(db, "0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2\n", 8)
    assert all(j[6] == 0 and j[7] == 0 for j in joins[0])


def test_reference_main_zipf():
    """The reference's own main, linked against this library, on a split Zipf join."""
    if not os.path.exists(REFMAIN_BIN):
        pytest.skip("build/queries_refmain is built only where the reference's main/queries_main.c is")
    _run(wl.gen_zipf_db(1_000_000), C4, 8, binary=REFMAIN_BIN)
