"""GPU parity of the sharded path BEHIND THE C BOUNDARY (SURVEY.md 8e / 8b): the same binaries
as tests/test_gpu_queries.py -- our driver and the reference's unchanged main -- run with
QCE_GPUS=n.  The host layer forks one process per rank before CUDA is touched; the ranks share
the visible devices (rank % device_count), so on a one-GPU box all of them drive the same B200
and still exchange tuples through CUDA-IPC-mapped windows exactly as they do over NVLink.

Two placements are exercised: QCE_REPLICATE_BYTES=0 row-shards EVERY relation (every query runs
on all ranks together, every join is an exchange by key range, every projection pushes its row
ids to the owners), the default replicates these small relations (whole queries are dealt to
single ranks and their stdout is collected in query order)."""
import os
import tempfile

import numpy as np
import pytest

from oracle import qce_oracle as orc
from oracle import workload as wl
from tests.helpers import QUERIES_BIN, REFMAIN_BIN, load_db, load_json, run_queries_bin

pytestmark = pytest.mark.gpu

SHARD_ALL = {"QCE_REPLICATE_BYTES": 0, "QCE_COMM_TIMEOUT_S": 60}


def _paths(db):
    return wl.write_db(tempfile.mkdtemp(), db)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("db_name,batch", [("ops_db.npz", "ops.json"), ("small_db.npz", "small_batch.json"),
                                           ("edge_db.npz", "edge.json")])
def test_golden_batches_row_sharded(world, db_name, batch, elide=1):
    """Every PDQ query of the golden batches with all relations row-sharded over `world` ranks:
    the recorded reference stdout, byte for byte (PDQ-D may be refused, never answered differently)."""
    db = load_db(db_name)
    paths = _paths(db)
    recs = [r for r in load_json(batch) if r["class"] in ("PDQ-T", "PDQ-D")]
    text = "".join(r["query"] + "\n" for r in recs)
    want = "".join(r["stdout"] for r in recs)
    env = dict(SHARD_ALL, QCE_GPUS=world)
    out, err, rc = run_queries_bin(QUERIES_BIN, paths, text, env=env, timeout=600)
    assert rc == 0, err[-2000:]
    if out != want:
        for r in recs:
            o, e, _ = run_queries_bin(QUERIES_BIN, paths, r["query"] + "\n", env=env)
            refused = o == "" and "refused" in e
            assert o == r["stdout"] or (r["class"] == "PDQ-D" and refused), (r, o, e[-1500:])


def test_golden_batch_row_sharded_eight_ranks():
    """QCE_GPUS=8 (the node's size): eight ranks, every relation row-sharded, the operational golden batch."""
    db = load_db("ops_db.npz")
    recs = [r for r in load_json("ops.json") if r["class"] in ("PDQ-T", "PDQ-D")]
    text = "".join(r["query"] + "\n" for r in recs)
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(db), text, env=dict(SHARD_ALL, QCE_GPUS=8, QCE_COMM_TIMEOUT_S=120), timeout=900)
    assert rc == 0, err[-2000:]
    assert out == "".join(r["stdout"] for r in recs)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_golden_batch_replicas(world):
    """Default placement: the small relations are held whole by every rank, whole queries are
    dealt to the ranks (and to several streams per rank), stdout comes back in query order."""
    db = load_db("small_db.npz")
    recs = [r for r in load_json("small_batch.json") if r["class"] == "PDQ-T"]
    text = "".join(r["query"] + "\n" for r in recs)
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(db), text, env={"QCE_GPUS": world}, timeout=600)
    assert rc == 0, err[-2000:]
    assert out == "".join(r["stdout"] for r in recs)


def test_reference_main_unchanged_sharded():
    """The reference's own main/queries_main.c, linked against this library, sharded over 2 ranks."""
    if not os.path.exists(REFMAIN_BIN):
        pytest.skip("build/queries_refmain is built only where the reference's main/queries_main.c is (make REF=<its checkout>)")
    db = wl.gen_pair_db(400_000, 400_000, filt_domain=1000)
    q = "0 1|0.1=1.1&0.2>500|0.0 1.0 1.2\n0|0.1<1000&0.2>500|0.0\n"
    out, err, rc = run_queries_bin(REFMAIN_BIN, _paths(db), q, env=dict(SHARD_ALL, QCE_GPUS=2))
    assert rc == 0, err[-2000:]
    assert out == orc.run_batch(db, q)


@pytest.mark.parametrize("elide", [1, 0])
@pytest.mark.parametrize("world", [2, 3])
def test_scaled_twins_row_sharded(world, elide):
    """C2 / C3 / C4 shapes (filter + join, PK-FK chain with a self-join predicate, Zipf FK side)
    at sizes where the exchange takes the MSD path, against the oracle -- with the bystander
    re-joins elided (the entity's columns travel with the exchanged tuples) and replayed faithfully
    (join_payloads' two runs exchanged by row-id range)."""
    env = dict(SHARD_ALL, QCE_GPUS=world, QCE_ELIDE=elide)
    db = wl.gen_pair_db(3_000_000, 3_000_000)
    q = "0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2\n"
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(db), q, env=env)
    assert rc == 0, err[-2000:]
    assert out == orc.run_batch(db, q)
    db = wl.gen_chain_db(300_000, nrel=4, seed=3)
    q = "0 1 2 3|0.1=0.2&0.1=1.0&1.1=2.0&2.1=3.0&0.3<900|0.3 1.3 2.3 3.3\n"
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(db), q, env=env)
    assert rc == 0, err[-2000:]
    assert out == orc.run_batch(db, q)
    db = wl.gen_zipf_db(300_000, seed=4)
    q = "0 1 2|0.1=1.0&1.1=2.0|0.0 1.2 2.1\n"
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(db), q, env=env)
    assert rc == 0, err[-2000:]
    assert out == orc.run_batch(db, q)


def test_abort_is_mirrored_sharded():
    """A reference exit(EXIT_FAILURE) site ends every rank; rank 0 has printed what the reference had."""
    edge = load_db("edge_db.npz")
    rec = [r for r in load_json("edge.json") if r["query"] == "2 2|0.0=1.0&0.2<8|0.2 1.2"][0]
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(edge), rec["query"] + "\n", env=dict(SHARD_ALL, QCE_GPUS=2))
    assert rc != 0 and out == rec["stdout"] == "18 " and "Something went really wrong" in err


def test_golden_batch_row_sharded_faithful_replay():
    """The golden batch with elided mode switched off: every bystander re-join is the exchanged replay."""
    db = load_db("small_db.npz")
    recs = [r for r in load_json("small_batch.json") if r["class"] == "PDQ-T"]
    text = "".join(r["query"] + "\n" for r in recs)
    out, err, rc = run_queries_bin(QUERIES_BIN, _paths(db), text, env=dict(SHARD_ALL, QCE_GPUS=2, QCE_ELIDE=0), timeout=600)
    assert rc == 0, err[-2000:]
    assert out == "".join(r["stdout"] for r in recs)
