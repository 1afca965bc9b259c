"""GPU parity, primitive by primitive: every CUDA operator called through the
C-ABI (libqce_b200.so) against the numpy oracle on the same seeded inputs.
Bar: bit-exact (all arithmetic on this path is uint64 / index work)."""
import numpy as np
import pytest

from oracle import qce_oracle as orc

pytestmark = pytest.mark.gpu
U64 = np.uint64

SIZES = [0, 1, 2, 31, 32, 33, 63, 64, 65, 4095, 4096, 4097, 8191, 12289, 100003, 1 << 20]


def _col(rng, n, domain):
    return rng.integers(0, max(1, domain), n, dtype=np.uint64)


def _assert_sorted_run(k, p, keys, payloads):
    """The run is sorted by key and is a permutation of the input tuples.  The
    order among EQUAL keys is unspecified (large runs take the MSD partition path,
    which is not stable -- neither is the reference's rand()-driven quicksort)."""
    order = np.argsort(keys, kind="stable")
    np.testing.assert_array_equal(k, keys[order])
    got = np.lexsort((p, k))
    want = np.lexsort((payloads[order], keys[order]))
    np.testing.assert_array_equal(p[got], payloads[order][want])


# ------------------------------------------------------------------ filter scan
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("op", ["<", ">", "="])
def test_filter_scan(engine, n, op):
    rng = np.random.default_rng(n * 3 + ord(op))
    col = _col(rng, n, 1000)
    engine.upload_column(100, 0, col)
    c = 500 if op != "=" else (int(col[n // 2]) if n else 7)
    h = engine.filter_scan(100, 0, op, c)
    got = engine.rowids_to_host(h)
    engine.rowids_free(h)
    np.testing.assert_array_equal(got, orc.filter_scan(col, op, c))


@pytest.mark.parametrize("sel", [0.0, 1.0, 0.001, 0.999])
def test_filter_scan_selectivity_extremes(engine, sel):
    rng = np.random.default_rng(5)
    n = 300007
    col = _col(rng, n, 1 << 40)  # wide values: compare is 64-bit unsigned
    c = int(sel * (1 << 40))
    engine.upload_column(100, 1, col)
    h = engine.filter_scan(100, 1, "<", c)
    np.testing.assert_array_equal(engine.rowids_to_host(h), orc.filter_scan(col, "<", c))
    engine.rowids_free(h)


def test_filter_wrong_operator(engine):
    import qce_b200
    engine.upload_column(100, 2, np.arange(10, dtype=U64))
    with pytest.raises(qce_b200.EngineError, match="Wrong operator"):
        engine.filter_scan(100, 2, "!", 3)


# ------------------------------------------------------------------ filter refine
@pytest.mark.parametrize("n", [0, 1, 33, 4096, 4097, 70001])
@pytest.mark.parametrize("op", ["<", ">", "="])
def test_filter_refine(engine, n, op):
    rng = np.random.default_rng(n + ord(op))
    rows = 50000
    col = _col(rng, rows, 100)
    engine.upload_column(101, 0, col)
    ids = rng.integers(0, rows, n, dtype=np.uint64)  # unsorted, with repeats
    h = engine.rowids_from_host(ids)
    cnt = engine.filter_refine(h, 101, 0, op, 40)
    want = orc.filter_refine(ids, col, op, 40)
    assert cnt == len(want)
    np.testing.assert_array_equal(engine.rowids_to_host(h), want)
    engine.rowids_free(h)


# ------------------------------------------------------------------ build + sort
@pytest.mark.parametrize("n", [0, 1, 2, 100, 4095, 4096, 4097, 8192, 100003, 1 << 20])
@pytest.mark.parametrize("domain", [1, 7, 1 << 8, 1 << 20, (1 << 32) - 1, 1 << 33, 1 << 62])
def test_build_and_sort_base(engine, n, domain):
    rng = np.random.default_rng(n ^ domain & 0xFFFF)
    col = _col(rng, n, domain)
    engine.upload_column(102, 0, col)
    t = engine.build_tuples(102, 0)
    k, p = engine.tuples_to_host(t)
    wk, wp = orc.build_tuples(col)
    np.testing.assert_array_equal(k, wk)
    np.testing.assert_array_equal(p, wp)
    engine.sort_tuples(t)
    assert engine.is_sorted(t)
    k, p = engine.tuples_to_host(t)
    _assert_sorted_run(k, p, wk, wp)
    if n < (1 << 20):  # below the MSD threshold the LSD passes keep ties in input order
        sk, sp = orc.sort_tuples(wk, wp)
        np.testing.assert_array_equal(p, sp)
    engine.tuples_free(t)


@pytest.mark.parametrize("n", [2, 4097, 2_500_000])
@pytest.mark.parametrize("kind", ["ascending", "ascending-with-ties", "one-inversion-at-the-end", "one-inversion-at-the-start"])
def test_sort_of_a_column_stored_in_order(engine, n, kind):
    """A run built from a whole base column is probed before it is sorted (k_probe_sorted): a column already
    in key order is left as it stands, a single inversion anywhere sends it through the sort."""
    col = np.arange(n, dtype=U64) * 3
    if kind == "ascending-with-ties":
        col = col // 12
    elif kind == "one-inversion-at-the-end":
        col[-1] = 0
    elif kind == "one-inversion-at-the-start":
        col[0] = col[-1] + 5
    engine.upload_column(104, 0, col)
    t = engine.build_tuples(104, 0)
    engine.sort_tuples(t)
    assert engine.is_sorted(t)
    k, p = engine.tuples_to_host(t)
    _assert_sorted_run(k, p, *orc.build_tuples(col))
    engine.tuples_free(t)


def test_sort_skewed_and_presorted(engine):
    rng = np.random.default_rng(9)
    n = 500000
    for keys in (np.zeros(n, dtype=U64), np.arange(n, dtype=U64), np.arange(n, dtype=U64)[::-1].copy(),
                 (rng.zipf(1.2, n) % (1 << 30)).astype(U64)):
        t = engine.tuples_from_host(keys, np.arange(n, dtype=U64))
        engine.sort_tuples(t)
        k, p = engine.tuples_to_host(t)
        sk, sp = orc.sort_tuples(keys, np.arange(n, dtype=U64))
        np.testing.assert_array_equal(k, sk)
        np.testing.assert_array_equal(p, sp)
        engine.tuples_free(t)


def test_build_through_rowids(engine):
    rng = np.random.default_rng(3)
    col = _col(rng, 100000, 1 << 20)
    engine.upload_column(103, 0, col)
    ids = np.sort(rng.choice(100000, 30000, replace=False)).astype(U64)
    h = engine.rowids_from_host(ids)
    t = engine.build_tuples(103, 0, h)
    k, p = engine.tuples_to_host(t)
    wk, wp = orc.build_tuples(col, ids)
    np.testing.assert_array_equal(k, wk)
    np.testing.assert_array_equal(p, wp)
    assert not engine.is_sorted(t)
    engine.tuples_free(t)
    engine.rowids_free(h)


# ------------------------------------------------------------------ merge join
def _join_case(engine, kR, pR, kS, pS, distinct=False):
    kR, pR = orc.sort_tuples(kR, pR)
    kS, pS = orc.sort_tuples(kS, pS)
    R = engine.tuples_from_host(kR, pR)
    S = engine.tuples_from_host(kS, pS)
    res = engine.merge_join(R, S, distinct=distinct)
    gR, gS = engine.rowids_to_host(res[0]), engine.rowids_to_host(res[1])
    wR, wS = orc.merge_join(kR, pR, kS, pS)
    np.testing.assert_array_equal(gR, wR)
    np.testing.assert_array_equal(gS, wS)
    if distinct:
        dR, dS = engine.rowids_to_host(res[2]), engine.rowids_to_host(res[3])
        wdR, wdS = orc.distinct_pairs(wR, wS)
        np.testing.assert_array_equal(dR, wdR)
        np.testing.assert_array_equal(dS, wdS)
    for h in res:
        engine.rowids_free(h)
    engine.tuples_free(R)
    engine.tuples_free(S)
    return len(wR)


@pytest.mark.parametrize("nR,nS,domain", [
    (0, 10, 5), (10, 0, 5), (1, 1, 1), (100, 100, 10), (5000, 3000, 1000), (2048, 2049, 4096),
    (100000, 100000, 100000), (300000, 1000, 1 << 20), (1000, 300000, 1 << 20), (50000, 50000, 1 << 34),
    (4097, 200000, 50),  # every R tile spans a window larger than the staging buffer
])
def test_merge_join(engine, nR, nS, domain):
    rng = np.random.default_rng(nR * 7 + nS)
    kR, kS = _col(rng, nR, domain), _col(rng, nS, domain)
    _join_case(engine, kR, np.arange(nR, dtype=U64), kS, np.arange(nS, dtype=U64))


def test_merge_join_heavy_key(engine):
    """One key with 3000 x 2000 matches: the pair list of a single group is split
    over many write CTAs."""
    rng = np.random.default_rng(1)
    kR = np.concatenate([np.full(3000, 77, dtype=U64), _col(rng, 5000, 1000)])
    kS = np.concatenate([np.full(2000, 77, dtype=U64), _col(rng, 5000, 1000)])
    m = _join_case(engine, kR, np.arange(len(kR), dtype=U64), kS, np.arange(len(kS), dtype=U64))
    assert m >= 6_000_000


def test_merge_join_distinct_pairs(engine):
    """Row ids repeat on both sides (as after an earlier join): the distinct
    (rowid_R,rowid_S) pairs are what the reference's Hashmap dedup keeps."""
    rng = np.random.default_rng(2)
    col_r, col_s = _col(rng, 400, 50), _col(rng, 300, 50)
    pR = rng.integers(0, 400, 3000, dtype=np.uint64)
    pS = rng.integers(0, 300, 2000, dtype=np.uint64)
    _join_case(engine, col_r[pR], pR, col_s[pS], pS, distinct=True)


# ------------------------------------------------------------------ scan join / rejoin / checksum
@pytest.mark.parametrize("nR,nS", [(0, 5), (100, 100), (5000, 4097), (70000, 90000)])
def test_scan_join(engine, nR, nS):
    rng = np.random.default_rng(nR + nS)
    colR, colS = _col(rng, 1000, 4), _col(rng, 2000, 4)
    engine.upload_column(104, 0, colR)
    engine.upload_column(105, 0, colS)
    iR, iS = rng.integers(0, 1000, nR, dtype=np.uint64), rng.integers(0, 2000, nS, dtype=np.uint64)
    hR, hS = engine.rowids_from_host(iR), engine.rowids_from_host(iS)
    oR, oS = engine.scan_join(104, 0, hR, 105, 0, hS)
    wR, wS = orc.scan_join(colR[iR], iR, colS[iS], iS)
    np.testing.assert_array_equal(engine.rowids_to_host(oR), wR)
    np.testing.assert_array_equal(engine.rowids_to_host(oS), wS)
    for h in (hR, hS, oR, oS):
        engine.rowids_free(h)


def test_scan_join_base(engine):
    rng = np.random.default_rng(8)
    a, b = _col(rng, 10000, 3), _col(rng, 10000, 3)
    engine.upload_column(106, 0, a)
    engine.upload_column(106, 1, b)
    oR, oS = engine.scan_join(106, 0, None, 106, 1, None)
    want = np.nonzero(a == b)[0].astype(U64)
    np.testing.assert_array_equal(engine.rowids_to_host(oR), want)
    np.testing.assert_array_equal(engine.rowids_to_host(oS), want)
    engine.rowids_free(oR)
    engine.rowids_free(oS)


@pytest.mark.parametrize("n,m", [(0, 0), (10, 0), (1000, 700), (50000, 120000)])
def test_rejoin(engine, n, m):
    rng = np.random.default_rng(n + m)
    last = rng.integers(0, 5000, n, dtype=np.uint64)
    edit = rng.integers(0, 9000, n + 3, dtype=np.uint64)  # longer than `last`: the tail is ignored
    driver = rng.integers(0, 5000, m, dtype=np.uint64)
    hd, hl, he = engine.rowids_from_host(driver), engine.rowids_from_host(last), engine.rowids_from_host(edit)
    out = engine.rejoin(hd, hl, he)
    np.testing.assert_array_equal(engine.rowids_to_host(out), orc.join_payloads(driver, last, edit))
    for h in (hd, hl, he, out):
        engine.rowids_free(h)


def test_rejoin_short_bystander_is_refused(engine):
    import qce_b200
    hd = engine.rowids_from_host(np.arange(4, dtype=U64))
    hl = engine.rowids_from_host(np.arange(10, dtype=U64))
    he = engine.rowids_from_host(np.arange(5, dtype=U64))
    with pytest.raises(qce_b200.EngineError, match="reads past"):
        engine.rejoin(hd, hl, he)
    for h in (hd, hl, he):
        engine.rowids_free(h)


@pytest.mark.parametrize("m", [0, 1, 3, 4, 5, 1023, 100001])
def test_checksum(engine, m):
    rng = np.random.default_rng(m)
    cols = [rng.integers(0, 1 << 63, 20000, dtype=np.uint64) * U64(2) + U64(1) for _ in range(3)]  # sums wrap
    for c, v in enumerate(cols):
        engine.upload_column(107, c, v)
    ids = rng.integers(0, 20000, m, dtype=np.uint64)
    h = engine.rowids_from_host(ids)
    got = engine.checksum(h, 107, [0, 1, 2])
    assert got == [orc.checksum(c, ids) for c in cols]
    assert engine.checksum(h, 107, [2]) == [orc.checksum(cols[2], ids)]
    engine.rowids_free(h)


# ------------------------------------------------------------------ exchange step
@pytest.mark.parametrize("nparts", [1, 2, 4, 8])
def test_partition_tuples(engine, nparts):
    rng = np.random.default_rng(nparts)
    n = 200003
    keys = _col(rng, n, 1 << 24)
    t = engine.tuples_from_host(keys, np.arange(n, dtype=U64))
    splitters = [(i + 1) * (1 << 24) // nparts for i in range(nparts - 1)]
    counts, buf = engine.partition_tuples(t, 24, splitters, nparts)
    part = np.searchsorted(np.array(splitters, dtype=U64), keys, side="right") if nparts > 1 else np.zeros(n, dtype=int)
    assert counts == [int((part == p).sum()) for p in range(nparts)]
    back = engine.tuples_from_device_packed(buf, n, 24, n)
    k, p = engine.tuples_to_host(back)
    # every destination's slice holds exactly its tuples (order inside a slice is unspecified:
    # the receiver sorts it)
    start = 0
    for d in range(nparts):
        sl = slice(start, start + counts[d])
        got = np.sort((k[sl] << U64(32)) | p[sl])
        want = np.sort((keys[part == d] << U64(32)) | np.arange(n, dtype=U64)[part == d])
        np.testing.assert_array_equal(got, want)
        start += counts[d]
    engine.exchange_release(buf)
    engine.tuples_free(back)
    engine.tuples_free(t)


@pytest.mark.parametrize("nR,nS,domain", [(1, 1, 1), (500, 400, 50), (5000, 9000, 300), (30000, 20000, 1 << 33)])
def test_merge_join_walk_unsorted_outer(engine, nR, nS, domain):
    """Outer run in arbitrary order, inner sorted: must equal the reference's
    literal pointer walk (oracle._merge_serial restates src/join.c:342-377)."""
    rng = np.random.default_rng(nR + nS)
    kR, pR = _col(rng, nR, domain), np.arange(nR, dtype=U64)
    kS, pS = orc.sort_tuples(_col(rng, nS, domain), np.arange(nS, dtype=U64))
    R, S = engine.tuples_from_host(kR, pR), engine.tuples_from_host(kS, pS)
    oR, oS = engine.merge_join_walk(R, S)
    wR, wS = orc._merge_serial(kR, pR, kS, pS)
    np.testing.assert_array_equal(engine.rowids_to_host(oR), wR)
    np.testing.assert_array_equal(engine.rowids_to_host(oS), wS)
    for h in (oR, oS):
        engine.rowids_free(h)
    engine.tuples_free(R)
    engine.tuples_free(S)


def test_checksum_bucketed_path():
    """The L2-bucketed gather (ids partitioned by their top bits first) is chosen
    by size; force it in a child process and compare with the oracle."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r)
import qce_b200
from oracle import qce_oracle as orc
e = qce_b200.Engine()
rng = np.random.default_rng(3)
for rows, m in ((1000, 1), (70000, 5), (300000, 123457), (1 << 20, 3000001)):
    cols = [rng.integers(0, 1 << 63, rows, dtype=np.uint64) * np.uint64(2) + np.uint64(1) for _ in range(2)]
    for c, v in enumerate(cols):
        e.upload_column(7, c, v)
    ids = rng.integers(0, rows, m, dtype=np.uint64)
    h = e.filter_scan(7, 0, ">", 0) if False else e.rowids_from_host(ids)
    assert e.checksum(h, 7, [0, 1]) == [orc.checksum(c, ids) for c in cols], (rows, m)
    e.rowids_free(h)
print("bucketed ok", e.profile_read())
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, QCE_BUCKETED_CHECKSUM="1")
    p = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert p.returncode == 0 and "bucketed ok" in p.stdout, p.stderr[-2000:]


@pytest.mark.parametrize("begin,count", [(0, 0), (0, 5000), (4096, 4097), (8192, 91808), (99998, 2)])
def test_row_window_scan_and_build(engine, begin, count):
    """Row-window variants (one rank's share of a sharded scan/build): row ids stay
    relation-global."""
    rng = np.random.default_rng(begin + count)
    col = _col(rng, 100000, 1 << 20)
    engine.upload_column(108, 0, col)
    h = engine.filter_scan(108, 0, "<", 1 << 19, rows=(begin, count))
    want = orc.filter_scan(col[begin:begin + count], "<", 1 << 19) + U64(begin)
    np.testing.assert_array_equal(engine.rowids_to_host(h), want)
    engine.rowids_free(h)
    t = engine.build_tuples(108, 0, rows=(begin, count))
    k, p = engine.tuples_to_host(t)
    np.testing.assert_array_equal(k, col[begin:begin + count])
    np.testing.assert_array_equal(p, np.arange(begin, begin + count, dtype=U64))
    engine.tuples_free(t)


@pytest.mark.parametrize("n,kind", [(3_000_000, "uniform27"), (2_500_001, "uniform20"), (3_000_000, "zipf"),
                                    (2_000_000, "few_keys"), (1_048_576, "dense"), (5_000_000, "uniform32"),
                                    (4_000_000, "heavy_in_sparse"), (6_000_000, "zipf_dense"), (3_000_000, "one_key_plus")])
def test_large_sort_msd_and_fallback(engine, n, kind):
    """Large packed runs: MSD partition + shared-memory finish for non-skewed keys; sub-buckets a heavy
    key overflows take one more multi-CTA counting pass (k_big_*); what neither covers falls back to LSD."""
    rng = np.random.default_rng(n)
    if kind == "uniform27":
        keys = rng.integers(0, 1 << 27, n, dtype=np.uint64)
    elif kind == "uniform20":
        keys = rng.integers(0, 1 << 20, n, dtype=np.uint64)
    elif kind == "uniform32":
        keys = rng.integers(0, (1 << 32) - 1, n, dtype=np.uint64)
    elif kind == "zipf":
        keys = (rng.zipf(1.2, n) % (1 << 27)).astype(np.uint64)
    elif kind == "few_keys":
        keys = rng.integers(0, 100, n, dtype=np.uint64)
    elif kind == "heavy_in_sparse":   # 30 % one key, a few keys of 5-20 K tuples, the rest uniform over 2^27
        keys = rng.integers(0, 1 << 27, n, dtype=np.uint64)
        keys[rng.random(n) < 0.3] = 77_777_777
        for k in range(12):
            keys[rng.choice(n, 5000 + 1500 * k, replace=False)] = 1_000_003 * (k + 1)
    elif kind == "zipf_dense":        # config 4's shape: Zipf(1.2) ranks scattered over the key range
        perm_mul = 48_271
        keys = ((rng.zipf(1.2, n) % n) * perm_mul % (1 << 26)).astype(np.uint64)
    elif kind == "one_key_plus":      # 99 % one key
        keys = rng.integers(0, 1 << 24, n, dtype=np.uint64)
        keys[rng.random(n) < 0.99] = 123_456
    else:
        keys = rng.permutation(n).astype(np.uint64)
    ids = np.arange(n, dtype=U64)
    t = engine.tuples_from_host(keys, ids)
    engine.sort_tuples(t)
    assert engine.is_sorted(t)
    k, p = engine.tuples_to_host(t)
    _assert_sorted_run(k, p, keys, ids)
    engine.tuples_free(t)


def test_arena_returns_to_empty(engine):
    """Every temporary of the operators goes back to the engine's HBM arena (Scratch scopes cover the
    error paths too): after the handles are freed nothing is in use."""
    e = engine
    rng = np.random.default_rng(9)
    n = 1_500_000
    e.upload_column(70, 0, np.arange(n, dtype=np.uint64))
    e.upload_column(70, 1, rng.integers(0, n, n, dtype=np.uint64))
    e.upload_column(71, 1, rng.integers(0, n, n, dtype=np.uint64))
    e.sync()
    _, used0 = e.mempool_stats()
    ids = e.filter_scan(70, 0, "<", n // 2)
    tl, tr = e.build_tuples(70, 1, ids), e.build_tuples(71, 1)
    e.sort_tuples(tl); e.sort_tuples(tr)
    a, b = e.merge_join(tl, tr)
    da, db = e.distinct_pairs(a, b)
    sums = e.checksum(a, 70, [0, 1])
    assert len(sums) == 2
    for h in (ids, a, b, da, db):
        e.rowids_free(h)
    e.tuples_free(tl); e.tuples_free(tr)
    e.sync()
    _, used1 = e.mempool_stats()
    assert used1 == used0


def test_worker_contexts_run_concurrently(engine):
    """SURVEY 8f-3: engine contexts (stream + scratch + arena each), one bound per host thread; the same
    operators from four threads at once give the single-threaded answers."""
    import ctypes as C
    import threading
    e = engine
    rng = np.random.default_rng(5)
    n = 400_000
    for c in range(2):
        e.upload_column(80, c, rng.integers(0, 1000, n, dtype=np.uint64))
        e.upload_column(81, c, rng.integers(0, 1000, n, dtype=np.uint64))
    col = [rng.integers(0, 1000, n, dtype=np.uint64) for _ in range(4)]  # not used on the device: reference answers
    want = {}
    for thr in (100, 300, 500, 700):
        ids = e.filter_scan(80, 0, "<", thr)
        want[thr] = (e.rowids_count(ids), e.checksum(ids, 80, [0, 1]))
        e.rowids_free(ids)
    ctxs = [e.lib.qce_ctx_create() for _ in range(4)]
    assert all(ctxs)
    got, errs = {}, []

    def work(ctx, thr):
        try:
            assert e.lib.qce_ctx_bind(ctx) == 0
            for _ in range(20):
                ids = e.filter_scan(80, 0, "<", thr)
                got[thr] = (e.rowids_count(ids), e.checksum(ids, 80, [0, 1]))
                e.rowids_free(ids)
            e.lib.qce_ctx_bind(None)
        except Exception as ex:  # noqa: BLE001
            errs.append(repr(ex))
    ts = [threading.Thread(target=work, args=(ctxs[i], thr)) for i, thr in enumerate((100, 300, 500, 700))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for c in ctxs:
        e.lib.qce_ctx_destroy(c)
    assert not errs, errs
    assert got == want


def test_sorted_run_cache_is_per_batch(engine):
    """Inside one batch the sorted run of a whole base column is built once and borrowed afterwards;
    nothing survives qce_batch_end."""
    import ctypes as C
    e = engine
    rng = np.random.default_rng(6)
    n = 300_000
    e.upload_column(82, 0, rng.integers(0, n, n, dtype=np.uint64))
    h0, m0 = C.c_uint64(), C.c_uint64()
    e.lib.qce_batch_cache_stats(C.byref(h0), C.byref(m0))
    assert e.lib.qce_batch_begin() == 0
    runs = []
    for _ in range(3):
        t = e.build_tuples(82, 0)
        e.sort_tuples(t)
        assert e.is_sorted(t)
        runs.append(t)
    k0, p0 = e.tuples_to_host(runs[0])
    k2, p2 = e.tuples_to_host(runs[2])
    np.testing.assert_array_equal(k0, k2)
    np.testing.assert_array_equal(p0, p2)
    for t in runs:
        e.tuples_free(t)
    assert e.lib.qce_batch_end() == 0
    h1, m1 = C.c_uint64(), C.c_uint64()
    e.lib.qce_batch_cache_stats(C.byref(h1), C.byref(m1))
    assert h1.value - h0.value == 2 and m1.value - m0.value == 1
    t = e.build_tuples(82, 0)   # outside a batch: built afresh, not sorted yet
    assert not e.is_sorted(t) or n < 2
    e.tuples_free(t)
