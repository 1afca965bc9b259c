"""GPU parity of the wide exchange primitives (keys >= 2^32: SoA u64 keys + u32 row ids) on ONE GPU,
the local window presented as `world` ranks (qce_xwin_loopback): the histogram of key - base,
k_push_wide into every destination's key and id regions as qce_exchange_plan lays them out, and the
received run viewed in the window and sorted, each against numpy."""
import numpy as np
import pytest

import qce_b200
from qce_b200 import engine as eng_mod

pytestmark = pytest.mark.gpu
U64 = np.uint64
WIN = 64 << 20
TOP = (1 << 64) - 1


@pytest.fixture(scope="module")
def xeng(engine):
    engine.xwin_create(WIN)
    yield engine
    engine.xwin_destroy()


def _keys(kind, n, rng):
    if kind == "uniform":
        k = rng.integers(0, TOP, n, dtype=np.uint64, endpoint=True)
        return k | U64(1 << 63) if n == 1 else k      # a lone key stays >= 2^32
    if kind == "offset":
        return U64(1 << 40) + rng.integers(0, 1 << 20, n, dtype=np.uint64)
    if kind == "ends":
        k = rng.integers(0, TOP, n, dtype=np.uint64, endpoint=True)
        k[: min(n, 2)] = np.array([0, TOP], dtype=U64)[: min(n, 2)]
        if n == 1:
            k[0] = TOP
        return k
    if kind == "heavy":
        k = U64(1 << 40) + rng.integers(0, 1 << 36, n, dtype=np.uint64)
        k[rng.random(n) < 0.3] = U64((1 << 40) + 12345)
        return k
    raise ValueError(kind)


def _bitlen(v):
    return int(v).bit_length()


@pytest.mark.parametrize("kind", ["uniform", "offset", "ends", "heavy"])
@pytest.mark.parametrize("n", [0, 1, 33, 4095, 4096, 4097, 100003, 1 << 20])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_push_wide_loopback(xeng, world, n, kind):
    e = xeng
    e.xwin_loopback(world)
    per = WIN // world // 4096 * 4096
    rng = np.random.default_rng(n * 7 + world + len(kind))
    keys = _keys(kind, n, rng)
    ids = rng.permutation(n).astype(U64)
    t = e.tuples_from_host(keys, ids)
    base = int(keys.min()) if n else 0
    kmax = int(keys.max()) if n else 0
    width = max(1, _bitlen(kmax - base))
    shift = max(width - 8, 0)
    hist = e.key_histogram_wide(t, base, width)
    offs = keys - U64(base)
    bins = ((offs >> U64(shift)) & U64(255)).astype(np.int64)
    np.testing.assert_array_equal(hist, np.bincount(bins, minlength=256).astype(U64))

    # this process is rank 0 of `world` ranks and holds every tuple
    H = np.zeros((world, 1, 256), dtype=U64)
    H[0, 0] = hist
    sp, recv, before, run_off, col_off, need, _ = eng_mod.exchange_plan(e.lib, H, world, 0, [1], width)
    assert need <= per
    bnd = np.array([256 if s == TOP else s >> shift for s in sp], dtype=np.int64)
    part = np.searchsorted(bnd, bins, side="right")
    words = run_off[0] // U64(8) + before[0]
    id_at = col_off[0] // U64(4) + before[0]
    e.push_tuples_wide(t, base, width, sp, world, words, id_at)
    e.sync()
    for d in range(world):
        want = part == d
        cnt = int(recv[0, d])
        assert cnt == int(want.sum())
        # the key range of destination d, as the exchange hands it to the view
        span = kmax - base
        c0 = sp[d - 1] if d > 0 else 0
        c1 = sp[d] if d < world - 1 else TOP
        lo = base + min(c0, span)
        hi = kmax if (c1 == TOP or c1 > span) else base + c1 - 1
        v = e.tuples_from_window_wide((per * d + int(run_off[0, d])) // 8, (per * d + int(col_off[0, d])) // 4, cnt,
                                      n, lo, max(lo, hi))
        k, p = e.tuples_to_host(v)
        got, exp = np.lexsort((p, k)), np.lexsort((ids[want], keys[want]))
        np.testing.assert_array_equal(k[got], keys[want][exp])      # the (key, id) multiset of the partition
        np.testing.assert_array_equal(p[got], ids[want][exp])
        if cnt:
            assert lo <= int(k.min()) and int(k.max()) <= hi
        e.sort_tuples(v)
        k2, p2 = e.tuples_to_host(v)
        np.testing.assert_array_equal(k2, np.sort(keys[want]))       # sorted over the low bitlen(lo ^ hi) bits only
        o = np.lexsort((p2, k2))
        np.testing.assert_array_equal(p2[o], ids[want][exp])
        e.tuples_free(v)
    e.tuples_free(t)


def test_wide_misuse_is_reported(xeng):
    e = xeng
    e.xwin_loopback(2)
    packed = e.tuples_from_host(np.arange(10, dtype=U64), np.arange(10, dtype=U64))
    with pytest.raises(qce_b200.EngineError, match="wide runs"):
        e.key_histogram_wide(packed, 0, 8)
    with pytest.raises(qce_b200.EngineError, match="wide runs"):
        e.push_tuples_wide(packed, 0, 8, [128], 2, np.zeros(2, dtype=U64), np.zeros(2, dtype=U64))
    e.tuples_free(packed)
    keys = U64(1 << 40) + np.arange(5000, dtype=U64)
    t = e.tuples_from_host(keys, np.arange(5000, dtype=U64))
    e.key_histogram_wide(t, 1 << 40, 13)
    with pytest.raises(qce_b200.EngineError, match="not on a boundary"):
        e.push_tuples_wide(t, 1 << 40, 13, [5], 2, np.zeros(2, dtype=U64), np.zeros(2, dtype=U64))
    per = WIN // 2 // 4096 * 4096
    with pytest.raises(qce_b200.EngineError, match="overrun"):   # the ids would run past rank 1's slice
        e.push_tuples_wide(t, 1 << 40, 13, [1 << 5], 2, np.zeros(2, dtype=U64), np.array([0, per // 4 - 8], dtype=U64))
    with pytest.raises(qce_b200.EngineError, match="exceeds the exchange window"):
        e.tuples_from_window_wide(0, WIN // 4, 16)
    e.tuples_free(t)
