"""CPU: qce_exchange_plan at the widths of a wide exchange (keys >= 2^32 binned by key - base over
33..64 bits) against a numpy restatement whose splitters are Python ints, so that the cut past the
last bin at 64 bits is 2^64 there and cannot wrap.  The engine returns that cut as 2^64 - 1."""
import numpy as np
import pytest

import qce_b200
from qce_b200 import engine as eng_mod
from tests.helpers import choose_splitters

TOP = (1 << 64) - 1


def _restated(H, world, rank, ncols, width):
    nsides = len(ncols)
    splitters = choose_splitters(H.sum(axis=(0, 1)), width, world)     # Python ints: 2^64 stays 2^64
    shift = max(width - 8, 0)
    bnd = [0] + [min(s >> shift, 256) for s in splitters] + [256]
    Hc = np.zeros((world, nsides, 257), dtype=np.int64)
    np.cumsum(H.astype(np.int64), axis=2, out=Hc[:, :, 1:])
    C = (Hc[:, :, bnd[1:]] - Hc[:, :, bnd[:-1]]).transpose(1, 0, 2)   # C[side, src, dst]
    recv = C.sum(axis=1)
    before = (np.cumsum(C, axis=1) - C)[:, rank, :]
    run_off, col_off = [], []
    top = np.zeros(world, dtype=np.int64)
    for k in range(nsides):
        run_off.append(top)
        top = (top + 8 * recv[k] + 15) // 16 * 16
        for _ in range(ncols[k]):
            col_off.append(top)
            top = (top + 4 * recv[k] + 15) // 16 * 16
    return splitters, recv, before, np.array(run_off), np.array(col_off).reshape(-1, world), int(top.max()), C


def _part(offset, splitters):
    """destination of a key offset under the engine's splitters (2^64 - 1 stands for the cut 2^64)"""
    return sum(offset >= (1 << 64 if s == TOP else s) for s in splitters)


@pytest.mark.parametrize("world", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("width", [33, 40, 56, 57, 63, 64])
def test_wide_exchange_plan_matches_restatement(world, width):
    lib = qce_b200.load_library()
    rng = np.random.default_rng(world * 1000 + width)
    for trial in range(6):
        nsides = int(rng.integers(1, 3))
        ncols = [1] * nsides                        # a wide side: its ids follow its keys as one column
        H = rng.integers(0, 50_000, (world, nsides, 256)).astype(np.uint64)
        if trial == 1:
            H[:, :, 10:] = 0                          # everything in a few bins: later parts are empty
        if trial == 2:
            H[:] = 0                                  # empty runs
        if trial == 3:
            H[:, :, 7] += np.uint64(10 ** 7)          # one heavy bin
        if trial == 4:
            H[:, :, 255] += np.uint64(10 ** 7)        # heavy last bin: the cuts land at bin 256
        layouts = []
        for rank in range(world):
            sp, recv, before, run_off, col_off, need, sent = eng_mod.exchange_plan(lib, H, world, rank, ncols, width)
            esp, erecv, ebefore, erun, ecol, eneed, C = _restated(H, world, rank, ncols, width)
            assert sp == [min(s, TOP) for s in esp]
            assert all(s <= 1 << width or s == TOP for s in sp)
            np.testing.assert_array_equal(recv.astype(np.int64), erecv)
            np.testing.assert_array_equal(before.astype(np.int64), ebefore)
            np.testing.assert_array_equal(run_off.astype(np.int64), erun)
            np.testing.assert_array_equal(col_off.astype(np.int64), ecol)
            assert need == eneed
            layouts.append((sp, recv.tobytes(), run_off.tobytes(), col_off.tobytes()))
            # the offsets at both ends of the key range land where the restatement puts them
            for off in (0, (1 << width) - 1, 1 << (width - 1)):
                assert _part(off, sp) == sum(off >= s for s in esp)
        assert all(l == layouts[0] for l in layouts)   # every rank derives the same plan
        for k in range(nsides):
            for d in range(world):
                starts = [int(eng_mod.exchange_plan(lib, H, world, r, ncols, width)[2][k, d]) for r in range(world)]
                sizes = [int(C[k, r, d]) for r in range(world)]
                assert starts == list(np.cumsum([0] + sizes[:-1]))   # segments tile the destination's run
                assert sum(sizes) == int(erecv[k, d])


def test_width_64_ends_and_wrap():
    """Keys 0 and 2^64 - 1 both present at width 64: bin 0 and bin 255 are both populated; with the
    weight on the last bin every cut lies at 2^64, which the engine returns as 2^64 - 1 (never 0)."""
    lib = qce_b200.load_library()
    world = 3
    H = np.zeros((world, 1, 256), dtype=np.uint64)
    H[0, 0, 0] = 5           # key 0
    H[2, 0, 255] = 10 ** 6   # key 2^64 - 1 (bin 255 = offsets >= 255 << 56)
    sp, recv, *_ = eng_mod.exchange_plan(lib, H, world, 0, [1], 64)
    assert sp == [TOP, TOP]
    assert _part(0, sp) == 0 and _part(TOP, sp) == 0   # everything on rank 0: the cuts lie past every key
    assert [int(x) for x in recv[0]] == [10 ** 6 + 5, 0, 0]
    H[0, 0, 0] = 10 ** 6
    sp, recv, *_ = eng_mod.exchange_plan(lib, H, world, 0, [1], 64)
    assert sp == [1 << 56, TOP]
    assert _part(0, sp) == 0 and _part(TOP, sp) == 1
    assert [int(x) for x in recv[0]] == [10 ** 6, 10 ** 6, 0]


@pytest.mark.parametrize("bad", [0, 65])
def test_width_out_of_range_is_refused(bad):
    lib = qce_b200.load_library()
    with pytest.raises(qce_b200.EngineError, match="1..64"):
        eng_mod.exchange_plan(lib, np.zeros((2, 1, 256), dtype=np.uint64), 2, 0, [1], bad)
