"""CPU: qce_split_plan, the exchange plan that may cut inside a heavy key (host arithmetic inside
libqce_b200.so, no device needed), on random key sets with planted heavy keys.  The tuples are
real keys per (source rank, side), so the sub-histograms the plan asks for and every count it
returns are checked against the tuples themselves, routed the way the split push routes them:
a key's destination is the number of cuts at or below it, an outer tuple of a split key goes by
its global position in the key's group, an inner one goes to every rank of the key's span."""
import numpy as np
import pytest

import qce_b200
from qce_b200 import engine as eng_mod


def _keys(rng, world, key_bits, n, heavy):
    """keys[s][side]: uniform keys plus, per (key, outer share, inner count), planted copies"""
    top = 1 << key_bits
    out = []
    for s in range(world):
        sides = []
        for side in range(2):
            k = rng.integers(0, top, int(rng.integers(n // 2, n + 1)), dtype=np.int64)
            extra = [np.full(int(share * n) if side == 0 else inner, key, dtype=np.int64)
                     for key, share, inner in heavy]
            sides.append(np.concatenate([k] + extra))
        out.append(sides)
    return out


def _hist(keys, key_bits):
    shift = max(key_bits - 8, 0)
    return np.array([[np.bincount(k >> shift, minlength=256)[:256] for k in side] for side in keys], dtype=np.uint64)


def _sub(keys, prefixes, shift):
    H = np.zeros((len(keys), 2, len(prefixes), 256), dtype=np.uint64)
    for s, sides in enumerate(keys):
        for side, k in enumerate(sides):
            for j, p in enumerate(prefixes):
                sel = k[(k >> shift) == p]
                H[s, side, j] = np.bincount((sel >> max(shift - 8, 0)) & ((1 << min(shift, 8)) - 1), minlength=256)[:256]
    return H


def _route(keys, plan, world):
    """count[side][source][dest] of the tuples, routed by the plan's cuts"""
    cut_key, cut_q = plan["cut_key"].astype(np.int64), plan["cut_q"].astype(np.int64)
    thr = np.where(cut_q == 0, cut_key, cut_key + 1)
    split = {int(k): j for j, k in enumerate(plan["split_key"])}
    C = np.zeros((2, world, world), dtype=np.int64)
    pre = {k: 0 for k in split}
    for s in range(world):
        for side in range(2):
            k = keys[s][side]
            d = np.searchsorted(np.sort(thr), k, side="right")
            plain = ~np.isin(k, list(split)) if split else np.ones(len(k), bool)
            C[side, s] += np.bincount(d[plain], minlength=world)[:world]
            for key, j in split.items():
                first, last = int(plan["split_first"][j]), int(plan["split_last"][j])
                cnt = int((k == key).sum())
                if side == 1:
                    C[1, s, first:last + 1] += cnt
                    continue
                at = cut_q[(cut_key == key) & (cut_q > 0)]           # global quotas of the span
                idx = pre[key] + np.arange(cnt)
                dd = first + np.searchsorted(at, idx, side="right")
                C[0, s] += np.bincount(dd, minlength=world)[:world]
                bound = plan["split_bound"][j, s, :last - first + 1].astype(np.int64)
                np.testing.assert_array_equal(bound, np.clip(np.concatenate([[0], at]) - pre[key], 0, cnt))
                pre[key] += cnt
    return C


def _check_cuts(keys, plan, world):
    """Every cut lands within share / 20 of its target k * T / W in the stream of tuples ordered by key
    (a key's inner tuples before its outer ones), unless the target falls inside a key that cannot be
    cut there -- fewer than two outer tuples, or the target inside the key's inner group -- and then the
    cut is at that key's nearer end.  Restated from the tuples, not from the plan's pieces."""
    outer = np.concatenate([keys[s][0] for s in range(world)])
    inner = np.concatenate([keys[s][1] for s in range(world)])
    uk = np.union1d(outer, inner)
    r = np.bincount(np.searchsorted(uk, outer), minlength=len(uk)).astype(np.int64)
    s = np.bincount(np.searchsorted(uk, inner), minlength=len(uk)).astype(np.int64)
    cum = np.concatenate([[0], np.cumsum(r + s)])
    T = int(cum[-1])
    tol = T / (20 * world)
    for k, (key, q) in enumerate(zip(plan["cut_key"].astype(np.int64), plan["cut_q"].astype(np.int64))):
        i = int(np.searchsorted(uk, key))
        pos = cum[i] + (s[i] + q if q else 0)
        t = T * (k + 1) / world
        j = int(np.searchsorted(cum, t, side="left")) - 1   # the key whose tuples hold the target
        cuttable = r[j] >= 2 and cum[j] + s[j] < t < cum[j] + s[j] + r[j]
        allowed = tol if cuttable else max(tol, min(t - cum[j], cum[j + 1] - t))
        assert abs(pos - t) <= allowed + 1, (k, key, q, pos, t, allowed)


CASES = {
    "one key over several shares": (20, [(77_777, 3.0, 3)]),
    "two adjacent heavy keys": (24, [(1 << 20, 1.5, 5), ((1 << 20) + 1, 1.2, 0)]),
    "heavy last bin": (32, [((1 << 32) - 1, 2.0, 2)]),
    "heavy both sides": (28, [(12_345_678, 1.0, 200)]),
    "uniform": (32, []),
    "tiny keys": (5, [(3, 0.8, 1)]),
}


@pytest.mark.parametrize("world", [2, 3, 8, 16])
@pytest.mark.parametrize("case", sorted(CASES))
def test_split_plan(world, case):
    lib = qce_b200.load_library()
    key_bits, heavy = CASES[case]
    rng = np.random.default_rng(world * 31 + len(case))
    n = 3000
    keys = _keys(rng, world, key_bits, n, heavy)
    H = _hist(keys, key_bits)
    ncols = [1, 2]
    plans = [eng_mod.split_plan(lib, H, world, r, ncols, key_bits, lambda p, sh: _sub(keys, p, sh)) for r in range(world)]
    p0 = plans[0]
    for p in plans[1:]:   # every rank derives the same plan; only `before` and `sent` are the rank's own
        for f in ("cut_key", "cut_q", "count", "recv", "run_off", "col_off", "key_lo", "key_hi", "split_bound"):
            np.testing.assert_array_equal(p[f], p0[f], err_msg=f)
        assert p["window_bytes"] == p0["window_bytes"] and p["levels"] == p0["levels"]
    C = p0["count"].astype(np.int64)
    np.testing.assert_array_equal(_route(keys, p0, world), C)
    for r, p in enumerate(plans):   # the segments of the sources tile each destination's run
        np.testing.assert_array_equal(p["before"].astype(np.int64), C[:, :r, :].sum(axis=1))
        np.testing.assert_array_equal(p["sent"].astype(np.int64), C[:, r, :].sum(axis=1) - C[:, r, r])
    np.testing.assert_array_equal(p0["recv"].astype(np.int64), C.sum(axis=1))
    top = np.zeros(world, dtype=np.int64)
    for side in range(2):
        np.testing.assert_array_equal(p0["run_off"][side].astype(np.int64), top)
        top = (top + 8 * C[side].sum(axis=0) + 15) // 16 * 16
        for _ in range(ncols[side]):
            top = (top + 4 * C[side].sum(axis=0) + 15) // 16 * 16
    assert p0["window_bytes"] == top.max()
    total = sum(len(k) for sides in keys for k in sides)
    copies = 0
    for j, key in enumerate(p0["split_key"]):   # a split key: quotas sum to its count, its inner group on every rank
        span = int(p0["split_last"][j] - p0["split_first"][j] + 1)
        outer = sum(int((keys[s][0] == key).sum()) for s in range(world))
        inner = sum(int((keys[s][1] == key).sum()) for s in range(world))
        assert span >= 2 and outer >= 2
        assert int(p0["split_count"][j, :, 0].sum()) == outer and int(p0["split_count"][j, :, 1].sum()) == inner
        first, last = int(p0["split_first"][j]), int(p0["split_last"][j])
        assert C[0, :, first:last + 1].sum() >= outer
        copies += inner * (span - 1)
        assert (p0["key_lo"][first + 1:last + 1] == key).all() and (p0["key_hi"][first:last] == key).all()
    assert C.sum() == total + copies
    if p0["refined"]:
        _check_cuts(keys, p0, world)
    # bins within 10 %: the plan is qce_exchange_plan's, exactly
    sp, recv, before, run_off, col_off, need, sent = eng_mod.exchange_plan(lib, H, world, 0, ncols, key_bits)
    bins_ok = max(recv.sum(axis=0)) <= 1.10 * total / world
    assert bool(p0["refined"]) == (not bins_ok)
    if bins_ok:
        assert p0["levels"] == 0 and p0["nsplit"] == 0 and list(p0["cut_key"]) == sp and not p0["cut_q"].any()
        np.testing.assert_array_equal(p0["recv"], recv)
        np.testing.assert_array_equal(p0["run_off"], run_off)
        np.testing.assert_array_equal(p0["col_off"], col_off)
        assert p0["window_bytes"] == need
    assert len(p0["requests"]) == p0["levels"] and all(k <= 15 for k, _ in p0["requests"])


def test_split_plan_cuts_a_key_over_several_shares():
    """One key on 60 % of R at 8 ranks: its outer group spans at least 3 ranks, within 10 % of a share."""
    lib = qce_b200.load_library()
    world, key_bits = 8, 21
    rng = np.random.default_rng(5)
    keys = _keys(rng, world, key_bits, 20_000, [(1_000_003, 1.5, 1)])
    p = eng_mod.split_plan(lib, _hist(keys, key_bits), world, 0, [0, 0], key_bits, lambda q, sh: _sub(keys, q, sh))
    assert p["refined"] and p["levels"] >= 1 and p["nsplit"] == 1
    assert p["split_last"][0] - p["split_first"][0] + 1 >= 3
    total = sum(len(k) for sides in keys for k in sides)
    assert p["count"].sum(axis=(0, 1)).max() <= 1.10 * total / world + world


def test_split_plan_keeps_an_inner_only_heavy_key_whole():
    """A key heavy on the inner side with one outer tuple is never split (its outer tuple's match count
    would spread over ranks)."""
    lib = qce_b200.load_library()
    world, key_bits = 4, 16
    rng = np.random.default_rng(9)
    keys = [[rng.integers(0, 1 << 16, 2000), np.concatenate([rng.integers(0, 1 << 16, 2000), np.full(20_000, 4242)])]
            for _ in range(world)]
    keys[0][0] = np.concatenate([keys[0][0], [4242]])
    p = eng_mod.split_plan(lib, _hist(keys, key_bits), world, 1, [0, 0], key_bits, lambda q, sh: _sub(keys, q, sh))
    assert p["refined"] and 4242 not in list(p["split_key"])
    np.testing.assert_array_equal(_route(keys, p, world), p["count"].astype(np.int64))
