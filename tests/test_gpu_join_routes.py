"""The merge join (qce_merge_join, _stats, _walk, qce_rejoin) route by route, against the oracle's merge.

merge_join_any -> merge_join_t -> merge_join_fused_t (csrc/qce_engine.cu) and the kernels of csrc/k_join.cuh pick
a route at four levels: the template instance by the key width of each run; the kernel sequence (single-pass,
two-phase or walk); per 2048-tuple R tile the bounds path (empty window, count table, staged search, bisection,
interpolated guess + gallop); and per tile of the single-pass kernel how its pairs are written (light, heavy,
deferred for size, deferred past the output guess).  `plan` restates that choice in numpy from the two runs as the
engine holds them.  The CPU test holds every case to the routes its label names and checks that every route has a
case, so a moved threshold shows up here first.  The GPU test joins every case in a fresh process per switch set
and checks the pairs (byte-equal to the oracle: R-major, S in run order), the min / max matches per outer tuple
that re-join elision relies on, the launch profile against the plan, and that the arena is balanced afterwards.
qce_distinct_pairs, which follows a join with distinct=True, is planned and checked the same way.
"""
import functools
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from tests.test_gpu_sort_routes import SORT_SWITCHES, _sw
from tests.test_gpu_sort_routes import plan as sort_plan

U64 = np.uint64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOP = (1 << 64) - 1

# ---- constants of the route choice -------------------------------------------------------------------------------
JTILE = 2048            # k_join.cuh:28   QCE_JTILE: R tuples per tile
JWIN = 4096             # k_join.cuh:30   QCE_JWIN: S window staged in shared memory
JCHUNK = 4096           # k_join.cuh:32   QCE_JCHUNK: output pairs per k_join_write CTA
JINTERP_MIN = 65536     # k_join.cuh:99   QCE_JINTERP_MIN: windows from here on take the guess + gallop search
JTAB = 8190             # k_join.cuh:160  QCE_JTAB: count table for tiles whose keys span less than this
JTAB_WIN = 16 * JTILE   # k_join.cuh:190, :331  ... and whose window holds at most this many S tuples
JFUSE_MAX = 16384       # k_join.cuh:289  QCE_JFUSE_MAX: single-pass tiles with more pairs are deferred
HEAVY = 16              # k_join.cuh:425  a tuple with more matches makes its tile "heavy"
SCAN_WARP_MAX = 512     # qce_engine.cu:880, :946  tile scans of up to 512 tiles run in one warp
ROWID_LIMIT = 1 << 32   # qce_engine.cu:863, :966  joins of 2^32 pairs or more are refused
SORT_TILE = 4096        # qce_engine.cu:450  BS_TILE: distinct_pairs sorts up to this many pairs in one CTA

JOIN_SWITCHES = ("QCE_JOIN_FUSED", "QCE_JOIN_CAP", "QCE_JOIN_TICKET", "QCE_JOIN_MINB")
JOIN_TAGS = ("join_partition", "join_fused", "join_bounds", "join_write", "scan_tiles", "join_keymax",
             "join_bounds_walk")
DISTINCT_TAGS = ("pack_pairs", "block_sort", "radix_hist", "onesweep_k", "unique_mask")

INSTANCES = ["nn", "wn", "nw", "ww"]                 # <WR, WS>: n = narrow (keys < 2^32), w = wide
SEQUENCES = ["fused", "two_phase", "walk", "no_launch"]
BOUNDS = ["b_empty", "b_table", "b_staged", "b_bisect", "b_gallop"]
WRITES = ["w_light", "w_heavy", "w_size", "w_cap"]
ROUTES = INSTANCES + SEQUENCES + BOUNDS + WRITES + ["scan_warp", "scan_block", "refused", "uniform"]
DISTINCT_ROUTES = ["d_none", "d_block", "d_onesweep"]


def switches(env):
    return {"fused": _sw(env, "QCE_JOIN_FUSED", 1), "cap": _sw(env, "QCE_JOIN_CAP", 0)}


def bounds_path(wn, span):
    """k_join_bounds / k_join_fused: the search a tile takes from its S window wn and its key span khi - klo."""
    if wn == 0:
        return "b_empty"
    if span < JTAB and wn <= JTAB_WIN:
        return "b_table"
    if wn <= JWIN:
        return "b_staged"
    return "b_bisect" if wn < JINTERP_MIN else "b_gallop"


def write_mode(tot, cmax, gbase, cap):
    """k_join_fused: how a tile's pairs are written."""
    if tot > JFUSE_MAX:
        return "w_size"
    if gbase + tot > cap:
        return "w_cap"
    return "w_heavy" if cmax > HEAVY else "w_light"


def run_of(keys, skewed=False):
    """A sorted (or, for the walk, outer) run as the join sees it: its keys, width and skew flag."""
    keys = np.asarray(keys, dtype=U64)
    return {"keys": keys, "wide": bool(len(keys)) and int(keys.max()) >= (1 << 32), "skewed": skewed}


def plan(R, S, env, walk=False, stats=False):
    """The route merge_join_any takes for runs R, S (see run_of) under the switches in `env`: a dict with the
    instance, the kernel launches {tag: n}, per tile the window, bounds path and write mode, the pair count m, the
    deferred chunk count, min / max matches per outer tuple, and `routes`, the set of labels it hits."""
    assert not (walk and stats), "the walk's stats launch runs only in the sharded join"
    sw = switches(env)
    kR, kS = R["keys"], S["keys"]
    nR, nS = len(kR), len(kS)
    inst = ("w" if R["wide"] else "n") + ("w" if S["wide"] else "n")
    out = {"instance": inst, "nR": nR, "nS": nS, "m": 0, "min": 0, "max": 0, "chunks": 0, "refused": False,
           "tags": {}, "routes": {inst}}
    if nR == 0 or nS == 0:
        out["routes"].add("no_launch")
        return out
    lb = np.searchsorted(kS, kR, side="left").astype(np.int64)
    cnt = np.searchsorted(kS, kR, side="right").astype(np.int64) - lb
    if walk:  # the reference's pointer walk: a tuple matches iff its key is >= every earlier key of R
        ok = np.ones(nR, dtype=bool)
        ok[1:] = kR[1:] >= np.maximum.accumulate(kR)[:-1]
        cnt = np.where(ok, cnt, 0)
    out["lb"], out["cnt"] = lb, cnt
    starts = np.arange(0, nR, JTILE)
    ntiles = len(starts)
    tot = np.add.reduceat(cnt, starts)
    cmax = np.maximum.reduceat(cnt, starts)
    m = int(tot.sum())
    out.update(m=m, min=int(cnt.min()), max=int(cnt.max()), refused=m >= ROWID_LIMIT, ntiles=ntiles,
               tile_total=tot.tolist())
    if out["min"] == out["max"]:
        out["routes"].add("uniform")
    chunks = -(-tot // JCHUNK)
    if walk:
        seq = "walk"
        tags = {"join_keymax": 2, "join_bounds_walk": 1, "scan_tiles": 2}
    else:
        last = np.minimum(starts + JTILE, nR) - 1
        klo, khi = kR[starts], kR[last]
        win_lo = np.searchsorted(kS, klo, side="left")
        wn = np.searchsorted(kS, khi, side="right") - win_lo
        paths = [bounds_path(int(w), int(s)) for w, s in zip(wn, khi - klo)]
        out.update(window=wn.tolist(), paths=paths)
        out["routes"].update(paths)
        if sw["fused"] and not R["skewed"] and not S["skewed"]:
            seq = "fused"
            cap = sw["cap"] if sw["cap"] > 0 else max(nR, nS)
            gbase = np.cumsum(tot) - tot
            modes = [write_mode(int(t), int(c), int(g), cap) for t, c, g in zip(tot, cmax, gbase)]
            out.update(cap=cap, gbase=gbase.tolist(), writes=modes)
            out["routes"].update(modes)
            chunks = np.where([w in ("w_size", "w_cap") for w in modes], chunks, 0)
            tags = {"join_partition": 1, "join_fused": 1}
            if int(chunks.sum()) and not out["refused"]:
                tags.update(scan_tiles=1, join_write=1)
        else:
            seq = "two_phase"
            tags = {"join_partition": 1, "join_bounds": 1, "scan_tiles": 2}
    if seq != "fused" and m > 0 and not out["refused"]:
        tags["join_write"] = 1
    out["chunks"] = int(chunks.sum())
    out["tags"] = tags
    out["routes"].add(seq)
    if out["refused"]:
        out["routes"].add("refused")
    if "scan_tiles" in tags:
        out["routes"].add("scan_warp" if ntiles <= SCAN_WARP_MAX else "scan_block")
    return out


def plan_distinct(pR, pS, boundR, boundS):
    """distinct_pairs: the sort of the packed pairs over the significant bits of both row-id columns (8-bit digits
    per side; an id bound of 0 = unknown = 32 bits)."""
    m = len(pR)
    if m == 0:
        return "d_none", {}, 0
    bits = lambda b: (b - 1).bit_length() if b else 32  # noqa: E731
    npass = -(-bits(boundS) // 8) + -(-bits(boundR) // 8)
    tags = {"pack_pairs": 1, "unique_mask": 1}
    if m <= 1 or npass == 0:
        route = "d_none"
    elif m <= SORT_TILE:
        route, tags["block_sort"] = "d_block", 1
    else:
        route = "d_onesweep"
        tags.update(radix_hist=1, onesweep_k=npass)
    return route, tags, npass


# ---- cases ---------------------------------------------------------------------------------------------------
# A case generator returns a dict: join kinds {"kR", "kS"} (keys in any order; row ids are assigned below),
# "sort": which runs the engine sorts itself ("R", "S"; the others are sorted here), rejoin {"driver", "last",
# "edit"}, distinct {"pR", "pS"}.
E = [0, (1 << 32) - 1, 1 << 32, 1 << 63, TOP]   # keys at the edges of the two widths


def _u(rng, n, lo, hi):
    return rng.integers(lo, hi, n, dtype=U64, endpoint=True)


def _a(*parts):
    return np.concatenate([np.asarray(p, dtype=U64) for p in parts])


def g_uniform(nR, nS, dom, pin=()):
    def g(rng):
        kS = _u(rng, nS, 0, dom - 1)
        kR = kS[:1].copy() if nR == 1 else _u(rng, nR, 0, dom - 1)
        kR[:len(pin)] = pin
        kS[:len(pin)] = pin
        return {"kR": kR, "kS": kS}
    return g


def g_span(span):
    """One tile whose keys span exactly `span`, over a window of about 2000 S tuples."""
    def g(rng):
        lo = 1_000_000
        kR = _u(rng, JTILE, lo, lo + span)
        kR[:2] = lo, lo + span
        return {"kR": kR, "kS": _u(rng, 3000, lo - 2000, lo + span + 2000)}
    return g


def g_win_table(w):
    """One tile over even keys 0..200 plus one odd key, a window of exactly w odd S keys: span 200."""
    def g(rng):
        kR = rng.integers(0, 101, JTILE, dtype=U64) * U64(2)
        kR[:3] = 0, 200, 101
        kS = _a(rng.integers(0, 100, w, dtype=U64) * U64(2) + U64(1), _u(rng, 500, 1000, 5000))
        return {"kR": kR, "kS": kS}
    return g


def g_win_search(w):
    """One tile over a span of 4 M keys and a window of exactly w S tuples (some of them R's keys)."""
    def g(rng):
        lo, hi = 5_000_000, 9_000_000
        kR = _u(rng, JTILE, lo, hi)
        kR[:2] = lo, hi
        kS = _a(rng.choice(kR, 300), _u(rng, w - 300, lo, hi), _u(rng, 400, 0, lo - 1), _u(rng, 400, hi + 1, hi + 10**6))
        return {"kR": kR, "kS": kS}
    return g


def g_gallop_top(rng):
    """Wide keys packed below 2^64 - 1 with uneven gaps and ties: windows of ~10^5 over the top of the range."""
    gaps = rng.integers(0, 1 << 44, 300_000, dtype=U64)
    gaps[rng.random(len(gaps)) < 0.1] = 0
    gaps[0] = 0
    kS = U64(TOP) - np.cumsum(gaps, dtype=U64)
    kR = _a(rng.choice(kS, 2000), _u(rng, 2000, int(kS.min()), TOP), [TOP, TOP, int(kS.min())])
    return {"kR": kR, "kS": kS}


def g_gallop_clusters(rng):
    """Three dense clusters far apart in the 64-bit range: the interpolated guess lands far from the answer."""
    kS = _a(_u(rng, 100_000, 1 << 32, 1 << 33), (1 << 63) + _u(rng, 100_000, 0, 1 << 20), _u(rng, 100_000, TOP - (1 << 30), TOP))
    kR = _a(rng.choice(kS, 3000), _u(rng, 1000, 1 << 32, TOP), [1 << 32, 1 << 63, TOP])
    return {"kR": kR, "kS": kS}


def g_gallop_mixed(rwide):
    """Windows of ~10^5 narrow keys; the R run (rwide) or the S run carries wide keys that match nothing."""
    def g(rng):
        kS = _u(rng, 150_000, 0, (1 << 32) - 1)
        kR = _a(rng.choice(kS, 1500), _u(rng, 1500, 0, (1 << 32) - 1), [0, (1 << 32) - 1])
        if rwide:
            kR = _a(kR, [1 << 32, TOP])
        else:
            kS = _a(kS, [1 << 32, TOP])
        return {"kR": kR, "kS": kS}
    return g


def g_gallop_one_key(wide):
    """A window of 70 000 copies of one key (ks0 == ks1: the interpolation scale is 0) matched by one R tuple."""
    def g(rng):
        if wide:
            kR = _a(_u(rng, JTILE - 1, 1 << 63, TOP - 1), [TOP])
            kS = _a(np.full(70_000, TOP, dtype=U64), _u(rng, 1000, 1 << 32, 1 << 62))
        else:
            kR = _a(rng.integers(0, 1 << 19, JTILE - 1, dtype=U64) * U64(2), [(1 << 19) + 1])
            kS = _a(np.full(70_000, (1 << 19) + 1, dtype=U64), _u(rng, 1000, 1 << 21, 1 << 22))
        return {"kR": kR, "kS": kS}
    return g


def g_matches(k):
    """One tile of distinct keys; one of them has k matches, the others at most a few."""
    def g(rng):
        kR = np.arange(JTILE, dtype=U64) * U64(3) + U64(10)
        others = np.delete(kR, 1000)
        return {"kR": kR, "kS": _a(rng.choice(others, 1500), np.full(k, kR[1000], dtype=U64))}
    return g


def g_tile_total(extra):
    """One tile whose 2048 tuples match 8 times each, plus `extra` more pairs on one tuple."""
    def g(rng):
        kR = np.arange(JTILE, dtype=U64) * U64(3)
        return {"kR": kR, "kS": _a(np.repeat(kR, 8), np.full(extra, kR[5], dtype=U64))}
    return g


CAP_EXACT = 10_000


def g_cap(last_extra):
    """Three tiles with 3000, 3000 and 4000 + last_extra pairs: under QCE_JOIN_CAP=10000 the last tile ends
    exactly at the guess, or one pair past it."""
    def g(rng):
        kR = np.arange(3 * JTILE, dtype=U64) * U64(2)
        hit = np.concatenate([np.arange(1000) + t * JTILE for t in range(3)])
        reps = np.repeat([3, 3, 4], 1000)
        reps[-1] += last_extra
        return {"kR": kR, "kS": np.repeat(kR[hit], reps)}
    return g


def g_edges(rw, sw_, disjoint=False):
    """Runs of each width with the edge keys 0, 2^32 - 1, 2^32, 2^63, 2^64 - 1 repeated.  A narrow run keeps the
    narrow ones.  disjoint: every narrow key lies below every wide key, so every window is empty."""
    narrow_e, wide_e = E[:2], E[2:]

    def side(rng, wide, other):
        if disjoint:
            return _a(_u(rng, 5000, 1 << 32, TOP), wide_e * 4) if wide else _a(_u(rng, 5000, 0, (1 << 32) - 1), narrow_e * 4)
        return _a(_u(rng, 5000, 0, TOP if (wide and other) else (1 << 32) - 1), (E if wide else narrow_e) * 4)

    def g(rng):
        kR = side(rng, rw, sw_)
        kS = side(rng, sw_, rw)
        if not disjoint:
            both = kR[kR < U64(1 << 32)] if not (rw and sw_) else kR
            kS = _a(kS, rng.choice(both, 1000), (E if sw_ else narrow_e) * 3)
        return {"kR": kR, "kS": kS}
    return g


def g_engine_sorted(side, n, dom):
    """A run of n tuples over [0, dom) that the engine sorts itself, against 20 000 tuples over the same keys."""
    def g(rng):
        big = _u(rng, n, 0, dom - 1)
        big[0] = dom - 1
        small = _u(rng, 20_000, 0, dom - 1)
        return {"kR": big, "kS": small, "sort": "R"} if side == "R" else {"kR": small, "kS": big, "sort": "S"}
    return g


def g_walk(order, rw, sw_):
    """The walk: an outer run in arbitrary order (random, descending, or ascending with dips across the tile
    boundaries) against a sorted inner run."""
    def g(rng):
        n = 7000
        hi = TOP if rw else (1 << 32) - 1
        if order == "random":
            kR = _a(_u(rng, n - 2, 0, 4999), [hi, 3])
        elif order == "desc":
            kR = np.sort(_a(_u(rng, n - 3, 0, hi), [hi, hi, hi]))[::-1].copy()
        else:
            kR = np.arange(n, dtype=U64) * U64(2) + U64(5000)
            kR[[700, 2047, 2048, 2049, 4095, 4096, 6000]] = U64(3000)
            if rw:
                kR[-1] = U64(TOP)
        kS = _a(_u(rng, 6000, 0, 5000 if order == "random" else 20_000), rng.choice(kR, 1500), [3, 3000])
        kS = kS[kS <= U64((1 << 32) - 1)] if not sw_ else _a(kS, [TOP, TOP, 1 << 40])
        return {"kR": kR, "kS": kS}
    return g


def g_uniform_k(k, step):
    """Every R tuple matches exactly k times; 5796 tuples, a partial last tile of 1700 that takes the same bounds
    path as the full ones."""
    def g(rng):
        kR = np.arange(2 * JTILE + 1700, dtype=U64) * U64(step) + U64(100)
        return {"kR": kR, "kS": np.repeat(kR, k)}
    return g


def g_rejoin(rng):
    """qce_rejoin with one driver row id repeated 20 000 times: its outer tiles defer."""
    last = _u(rng, 3000, 0, 4999)
    last[[10, 1500, 2999]] = 77
    return {"driver": _a(np.full(20_000, 77), _u(rng, 5000, 0, 4999)), "last": last, "edit": _u(rng, 3003, 0, 8999)}


def g_distinct(bound, m):
    def g(rng):
        pool = max(1, m // 3)
        a, b = _u(rng, pool, 0, bound - 1), _u(rng, pool, 0, bound - 1)
        a[0], b[-1] = bound - 1, bound - 1
        idx = rng.integers(0, pool, m)
        idx[:pool] = np.arange(pool)  # every pool pair occurs: the id bounds are exactly `bound`
        return {"pR": a[idx], "pS": b[idx]}
    return g


def g_old(i):
    """The six joins the single-pass kernel was first routed with."""
    def g(rng):
        u = lambda n, d: rng.integers(0, d, n, dtype=U64)  # noqa: E731
        return [lambda: {"kR": u(100_000, 100_000), "kS": u(100_000, 100_000)},
                lambda: {"kR": u(40_000, 3000), "kS": u(60_000, 3000)},
                lambda: {"kR": _a(np.full(3000, 77), u(5000, 1000)), "kS": _a(np.full(2000, 77), u(5000, 1000))},
                lambda: {"kR": u(4097, 50), "kS": u(200_000, 50)},
                lambda: {"kR": u(50_000, 1 << 34), "kS": u(50_000, 1 << 34)},
                lambda: {"kR": u(300_000, 1 << 20), "kS": u(1000, 1 << 20)}][i]()
    return g


BIG = SCAN_WARP_MAX * JTILE
CASES = {
    # outer run sizes at the tile edges and the tile-scan switch (a planted key defers one tile, so the scan runs)
    "nR_1": ("join", g_uniform(1, 6000, 4000)),
    **{"nR_%d" % n: ("join", g_uniform(n, 6000, 4000)) for n in (2047, 2048, 2049)},
    "nR_512x2048": ("join", g_uniform(BIG, 200_000, 1 << 21, pin=[777_777] * 150)),
    "nR_512x2048+1": ("join", g_uniform(BIG + 1, 200_000, 1 << 21, pin=[777_777] * 150)),
    # the bounds path at its edges
    "span_8189": ("join", g_span(JTAB - 1)),
    "span_8190": ("join", g_span(JTAB)),
    "win_32768": ("join", g_win_table(JTAB_WIN)),
    "win_32769": ("join", g_win_table(JTAB_WIN + 1)),
    "win_4096": ("join", g_win_search(JWIN)),
    "win_4097": ("join", g_win_search(JWIN + 1)),
    "win_65535": ("join", g_win_search(JINTERP_MIN - 1)),
    "win_65536": ("join", g_win_search(JINTERP_MIN)),
    "gallop_ww_top": ("join", g_gallop_top),
    "gallop_ww_clusters": ("join", g_gallop_clusters),
    "gallop_wn": ("join", g_gallop_mixed(True)),
    "gallop_nw": ("join", g_gallop_mixed(False)),
    "gallop_one_key_nn": ("join", g_gallop_one_key(False)),
    "gallop_one_key_ww": ("join", g_gallop_one_key(True)),
    # the write mode at its edges
    "matches_16": ("join", g_matches(HEAVY)),
    "matches_17": ("join", g_matches(HEAVY + 1)),
    "tile_16384": ("join", g_tile_total(0)),
    "tile_16385": ("join", g_tile_total(1)),
    "cap_hit": ("join", g_cap(0)),
    "cap_miss": ("join", g_cap(1)),
    # the four width instances
    "edges_nn": ("join", g_edges(False, False)),
    "edges_ww": ("join", g_edges(True, True)),
    "edges_wn": ("join", g_edges(True, False)),
    "edges_nw": ("join", g_edges(False, True)),
    "disjoint_wn": ("join", g_edges(True, False, disjoint=True)),
    "disjoint_nw": ("join", g_edges(False, True, disjoint=True)),
    # runs the engine sorts: 2^20 + 1 tuples over 2^16 keys are skewed (two-phase), over 2^17 they are not
    "skewed_R": ("join", g_engine_sorted("R", (1 << 20) + 1, 1 << 16)),
    "skewed_S": ("join", g_engine_sorted("S", (1 << 20) + 1, 1 << 16)),
    "engine_sorted_R": ("join", g_engine_sorted("R", (1 << 20) + 1, 1 << 17)),
    # the walk
    "walk_random_nn": ("walk", g_walk("random", False, False)),
    "walk_random_ww": ("walk", g_walk("random", True, True)),
    "walk_desc_nw": ("walk", g_walk("desc", False, True)),
    "walk_desc_ww": ("walk", g_walk("desc", True, True)),
    "walk_dips_nn": ("walk", g_walk("dips", False, False)),
    "walk_dips_wn": ("walk", g_walk("dips", True, False)),
    "walk_dips_nw": ("walk", g_walk("dips", False, True)),
    # an empty side; uniform multiplicity (min == max) over a partial last tile, on three bounds paths
    "empty_R": ("join", lambda rng: {"kR": np.zeros(0, dtype=U64), "kS": _u(rng, 100, 0, 99)}),
    "empty_S": ("join", lambda rng: {"kR": _u(rng, 100, 0, 99), "kS": np.zeros(0, dtype=U64)}),
    "uniform_k3_table": ("join", g_uniform_k(3, 1)),
    "uniform_k1_staged": ("join", g_uniform_k(1, 5)),
    "uniform_k3_bisect": ("join", g_uniform_k(3, 5)),
    # qce_rejoin: the WRITE_R-only instance
    "rejoin_heavy": ("rejoin", g_rejoin),
    # 66 000 x 66 000 tuples of one key: 4.36 G pairs
    "refuse_2^32": ("refuse", lambda rng: {"kR": np.full(66_000, 7, dtype=U64), "kS": np.full(66_000, 7, dtype=U64)}),
    # qce_distinct_pairs: id bounds at the digit edges, pair counts on both sides of the one-CTA sort
    **{"distinct_b%d_m%d" % (b, m): ("distinct", g_distinct(b, m))
       for b in (1, 256, 257, 65536, 65537, (1 << 24) + 1) for m in (3000, 20_000)},
    **{"old_%d" % i: ("join", g_old(i)) for i in range(6)},
}


@functools.lru_cache(maxsize=4)
def case_data(name):
    """The case's inputs: join kinds get row ids (a permutation, so that a pair written from the wrong tuple shows)
    and are sorted here unless the engine sorts them ("sort")."""
    kind, gen = CASES[name]
    d = gen(np.random.default_rng(zlib.crc32(name.encode())))
    if kind in ("join", "walk", "refuse"):
        for s in ("R", "S"):
            k = d["k" + s]
            p = np.random.default_rng(len(k)).permutation(len(k)).astype(U64)
            if kind == "walk" and s == "R" or s in d.get("sort", ""):
                d["k" + s], d["p" + s] = k, p
            else:
                o = np.argsort(k, kind="stable")
                d["k" + s], d["p" + s] = k[o], p[o]
    return kind, d


def planned_runs(name, env):
    """The runs R, S as the engine holds them when it joins (the planner's inputs), from the case data alone."""
    kind, d = case_data(name)
    if kind == "rejoin":
        return run_of(np.sort(d["last"])), run_of(np.sort(d["driver"]))
    runs = []
    for s in ("R", "S"):
        k = d["k" + s]
        skewed = False
        if s in d.get("sort", ""):
            kb = max(1, int(k.max()).bit_length())
            srun = {"kind": "host", "n": len(k), "key_bits": kb, "key_min": 0, "key_max": int(k.max()), "wide": kb > 32,
                    "built": False, "hist_arg": None, "in_order": False}
            skewed = sort_plan(srun, k, env)[2]["skewed"]
            k = np.sort(k)
        runs.append(run_of(k, skewed))
    return tuple(runs)


def case_plan(name, env):
    kind, d = case_data(name)
    if kind == "distinct":
        b = lambda p: int(p.max()) + 1  # noqa: E731  (qce_rowids_from_host: max + 1)
        route, tags, npass = plan_distinct(d["pR"], d["pS"], b(d["pR"]), b(d["pS"]))
        return {"routes": {route, "passes_%d" % npass}, "tags": tags}
    R, S = planned_runs(name, env)
    return plan(R, S, env, walk=kind == "walk", stats=kind in ("join", "refuse"))


def _labels(s):
    return frozenset(s.split())


# switch set -> (environment, {case: the exact set of routes it plans to})
DEFAULT_LABELS = {c: _labels(l) for c, l in {
    "nR_1": "nn fused b_table w_light uniform",
    "nR_2047": "nn fused b_table w_light",
    "nR_2048": "nn fused b_table w_light",
    "nR_2049": "nn fused b_table w_light",
    "nR_512x2048": "nn fused b_table w_light w_size scan_warp",
    "nR_512x2048+1": "nn fused b_empty b_table w_light w_size scan_block",
    "span_8189": "nn fused b_table w_light",
    "span_8190": "nn fused b_staged w_light",
    "win_32768": "nn fused b_table w_heavy",
    "win_32769": "nn fused b_bisect w_heavy",
    "win_4096": "nn fused b_staged w_light",
    "win_4097": "nn fused b_bisect w_light",
    "win_65535": "nn fused b_bisect w_light",
    "win_65536": "nn fused b_gallop w_light",
    "gallop_ww_top": "ww fused b_gallop w_light",
    "gallop_ww_clusters": "ww fused b_gallop w_light",
    "gallop_wn": "wn fused b_bisect b_gallop w_light",
    "gallop_nw": "nw fused b_bisect b_gallop w_light",
    "gallop_one_key_nn": "nn fused b_gallop w_size scan_warp",
    "gallop_one_key_ww": "ww fused b_gallop w_size scan_warp",
    "matches_16": "nn fused b_table w_light",
    "matches_17": "nn fused b_table w_heavy",
    "tile_16384": "nn fused b_table w_light uniform",
    "tile_16385": "nn fused b_table w_size scan_warp",
    "edges_nn": "nn fused b_staged w_light",
    "edges_ww": "ww fused b_staged w_light",
    "edges_wn": "wn fused b_staged w_light",
    "edges_nw": "nw fused b_staged w_light",
    "disjoint_wn": "wn fused b_empty w_light uniform",
    "disjoint_nw": "nw fused b_empty w_light uniform",
    "skewed_R": "nn two_phase b_empty b_table scan_block",
    "skewed_S": "nn two_phase b_gallop scan_warp",
    "engine_sorted_R": "nn fused b_empty b_table w_light",
    "walk_random_nn": "nn walk scan_warp",
    "walk_random_ww": "ww walk scan_warp",
    "walk_desc_nw": "nw walk scan_warp",
    "walk_desc_ww": "ww walk scan_warp",
    "walk_dips_nn": "nn walk scan_warp",
    "walk_dips_wn": "wn walk scan_warp",
    "walk_dips_nw": "nw walk scan_warp",
    "empty_R": "nn no_launch",
    "empty_S": "nn no_launch",
    "uniform_k3_table": "nn fused b_table w_light uniform",
    "uniform_k1_staged": "nn fused b_staged w_light uniform",
    "uniform_k3_bisect": "nn fused b_bisect w_light uniform",
    "rejoin_heavy": "nn fused b_table w_size w_cap scan_warp",
    "refuse_2^32": "nn fused b_gallop w_size refused uniform",
    "old_0": "nn fused b_table w_light",
    "old_1": "nn fused b_table w_size scan_warp",
    "old_2": "nn fused b_table w_size w_cap scan_warp",
    "old_3": "nn fused b_table b_gallop w_size w_cap scan_warp",
    "old_4": "ww fused b_staged w_light uniform",
    "old_5": "nn fused b_empty b_table w_light",
}.items()}
DEFAULT_LABELS.update({"distinct_b%d_m%d" % (b, m): _labels("%s passes_%d" % (r, p))
                       for b, p in ((1, 0), (256, 2), (257, 4), (65536, 4), (65537, 6), ((1 << 24) + 1, 8))
                       for m, r in ((3000, "d_block"), (20_000, "d_onesweep"))})
DEFAULT_LABELS.update({"distinct_b1_m3000": _labels("d_none passes_0"), "distinct_b1_m20000": _labels("d_none passes_0")})

_SAME = ["nR_2049", "matches_17", "tile_16385", "gallop_ww_top", "gallop_one_key_ww", "edges_wn", "edges_nw",
         "uniform_k3_table"] + ["old_%d" % i for i in range(6)]
SWITCH_SETS = {
    "defaults": ({}, {c: l for c, l in DEFAULT_LABELS.items() if not c.startswith("cap_")}),
    "two-phase": ({"QCE_JOIN_FUSED": "0"}, {c: _labels(l) for c, l in {
        "nR_2049": "nn two_phase b_table scan_warp",
        "nR_512x2048": "nn two_phase b_table scan_warp",
        "nR_512x2048+1": "nn two_phase b_empty b_table scan_block",
        "span_8189": "nn two_phase b_table scan_warp",
        "span_8190": "nn two_phase b_staged scan_warp",
        "win_32768": "nn two_phase b_table scan_warp",
        "win_32769": "nn two_phase b_bisect scan_warp",
        "win_4096": "nn two_phase b_staged scan_warp",
        "win_4097": "nn two_phase b_bisect scan_warp",
        "win_65536": "nn two_phase b_gallop scan_warp",
        "gallop_ww_top": "ww two_phase b_gallop scan_warp",
        "gallop_ww_clusters": "ww two_phase b_gallop scan_warp",
        "gallop_one_key_nn": "nn two_phase b_gallop scan_warp",
        "gallop_one_key_ww": "ww two_phase b_gallop scan_warp",
        "edges_wn": "wn two_phase b_staged scan_warp",
        "edges_nw": "nw two_phase b_staged scan_warp",
        "disjoint_wn": "wn two_phase b_empty scan_warp uniform",
        "empty_S": "nn no_launch",
        "uniform_k3_table": "nn two_phase b_table scan_warp uniform",
        "uniform_k1_staged": "nn two_phase b_staged scan_warp uniform",
        "uniform_k3_bisect": "nn two_phase b_bisect scan_warp uniform",
        "rejoin_heavy": "nn two_phase b_table scan_warp",
        "refuse_2^32": "nn two_phase b_gallop scan_warp refused uniform",
        "old_0": "nn two_phase b_table scan_warp",
        "old_1": "nn two_phase b_table scan_warp",
        "old_2": "nn two_phase b_table scan_warp",
        "old_3": "nn two_phase b_table b_gallop scan_warp",
        "old_4": "ww two_phase b_staged scan_warp uniform",
        "old_5": "nn two_phase b_empty b_table scan_warp",
    }.items()}),
    "guess-1": ({"QCE_JOIN_CAP": "1"}, {c: _labels(l) for c, l in {
        "nR_2049": "nn fused b_table w_cap scan_warp",
        "matches_17": "nn fused b_table w_cap scan_warp",
        "tile_16384": "nn fused b_table w_cap scan_warp uniform",
        "gallop_ww_top": "ww fused b_gallop w_cap scan_warp",
        "edges_wn": "wn fused b_staged w_cap scan_warp",
        "edges_nw": "nw fused b_staged w_cap scan_warp",
        "uniform_k3_table": "nn fused b_table w_cap scan_warp uniform",
        "skewed_S": "nn two_phase b_gallop scan_warp",
        "rejoin_heavy": "nn fused b_table w_size w_cap scan_warp",
        "old_0": "nn fused b_table w_cap scan_warp",
        "old_1": "nn fused b_table w_size scan_warp",
        "old_2": "nn fused b_table w_cap w_size scan_warp",
        "old_3": "nn fused b_table b_gallop w_size w_cap scan_warp",
        "old_4": "ww fused b_staged w_light uniform",
        "old_5": "nn fused b_empty b_table w_cap scan_warp",
    }.items()}),
    "guess-10000": ({"QCE_JOIN_CAP": str(CAP_EXACT)}, {c: _labels(l) for c, l in {
        "cap_hit": "nn fused b_table w_light",
        "cap_miss": "nn fused b_table w_light w_cap scan_warp",
        "old_0": "nn fused b_table w_light w_cap scan_warp",
        "old_1": "nn fused b_table w_size scan_warp",
        "old_2": "nn fused b_table w_size w_cap scan_warp",
        "old_3": "nn fused b_table b_gallop w_size w_cap scan_warp",
        "old_4": "ww fused b_staged w_light uniform",
        "old_5": "nn fused b_empty b_table w_light",
    }.items()}),
    "block-order": ({"QCE_JOIN_TICKET": "0"}, {c: DEFAULT_LABELS[c] for c in _SAME}),
    "4-ctas": ({"QCE_JOIN_MINB": "4"}, {c: DEFAULT_LABELS[c] for c in _SAME}),
}


# ---- CPU: the case list plans to its labels -------------------------------------------------------------------
def test_cases_plan_to_their_routes():
    """Every case plans to exactly the routes its label names under its switch set, and every instance, kernel
    sequence, bounds path, write mode, tile scan and distinct-pairs sort has a case.  Runs without a GPU: a moved
    threshold shows up here as a stale label."""
    wrong, covered = [], set()
    for sset, (env, cases) in SWITCH_SETS.items():
        assert set(env) <= set(JOIN_SWITCHES), sset
        for c, labels in cases.items():
            assert c in CASES, (sset, c)
            assert labels <= set(ROUTES + DISTINCT_ROUTES) | {"passes_%d" % p for p in range(9)}, (sset, c, labels)
            got = case_plan(c, env)["routes"]
            covered |= got
            if got != labels:
                wrong.append((sset, c, " ".join(sorted(labels)), " ".join(sorted(got))))
    assert not wrong, "\n".join("%s/%s: labelled %s, plans to %s" % w for w in wrong)
    assert not set(ROUTES + DISTINCT_ROUTES) - covered, sorted(set(ROUTES + DISTINCT_ROUTES) - covered)
    assert not set(CASES) - set().union(*(cs for _, cs in SWITCH_SETS.values()))
    # the refusal is a one-key join: every tile defers, so it needs no more output than the guess of 66 000
    p = case_plan("refuse_2^32", {})
    assert p["m"] == 66_000 ** 2 >= ROWID_LIMIT and p["cap"] == 66_000


def test_cases_sit_on_their_edges():
    """The edge cases are at the edges they are named for."""
    one = lambda c, key, env={}: case_plan(c, env)[key]  # noqa: E731
    for c, n in (("nR_1", 1), ("nR_2047", 2047), ("nR_2048", 2048), ("nR_2049", 2049), ("nR_512x2048", BIG),
                 ("nR_512x2048+1", BIG + 1)):
        assert one(c, "nR") == n, c
    for c, w in (("win_32768", 32768), ("win_32769", 32769), ("win_4096", 4096), ("win_4097", 4097),
                 ("win_65535", 65535), ("win_65536", 65536)):
        assert one(c, "window") == [w], c
    for c, s in (("span_8189", 8189), ("span_8190", 8190)):
        R, _ = planned_runs(c, {})
        assert int(R["keys"][-1] - R["keys"][0]) == s
    assert one("matches_16", "max") == 16 and one("matches_17", "max") == 17
    assert one("tile_16384", "tile_total") == [16384] and one("tile_16385", "tile_total") == [16385]
    env = {"QCE_JOIN_CAP": str(CAP_EXACT)}
    assert one("cap_hit", "m", env) == CAP_EXACT and one("cap_miss", "m", env) == CAP_EXACT + 1
    for c in ("gallop_one_key_nn", "gallop_one_key_ww"):
        R, S = planned_runs(c, {})
        k = S["keys"][(S["keys"] >= R["keys"][0]) & (S["keys"] <= R["keys"][-1])]  # the tile's window
        assert len(k) >= JINTERP_MIN and k.min() == k.max()  # ks0 == ks1
    R, S = planned_runs("gallop_ww_top", {})
    assert R["keys"][-1] == S["keys"][-1] == U64(TOP)
    for c in ("edges_nn", "edges_ww", "edges_wn", "edges_nw"):
        R, S = planned_runs(c, {})
        for run, wide in zip((R, S), (c[-2] == "w", c[-1] == "w")):
            assert set(E if wide else E[:2]) <= set(int(k) for k in run["keys"]), (c, wide)
    for c in ("uniform_k3_table", "uniform_k1_staged", "uniform_k3_bisect"):
        p = case_plan(c, {})
        assert p["nR"] % JTILE and p["min"] == p["max"] > 0
    assert planned_runs("skewed_R", {})[0]["skewed"] and planned_runs("skewed_S", {})[1]["skewed"]
    assert not planned_runs("engine_sorted_R", {})[0]["skewed"]
    assert not planned_runs("skewed_R", {"QCE_MSD": "0"})[0]["skewed"]  # the sort's flag comes with its MSD route
    _, d = case_data("rejoin_heavy")
    assert (d["driver"] == 77).sum() >= 20_000 and len(d["last"]) < (1 << 20)  # below the MSD sort: stable


def test_planner_restates_edges():
    """Spot checks of the restated constants at their edges."""
    assert bounds_path(0, 0) == "b_empty"
    assert bounds_path(JTAB_WIN, JTAB - 1) == "b_table" and bounds_path(JTAB_WIN + 1, JTAB - 1) == "b_bisect"
    assert bounds_path(1, JTAB) == "b_staged" and bounds_path(JWIN, JTAB) == "b_staged"
    assert bounds_path(JWIN + 1, JTAB) == "b_bisect" and bounds_path(JWIN + 1, 0) == "b_table"
    assert bounds_path(JINTERP_MIN - 1, 1 << 40) == "b_bisect" and bounds_path(JINTERP_MIN, 1 << 40) == "b_gallop"
    assert write_mode(JFUSE_MAX, HEAVY, 0, JFUSE_MAX) == "w_light"
    assert write_mode(JFUSE_MAX, HEAVY + 1, 0, JFUSE_MAX) == "w_heavy"
    assert write_mode(JFUSE_MAX + 1, 1, 0, 1 << 40) == "w_size"
    assert write_mode(10, 1, 5, 15) == "w_light" and write_mode(10, 1, 6, 15) == "w_cap"
    assert switches({}) == {"fused": 1, "cap": 0} and switches({"QCE_JOIN_FUSED": "off"})["fused"] == 0
    ids = np.arange(5, dtype=U64)
    assert plan_distinct(ids, ids, 1, 1)[2] == 0 and plan_distinct(ids, ids, 256, 257)[2] == 3
    assert plan_distinct(ids, ids, 0, 65537)[2] == 7 and plan_distinct(ids, ids, 1 << 24, 1)[2] == 3
    # the tile scan: 512 tiles in one warp, 513 in the block scan
    for n, kind in ((BIG, "scan_warp"), (BIG + 1, "scan_block")):
        k = np.arange(n, dtype=U64)
        assert kind in plan(run_of(k), run_of(k[:1]), {"QCE_JOIN_FUSED": "0"})["routes"]
    # the walk matches a tuple only when its key is at least every earlier key
    p = plan(run_of([5, 3, 5, 7, 6, 7]), run_of([3, 5, 6, 7, 7]), {}, walk=True)
    assert p["cnt"].tolist() == [1, 0, 1, 2, 0, 2] and p["m"] == 6 and p["tags"]["join_write"] == 1


# ---- GPU: every switch set in a fresh process (the switches are read once per process) --------------------------
def _free(e, handles):
    for h in handles:
        e.rowids_free(h)


def _check_join(e, name, env, fails):
    """One join case: runs, pairs, stats, launches, arena."""
    import ctypes as C
    from oracle import qce_oracle as orc
    kind, d = case_data(name)
    e.sync()
    used0 = e.mempool_stats()[1]
    R, S = e.tuples_from_host(d["kR"], d["pR"]), e.tuples_from_host(d["kS"], d["pS"])
    for s, h in (("R", R), ("S", S)):
        if s in d.get("sort", ""):
            e.sort_tuples(h)
    (kR, pR), (kS, pS) = e.tuples_to_host(R), e.tuples_to_host(S)
    want_runs = planned_runs(name, env)
    np.testing.assert_array_equal(kR, want_runs[0]["keys"])
    np.testing.assert_array_equal(kS, want_runs[1]["keys"])
    p = case_plan(name, env)
    calls = {"walk": ["walk"], "refuse": ["join"]}.get(kind, ["join", "stats"])
    try:
        for call in calls:
            e.profile(True)
            if kind == "refuse":
                import qce_b200
                with pytest.raises(qce_b200.EngineError, match=r"exceeds the 2\^32 row-id column limit"):
                    e.merge_join(R, S)
                res = ()
            elif call == "walk":
                res = e.merge_join_walk(R, S)
            elif call == "join":
                res = e.merge_join(R, S)
            else:
                oR, oS, mn, mx = C.c_void_p(), C.c_void_p(), C.c_uint32(), C.c_uint32()
                e._ck(e.lib.qce_merge_join_stats(R, S, C.byref(oR), C.byref(oS), C.byref(mn), C.byref(mx)))
                res = (oR.value, oS.value)
            prof = e.profile_read()
            e.profile(False)
            got = {t: prof[t]["launches"] for t in JOIN_TAGS if t in prof}
            try:
                if kind != "refuse":
                    gR, gS = e.rowids_to_host(res[0]), e.rowids_to_host(res[1])
                    wR, wS = orc._merge_serial(kR, pR, kS, pS) if kind == "walk" else orc.merge_join(kR, pR, kS, pS)
                    assert len(gR) == len(gS) == len(wR) == p["m"], ("pairs", len(gR), len(gS), len(wR), p["m"])
                    bad = np.flatnonzero((gR != wR) | (gS != wS))
                    assert not len(bad), "%d pairs differ, first at %d of %d" % (len(bad), bad[0], len(wR))
                if call == "stats":
                    assert (mn.value, mx.value) == (p["min"], p["max"]), \
                        "min/max matches %s, numpy %s" % ((mn.value, mx.value), (p["min"], p["max"]))
                assert got == p["tags"], "launches %s, planned %s" % (got, p["tags"])
            except Exception as ex:  # noqa: BLE001 -- each call reports on its own
                fails.append("%s [%s]: %s" % (name, call, str(ex)[:1500]))
            finally:
                _free(e, res)
            if kind == "refuse":  # the engine still joins afterwards (the arena is checked below)
                _check_join(e, "nR_2049", env, fails)
    finally:
        e.tuples_free(R)
        e.tuples_free(S)
    e.sync()
    used1 = e.mempool_stats()[1]
    if used1 != used0:
        fails.append("%s: arena used %d bytes before, %d after" % (name, used0, used1))


def _check_rejoin(e, name, env, fails):
    from oracle import qce_oracle as orc
    _, d = case_data(name)
    p = case_plan(name, env)
    e.sync()
    used0 = e.mempool_stats()[1]
    hs = [e.rowids_from_host(d[k]) for k in ("driver", "last", "edit")]
    e.profile(True)
    out = e.rejoin(*hs)
    prof = e.profile_read()
    e.profile(False)
    got = {t: prof[t]["launches"] for t in JOIN_TAGS if t in prof}
    try:
        g, w = e.rowids_to_host(out), orc.join_payloads(d["driver"], d["last"], d["edit"])
        assert len(g) == len(w) == p["m"], ("pairs", len(g), len(w), p["m"])
        assert (g == w).all(), "%d row ids differ" % int((g != w).sum())
        assert got == p["tags"], "launches %s, planned %s" % (got, p["tags"])
    except Exception as ex:  # noqa: BLE001
        fails.append("%s: %s" % (name, str(ex)[:1500]))
    _free(e, hs + [out])
    e.sync()
    if e.mempool_stats()[1] != used0:
        fails.append("%s: arena unbalanced" % name)


def _check_distinct(e, name, env, fails):
    from oracle import qce_oracle as orc
    _, d = case_data(name)
    p = case_plan(name, env)
    e.sync()
    used0 = e.mempool_stats()[1]
    hR, hS = e.rowids_from_host(d["pR"]), e.rowids_from_host(d["pS"])
    e.profile(True)
    dR, dS = e.distinct_pairs(hR, hS)
    prof = e.profile_read()
    e.profile(False)
    got = {t: prof[t]["launches"] for t in DISTINCT_TAGS if t in prof}
    try:
        wR, wS = orc.distinct_pairs(d["pR"], d["pS"])
        np.testing.assert_array_equal(e.rowids_to_host(dR), wR)
        np.testing.assert_array_equal(e.rowids_to_host(dS), wS)
        assert got == p["tags"], "launches %s, planned %s" % (got, p["tags"])
    except Exception as ex:  # noqa: BLE001
        fails.append("%s: %s" % (name, str(ex)[:1500]))
    _free(e, (hR, hS, dR, dS))
    e.sync()
    if e.mempool_stats()[1] != used0:
        fails.append("%s: arena unbalanced" % name)


def run_cases(sset):
    """Every case of switch set `sset` under this process's switches; return the list of failures."""
    import qce_b200
    e = qce_b200.Engine()
    env = dict(os.environ)
    fails = []
    for name, labels in SWITCH_SETS[sset][1].items():
        kind = CASES[name][0]
        n0 = len(fails)
        try:
            assert case_plan(name, env)["routes"] == labels, "stale label"
            {"rejoin": _check_rejoin, "distinct": _check_distinct}.get(kind, _check_join)(e, name, env, fails)
        except Exception as ex:  # noqa: BLE001 -- every case runs; the parent reports them all
            fails.append("%s: %s" % (name, str(ex)[:1500]))
        print(("ok %s" % name) if len(fails) == n0 else "FAIL " + "\nFAIL ".join(fails[n0:]), flush=True)
    return fails


_CHILD = r"""
import sys
sys.path.insert(0, %r)
from tests.test_gpu_join_routes import run_cases
fails = run_cases(sys.argv[1])
print("ok" if not fails else "%%d failed" %% len(fails))
"""


@pytest.mark.gpu
@pytest.mark.parametrize("sset", list(SWITCH_SETS))
def test_join_routes(sset):
    """Every case of the switch set in a fresh process: the pairs equal the oracle's merge byte for byte, the
    min / max matches equal numpy's, the launch profile shows the planned kernels, the arena is balanced."""
    env = SWITCH_SETS[sset][0]
    base = {k: v for k, v in os.environ.items() if k not in JOIN_SWITCHES + SORT_SWITCHES}
    p = subprocess.run([sys.executable, "-c", _CHILD % ROOT, sset], env=dict(base, **env), capture_output=True,
                       text=True, timeout=1500)
    out = p.stdout.strip().splitlines()
    assert p.returncode == 0 and out and out[-1] == "ok", \
        "\n".join([l for l in out if not l.startswith("ok ")] + [p.stderr[-3000:]])
