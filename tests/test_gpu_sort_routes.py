"""The tuple sort (qce_sort_tuples) route by route, against numpy's stable argsort.

qce_sort_tuples -> sort_packed -> msd_sort -> radix_sort (csrc/qce_engine.cu) choose one of about a dozen kernel
sequences from the run's size, its key range and the sizes of its MSD sub-buckets, and from switches that are read
once per process.  `plan` restates that choice in Python.  The CPU test holds every case to the route its label
names and checks that every route has a case, so a changed threshold shows up here first.  The GPU tests sort every
case in a fresh process per switch set and check from the launch profile (qce_profile_json) that the planned
kernels are the ones that ran.

Bar: the stable routes (block sort, LSD one-sweep, wide key/value sort, the LSD passes after an MSD attempt) give
exactly the order of a stable sort, keys and row ids.  The MSD routes are unstable by design: they give the sorted
key column exactly and the same (key, row id) multiset.
"""
import functools
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

U64 = np.uint64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- constants of the route choice (csrc/qce_engine.cu) ----------------------------------------------------------
BS_TILE = 4096                      # k_block_sort: runs of at most this many tuples
MSD_MIN_N, RUN_LIMIT = 1 << 20, 1 << 30
MSD_MIN_BITS, MSD_MAX_BITS = 9, 32
P_MIN, P_MAX, P_AVG = 9, 16, 2700   # partition bits: the smallest P whose average sub-bucket holds <= 2700 tuples
MSD_LOCAL_CAP = 4096                # largest finish tile (k_msd_local_sort<256, 16>, k_msd_count_sort<512, 8>)
BIG_CAP, BIG_MAX = 3072, 8192       # k_big_list: sub-buckets over 3072 tuples, at most 8192 of them
COUNT_MAX_R = 12                    # the count sort holds 2^R <= 4096 counters
BULK_COUNT_CAP = 3072               # k_msd_count_sort_bulk<256, 12>: sub-buckets of up to 3072 tuples
ONESWEEP_TILE = 256 * 16            # k_onesweep: threads x items

SORT_SWITCHES = ("QCE_MSD", "QCE_MSD_BIG", "QCE_FUSED_BUILD_HIST", "QCE_SORT_PROBE")

# kernel families whose launch counts identify a route (a tag names a family, not a template instance)
WATCH = ("block_sort", "radix_hist", "onesweep_k", "onesweep_kv", "msd_hist", "msd_partition", "msd_count_sort",
         "msd_local_sort", "msd_big_partition")

ROUTES = ["block", "lsd", "msd_bulk_1024", "msd_bulk_2048", "msd_bulk_4096", "msd_count_512x8x3", "msd_big", "msd_local",
          "msd_r0", "msd_lsd_fallback", "wide_block", "wide_onesweep", "in_order"]
STABLE = {"block", "lsd", "msd_lsd_fallback", "wide_block", "wide_onesweep", "in_order"}


def _bitlen(x: int) -> int:
    return int(x).bit_length()


def _sw(env, name, default):
    """A switch as the engine reads it (atoi; unset = default)."""
    v = env.get(name)
    if v is None:
        return default
    try:
        return int(v)
    except ValueError:
        return 0


def switches(env):
    return {"msd": _sw(env, "QCE_MSD", 1), "big": _sw(env, "QCE_MSD_BIG", 1),
            "fused_hist": _sw(env, "QCE_FUSED_BUILD_HIST", 1), "probe": _sw(env, "QCE_SORT_PROBE", 1)}


def partition_bits(n: int, span: int):
    """P of msd_sort for a run of n tuples whose keys - key_min lie in [0, span]; None when too dense."""
    kb = _bitlen(span)
    P = P_MIN
    while P < P_MAX and P < kb and n // ((span >> (kb - P)) + 1) > P_AVG:
        P += 1
    return None if n // ((span >> (kb - P)) + 1) > P_AVG else P


def _msd(keys, n, kmin, kmax, hist_bits, sw, info):
    """msd_sort: (route or None, tags launched).  None = the LSD passes sort the run.  info["skewed"]: the flag
    the sort leaves on the run (msd_plan: 16 or more tuples per possible key; msd_after_level_a: a sub-bucket over
    BIG_CAP tuples), which sends its joins down the two-phase route."""
    if not sw["msd"] or n < MSD_MIN_N:
        return None, {}
    span = kmax - kmin
    info["skewed"] = n // (span + 1) >= 16
    if n >= RUN_LIMIT:
        return None, {}
    kb = _bitlen(span)
    info["msd_key_bits"] = kb
    if kb < MSD_MIN_BITS or kb > MSD_MAX_BITS:
        return None, {}
    P = partition_bits(n, span)
    info["P"] = P
    if P is None:
        return None, {}
    R = kb - P
    cached = hist_bits is not None and kmin == 0 and hist_bits == kb
    sub = np.bincount(((keys - U64(kmin)) >> U64(R)).astype(np.int64), minlength=1 << P)
    max_sub, nbig = int(sub.max()), int((sub > BIG_CAP).sum())
    info.update(R=R, cached_hist=cached, max_sub=max_sub, nbig=nbig)
    if max_sub > BIG_CAP:
        info["skewed"] = True
    tags = {"msd_hist": 1 if cached else 2, "msd_partition": 1}
    big_route = max_sub > MSD_LOCAL_CAP and bool(sw["big"]) and 0 < R <= COUNT_MAX_R and nbig <= BIG_MAX
    if not (max_sub <= MSD_LOCAL_CAP or R == 0 or big_route):
        return None, tags  # level B counted, nothing moved: the LSD passes take the run as it was
    tags["msd_partition"] = 2
    if R == 0:
        return "msd_r0", tags
    if R > COUNT_MAX_R:
        tags["msd_local_sort"] = 1
        return "msd_local", tags
    tags["msd_count_sort"] = 1
    if max_sub <= BULK_COUNT_CAP or big_route:
        maxb = 1024 if R <= 10 else (2048 if R == 11 else 4096)
        info["count_sort"] = "bulk_%d" % maxb
        route = "msd_bulk_%d" % maxb
    else:  # BULK_COUNT_CAP < max_sub <= MSD_LOCAL_CAP
        info["count_sort"] = "512x8x3"
        route = "msd_count_512x8x3"
    if big_route:
        tags["msd_big_partition"] = 1
        route = "msd_big"
    return route, tags


def plan(run, keys, env):
    """The route qce_sort_tuples takes for `run` (see case_data) under the switches in `env`:
    (route, {tag: launches} for the tags in WATCH, the planner's inputs and intermediates)."""
    sw = switches(env)
    n, key_bits, kmin, kmax = run["n"], run["key_bits"], run["key_min"], run["key_max"]
    info = {"n": n, "key_bits": key_bits, "key_min": kmin, "key_max": kmax, "kind": run["kind"], "skewed": False}
    if run["in_order"] and sw["probe"]:
        info["skewed"] = kmax < (1 << 64) - 1 and n // (kmax + 1) >= 16  # qce_sort_tuples: from the statistics
        return "in_order", {}, info
    if run["wide"]:
        npass = -(-key_bits // 8)
        info["passes"] = npass
        if n <= BS_TILE:
            return "wide_block", {"block_sort": 1}, info
        return "wide_onesweep", {"radix_hist": 1, "onesweep_kv": npass}, info
    # the cached level-A histogram: taken by the build kernel or left by qce_key_histogram
    hist = run["hist_arg"]
    if hist is None and run["built"] and sw["fused_hist"] and n >= MSD_MIN_N and key_bits >= MSD_MIN_BITS:
        hist = key_bits
    info["hist_key_bits"] = hist
    if hist is not None and _bitlen(kmax) != hist:  # qce_sort_tuples: the statistics are not the column's own
        hist = -1
    if kmax == 0 or kmax >= (1 << key_bits):
        kmax = (1 << key_bits) - 1
    if kmin > kmax:
        kmin = 0
    route, tags = _msd(keys, n, kmin, kmax, hist, sw, info)
    if route is not None:
        return route, tags, info
    if n <= BS_TILE:
        return "block", {"block_sort": 1}, info
    tags.update(radix_hist=1, onesweep_k=-(-key_bits // 8))
    return ("msd_lsd_fallback" if tags.get("msd_hist") else "lsd"), tags, info


# ---- cases ---------------------------------------------------------------------------------------------------
# name -> spec.  kinds: host (qce_tuples_from_host, row ids shuffled so that a tie's input order is not its id
# order), built (a whole base column), built_ids (a column through a row-id subset), device (a host run moved
# through qce_partition_tuples with one part into qce_tuples_from_device_packed with key_lo / key_hi).
# keys: uniform = uniform over [lo, lo + 2^bits) with the top key planted; plant = uniform background with one
# sub-bucket of exactly `size` tuples over distinct keys; many_big = more than BIG_MAX sub-buckets over BIG_CAP.
N_ODD = 1_450_001  # P = 10 at any key width: ~1400 tuples per sub-bucket, well below the planted sizes
CASES = {
    # block sort and LSD one-sweep sizes
    "block_1000_b12": dict(kind="host", n=1000, bits=12),
    "block_4096_b27": dict(kind="host", n=4096, bits=27),
    "lsd_4097_b27": dict(kind="host", n=4097, bits=27),
    "lsd_2^20-1_b20": dict(kind="host", n=(1 << 20) - 1, bits=20),
    "lsd_2^20+1_b8": dict(kind="host", n=(1 << 20) + 1, bits=8),            # key bits below 9: no MSD attempt
    "lsd_dense_b9": dict(kind="host", n=1_500_001, bits=9),                  # P cannot reach 2700 per sub-bucket
    **{"lsd_%d_b27" % (3 * ONESWEEP_TILE + d): dict(kind="host", n=3 * ONESWEEP_TILE + d, bits=27) for d in (-1, 1)},
    # MSD at R = 0 .. 20 remaining bits
    "r0_2^20_b9": dict(kind="host", n=1 << 20, bits=9),
    "r0_odd_b10": dict(kind="host", n=N_ODD, bits=10),
    "r1_odd_b11": dict(kind="host", n=N_ODD, bits=11),
    "r10_odd_b20": dict(kind="host", n=N_ODD, bits=20),
    "r11_odd_b21": dict(kind="host", n=N_ODD, bits=21),
    "r12_odd_b22": dict(kind="host", n=N_ODD, bits=22),
    "r12_2^20_b21": dict(kind="host", n=1 << 20, bits=21),
    "r13_odd_b23": dict(kind="host", n=N_ODD, bits=23),
    "r16_odd_b26": dict(kind="host", n=N_ODD, bits=26),
    "r20_odd_b30": dict(kind="host", n=N_ODD, bits=30),
    # one sub-bucket planted at the edges of the finish kernels
    **{"plant%d_r%d" % (s, b - 10): dict(kind="host", n=N_ODD, bits=b, plant=s)
       for b in (20, 21, 22) for s in (2048, 2049, 3072, 3073, 4096, 4097)},
    "plant4096_r13": dict(kind="host", n=N_ODD, bits=23, plant=4096),
    "plant4097_r13": dict(kind="host", n=N_ODD, bits=23, plant=4097),
    "many_big_r12": dict(kind="host", many_big=True, bits=26),
    # a rank's share: keys in [key_lo, key_hi], level A on key - key_lo
    "dev_lo_hi_unknown": dict(kind="device", n=N_ODD, lo=(1 << 31) + 5, hi=(1 << 32) - 1, key_hi=0),
    "dev_lo_hi_b22": dict(kind="device", n=N_ODD, lo=(1 << 31) + 5, bits=22, key_hi=(1 << 31) + 5 + (1 << 22) - 1),
    "dev_lo_eq_hi": dict(kind="device", n=(1 << 20) + 1, lo=(1 << 31) + 5, bits=0, key_hi=(1 << 31) + 5),
    "dev_lo_plant4097": dict(kind="device", n=N_ODD, lo=(1 << 31) + 5, bits=22, key_hi=(1 << 31) + 5 + (1 << 22) - 1,
                             plant=4097),
    # runs with a cached level-A histogram
    "built_b22": dict(kind="built", n=N_ODD, bits=22),
    "built_ids_b24": dict(kind="built_ids", n=1_300_001, rows=3_000_001, bits=24),
    "built_b22_hist24": dict(kind="built", n=N_ODD, bits=22, hist=24),       # statistics that do not match
    "built_b22_hist22": dict(kind="built", n=N_ODD, bits=22, hist=22),
    "host_b22_hist22": dict(kind="host", n=N_ODD, bits=22, hist=22),
    "in_order_2^20+1": dict(kind="built", n=(1 << 20) + 1, in_order=True),
    # wide keys (>= 2^32): key / row-id sort, 8-bit digits over all 64 bits
    "wide_block_max_4096": dict(kind="host", n=4096, wide="max"),
    "wide_block_hi_3001": dict(kind="host", n=3001, wide="hi"),
    "wide_os_max_4097": dict(kind="host", n=4097, wide="max"),
    "wide_os_hi_12289": dict(kind="host", n=12289, wide="hi"),
    "wide_os_top_18433": dict(kind="host", n=18433, wide="top"),
    "wide_os_hi_100003": dict(kind="host", n=100003, wide="hi"),
}

_LSD_TILES = ["lsd_%d_b27" % (3 * ONESWEEP_TILE + d) for d in (-1, 1)]
_WIDE = ["wide_block_max_4096", "wide_block_hi_3001", "wide_os_max_4097", "wide_os_hi_12289", "wide_os_top_18433",
         "wide_os_hi_100003"]
_WIDE_ROUTES = {c: ("wide_block" if CASES[c]["n"] <= BS_TILE else "wide_onesweep") for c in _WIDE}
_BULK_PLANTS = {"plant%d_r%d" % (s, r): ("msd_bulk_%d" % m if s <= BULK_COUNT_CAP else
                                         ("msd_count_512x8x3" if s <= MSD_LOCAL_CAP else "msd_big"))
                for r, m in ((10, 1024), (11, 2048), (12, 4096)) for s in (2048, 2049, 3072, 3073, 4096, 4097)}


# switch set -> (environment, {case: route it must take})
SWITCH_SETS = {
    "defaults": ({}, {
        "block_1000_b12": "block", "block_4096_b27": "block", "lsd_4097_b27": "lsd", "lsd_2^20-1_b20": "lsd",
        "lsd_2^20+1_b8": "lsd", "lsd_dense_b9": "lsd", **{c: "lsd" for c in _LSD_TILES},
        "r0_2^20_b9": "msd_r0", "r0_odd_b10": "msd_r0", "r1_odd_b11": "msd_bulk_1024", "r10_odd_b20": "msd_bulk_1024",
        "r11_odd_b21": "msd_bulk_2048", "r12_odd_b22": "msd_bulk_4096", "r12_2^20_b21": "msd_bulk_4096",
        "r13_odd_b23": "msd_local", "r16_odd_b26": "msd_local", "r20_odd_b30": "msd_local",
        **_BULK_PLANTS, "plant4096_r13": "msd_local", "plant4097_r13": "msd_lsd_fallback",
        "many_big_r12": "msd_lsd_fallback",
        "dev_lo_hi_unknown": "msd_local", "dev_lo_hi_b22": "msd_bulk_4096", "dev_lo_eq_hi": "lsd",
        "dev_lo_plant4097": "msd_big",
        "built_b22": "msd_bulk_4096", "built_ids_b24": "msd_local", "built_b22_hist24": "msd_bulk_4096",
        "built_b22_hist22": "msd_bulk_4096", "host_b22_hist22": "msd_bulk_4096", "in_order_2^20+1": "in_order",
        **_WIDE_ROUTES}),
    "msd-off": ({"QCE_MSD": "0"}, {"r12_odd_b22": "lsd", "r0_2^20_b9": "lsd", "plant4097_r12": "lsd",
                                   "built_b22": "lsd", "dev_lo_hi_b22": "lsd"}),
    "big-off": ({"QCE_MSD_BIG": "0"}, {"plant4097_r12": "msd_lsd_fallback", "plant4097_r10": "msd_lsd_fallback",
                                       "dev_lo_plant4097": "msd_lsd_fallback", "plant4096_r12": "msd_count_512x8x3"}),
    "build-hist-off": ({"QCE_FUSED_BUILD_HIST": "0"}, {"built_b22": "msd_bulk_4096", "built_ids_b24": "msd_local",
                                                        "built_b22_hist22": "msd_bulk_4096"}),
    "probe-off": ({"QCE_SORT_PROBE": "0"}, {"in_order_2^20+1": "msd_bulk_4096", "built_b22": "msd_bulk_4096"}),
}


def _uniform(rng, n, lo, hi):
    keys = rng.integers(lo, hi, n, dtype=U64, endpoint=True)
    keys[rng.integers(0, n)] = hi  # pin key_max, so that P and R are what the case intends
    return keys


def _planted(rng, n, lo, bits, size):
    """Uniform keys over [lo, lo + 2^bits) with one sub-bucket (at the P the run gets) of exactly `size` tuples,
    spread over the keys inside it; no other sub-bucket comes near `size`."""
    P = partition_bits(n, (1 << bits) - 1)
    R = bits - P
    j = (1 << P) // 3
    u = rng.integers(0, (1 << bits) - (1 << R), n - size, dtype=U64)
    u[u >= U64(j << R)] += U64(1 << R)                     # the background skips sub-bucket j
    u[rng.integers(0, n - size)] = (1 << bits) - 1
    hot = U64(j << R) | rng.integers(0, 1 << R, size, dtype=U64)
    return rng.permutation(np.concatenate([u, hot])) + U64(lo)


def _many_big(rng, bits):
    """BIG_MAX + 8 sub-buckets of 3100 tuples and one of 4097 at P = 14, R = 12: too many to list."""
    R = 12
    nb = BIG_MAX + 8
    sizes = np.full(nb, 3100, dtype=np.int64)
    sizes[nb // 2] = 4097
    sub = np.repeat(np.arange(nb, dtype=U64), sizes)
    keys = (sub << U64(R)) | rng.integers(0, 1 << R, len(sub), dtype=U64)
    return rng.permutation(np.append(keys, U64((1 << bits) - 1)))


def _wide(rng, n, how):
    if how == "max":    # bit 63 on about half the keys, UINT64_MAX and 2^63 repeated
        keys = rng.integers(0, 1 << 63, n, dtype=U64) | (rng.integers(0, 2, n, dtype=U64) << U64(63))
        keys[rng.choice(n, 40, replace=False)] = U64(0xFFFFFFFFFFFFFFFF)
        keys[rng.choice(n, 40, replace=False)] = U64(1 << 63)
        keys[rng.choice(n, 40, replace=False)] = U64(0)
        return keys
    if how == "hi":     # every key shares its high word: the order is in the low word, with ties
        return U64(0xDEADBEEF << 32) | rng.integers(0, max(2, n // 4), n, dtype=U64)
    # "top": few distinct keys near the top of the range, each differing in one byte
    vals = np.array([0xFFFFFFFFFFFFFFFF - (1 << (8 * b)) + 1 for b in range(8)] + [1 << 32, (1 << 63) | 1], dtype=U64)
    return vals[rng.integers(0, len(vals), n)]


@functools.lru_cache(maxsize=2)
def case_data(name):
    """(keys, row ids, column, run): the tuples of case `name` as handed to the engine (the base column for built
    runs), and the run's statistics as the engine will hold them (the planner's inputs)."""
    spec = CASES[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    lo = spec.get("lo", 0)
    kind = spec["kind"]
    if spec.get("many_big"):
        keys = _many_big(rng, spec["bits"])
    elif "wide" in spec:
        keys = _wide(rng, spec["n"], spec["wide"])
    elif spec.get("in_order"):
        keys = np.arange(spec["n"], dtype=U64) * U64(3)
    elif kind == "built_ids":
        keys = _uniform(rng, spec["rows"], 0, (1 << spec["bits"]) - 1)
    elif "hi" in spec:
        keys = _uniform(rng, spec["n"], lo, spec["hi"])
    elif spec["bits"] == 0:
        keys = np.full(spec["n"], lo, dtype=U64)
    elif "plant" in spec:
        keys = _planted(rng, spec["n"], lo, spec["bits"], spec["plant"])
    else:
        keys = _uniform(rng, spec["n"], lo, lo + (1 << spec["bits"]) - 1)
    col = None
    if kind == "built":
        col, ids = keys, np.arange(len(keys), dtype=U64)
    elif kind == "built_ids":
        col = keys
        ids = np.sort(rng.choice(len(col), spec["n"], replace=False)).astype(U64)
        keys = col[ids]
    else:
        ids = rng.permutation(len(keys)).astype(U64)
    top = int(col.max() if col is not None else keys.max())
    kb = max(1, _bitlen(top))
    run = {"kind": kind, "n": len(keys), "key_bits": kb, "key_min": 0, "key_max": top, "wide": kb > 32,
           "built": col is not None, "hist_arg": spec.get("hist"),
           "in_order": kind == "built" and bool(np.all(col[1:] >= col[:-1]))}
    if kind == "device":
        run.update(key_bits=32, key_min=lo, key_max=spec["key_hi"])
    return keys, ids, col, run


# ---- CPU: the case list plans to its labels -------------------------------------------------------------------
def test_cases_plan_to_their_routes():
    """Every case plans to the route its label names under its switch set, and every route has a case.  Runs
    without a GPU: a changed threshold in the route choice shows up here as a stale label."""
    by_case = {}
    for sset, (env, cases) in SWITCH_SETS.items():
        assert set(env) <= set(SORT_SWITCHES), sset
        for c, route in cases.items():
            assert c in CASES, (sset, c)
            assert route in ROUTES, (sset, c, route)
            by_case.setdefault(c, []).append((sset, env, route))
    wrong, covered = [], set()
    for c in CASES:
        assert c in by_case, "case %s is in no switch set" % c
        keys, _, _, run = case_data(c)
        for sset, env, route in by_case[c]:
            got, tags, info = plan(run, keys, env)
            covered.add(got)
            if got != route:
                wrong.append((sset, c, route, got, info))
    assert not wrong, "\n".join("%s/%s: labelled %s, plans to %s %s" % w for w in wrong)
    assert covered == set(ROUTES), sorted(set(ROUTES) - covered)
    # the oversized-sub-bucket case is as large as the issue needs and no larger: it runs in one process only
    assert [s for s, (_, cs) in SWITCH_SETS.items() if "many_big_r12" in cs] == ["defaults"]


def test_planner_restates_edges():
    """Spot checks of the restated constants at their edges."""
    assert partition_bits(1 << 20, 511) == 9                    # 2048 per sub-bucket at P = 9: R == 0
    assert partition_bits(1_500_001, 511) is None               # P cannot grow past the key bits
    assert partition_bits(N_ODD, (1 << 22) - 1) == 10
    assert partition_bits(2700 * 512, (1 << 20) - 1) == 9 and partition_bits(2700 * 512 + 512, (1 << 20) - 1) == 10
    assert partition_bits(26_000_000, (1 << 26) - 1) == 14
    assert partition_bits(P_AVG * (1 << 16) + (1 << 16), (1 << 32) - 1) is None
    assert switches({}) == {"msd": 1, "big": 1, "fused_hist": 1, "probe": 1}
    assert switches({"QCE_MSD_BIG": "off"})["big"] == 0        # atoi: a value that is not a number reads as 0


# ---- GPU: every switch set in a fresh process (the switches are read once per process) --------------------------
def _make_run(e, name):
    keys, ids, col, run = case_data(name)
    rel = 121
    kind = run["kind"]
    if kind == "built":
        e.upload_column(rel, 0, col)
        return e.build_tuples(rel, 0)
    if kind == "built_ids":
        e.upload_column(rel, 0, col)
        h = e.rowids_from_host(ids)
        t = e.build_tuples(rel, 0, h)
        e.rowids_free(h)
        return t
    t = e.tuples_from_host(keys, ids)
    if kind == "device":
        counts, buf = e.partition_tuples(t, 32, [], 1)
        assert counts == [len(keys)]
        e.tuples_free(t)
        t = e.tuples_from_device_packed(buf, len(keys), 32, len(keys), run["key_min"], run["key_max"])
        e.exchange_release(buf)
    return t


def run_cases(cases):
    """Sort every (case, route) under this process's switches; return the list of failures."""
    import qce_b200
    from tests.test_gpu_primitives import _assert_sorted_run
    e = qce_b200.Engine()
    env = dict(os.environ)
    fails = []
    for name, label in cases:
        keys, ids, _, run = case_data(name)
        route, want, info = plan(run, keys, env)
        where = "%s (labelled %s, planned %s) planner inputs %s" % (name, label, route, json.dumps(info))
        try:
            assert route == label, "stale label"
            spec = CASES[name]
            t = _make_run(e, name)
            if spec.get("hist") is not None:
                e.key_histogram(t, spec["hist"])
            in_k, in_p = e.tuples_to_host(t)    # the order the sort starts from
            if run["kind"] == "device":         # the one-part partition may reorder the tuples, nothing else
                np.testing.assert_array_equal(np.sort((in_k << U64(32)) | in_p), np.sort((keys << U64(32)) | ids))
            else:
                np.testing.assert_array_equal(in_k, keys)
                np.testing.assert_array_equal(in_p, ids)
            e.profile(True)
            e.sort_tuples(t)
            prof = e.profile_read()
            e.profile(False)
            got = {tag: prof[tag]["launches"] for tag in WATCH if tag in prof}
            assert got == want, "launches %s, planned %s" % (got, want)
            assert e.is_sorted(t), "qce_tuples_is_sorted: not sorted"
            k, p = e.tuples_to_host(t)
            e.tuples_free(t)
            if route in STABLE:
                order = np.argsort(in_k, kind="stable")
                np.testing.assert_array_equal(k, in_k[order])
                np.testing.assert_array_equal(p, in_p[order])
            else:
                _assert_sorted_run(k, p, in_k, in_p)
            print("ok %s %s %s" % (name, route, json.dumps(got)), flush=True)
        except Exception as ex:  # noqa: BLE001 -- every case runs; the parent reports them all
            fails.append("%s: %s" % (where, str(ex)[:1500]))
            print("FAIL " + fails[-1], flush=True)
    return fails


_CHILD = r"""
import json, sys
sys.path.insert(0, %r)
from tests.test_gpu_sort_routes import run_cases
fails = run_cases(json.loads(sys.argv[1]))
print("ok" if not fails else "%%d failed" %% len(fails))
"""


@pytest.mark.gpu
@pytest.mark.parametrize("sset", list(SWITCH_SETS))
def test_sort_routes(sset):
    """Every case of the switch set in a fresh process: the launch profile shows the planned route, and the
    sorted run matches numpy's stable argsort (exactly on the stable routes, as a sorted multiset on MSD)."""
    env, cases = SWITCH_SETS[sset]
    base = {k: v for k, v in os.environ.items() if k not in SORT_SWITCHES}  # exactly this set's switches
    p = subprocess.run([sys.executable, "-c", _CHILD % ROOT, json.dumps(list(cases.items()))],
                       env=dict(base, **env), capture_output=True, text=True, timeout=1500)
    out = p.stdout.strip().splitlines()
    assert p.returncode == 0 and out and out[-1] == "ok", \
        "\n".join([l for l in out if not l.startswith("ok ")] + [p.stderr[-3000:]])
