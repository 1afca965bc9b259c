"""qce_build_sorted_tuples_base against qce_build_tuples_base + qce_sort_tuples on the same column.

A whole column with its level-A histogram (taken with the upload's statistics) whose run takes the MSD route is
sorted without being built first: MSD level A reads the column itself.  Every other column is built, then sorted.
Both give the same sorted keys, the same (key, row id) multiset and the same `skewed` flag (seen here as the join
route: a skewed run keeps the merge join off its single-pass kernel).  The launch profile shows which way a run
went; the expected launches come from the route planner of test_gpu_sort_routes.
"""
import json
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest

from tests.helpers import PKG
from tests.test_gpu_sort_routes import MSD_MIN_N, WATCH, partition_bits, plan

U64 = np.uint64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAGS = WATCH + ("build_tuples",)
N_ODD = 1_450_001


def _uniform(rng, n, bits):
    keys = rng.integers(0, 1 << bits, n, dtype=U64)
    keys[rng.integers(0, n)] = (1 << bits) - 1  # pin the bit length
    return keys


def _mixed(rng, n_small):
    """27-bit keys with every bit length below, keys < 128 among them; n_small keys of at most 17 bits."""
    bg = _uniform(rng, N_ODD, 27)
    lens = rng.integers(18, 27, 9000)
    mid = (U64(1) << lens.astype(U64)) | rng.integers(0, 1 << 17, len(lens), dtype=U64)
    small_lens = rng.integers(0, 18, n_small)
    small = rng.integers(0, 1 << 17, n_small, dtype=U64) & ((U64(1) << small_lens.astype(U64)) - U64(1))
    small[: min(300, n_small)] = rng.integers(0, 128, min(300, n_small), dtype=U64)
    return rng.permutation(np.concatenate([bg, mid, small]))


def _heavy(rng, bits, copies):
    keys = _uniform(rng, N_ODD, bits)
    keys[rng.choice(N_ODD, copies, replace=False)] = U64(12345 << (bits - 14))
    return keys


def column(name):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return {
        "n2^20-1_b27": lambda: _uniform(rng, (1 << 20) - 1, 27),
        "n2^20_b27": lambda: _uniform(rng, 1 << 20, 27),
        "n2^20+1_b22": lambda: _uniform(rng, (1 << 20) + 1, 22),         # last tile holds one odd word
        "n100M_b27": lambda: _uniform(rng, 100_000_000, 27),
        "b8": lambda: _uniform(rng, 1 << 20, 8),
        "b9": lambda: _uniform(rng, 1 << 20, 9),                            # R = 0, 2048 tuples per key: skewed
        "b27_odd": lambda: _uniform(rng, N_ODD, 27),
        "b32": lambda: _uniform(rng, N_ODD, 32),
        "mixed_lengths": lambda: _mixed(rng, 2000),
        "mixed_lengths_lsd": lambda: _mixed(rng, 400_000),                  # sub-bucket 0 too heavy, R = 17: LSD
        "dense_b9": lambda: _uniform(rng, 1_500_001, 9),                    # too dense for 16 partition bits
        "heavy_big_r12": lambda: _heavy(rng, 22, 5000),                     # R = 12: the big-bucket route
        "heavy_lsd_r13": lambda: _heavy(rng, 23, 5000),                     # R = 13: LSD after the fused level A
        "in_order": lambda: np.arange((1 << 20) + 1, dtype=U64) * U64(3),
        "wide": lambda: _uniform(rng, 1 << 20, 40),
        "empty": lambda: np.zeros(0, dtype=U64),
    }[name]()


# case -> the route of the fused entry ("fused" / "fused_lsd" / "unfused") under the default switches
CASES = {"n2^20-1_b27": "unfused", "n2^20_b27": "fused", "n2^20+1_b22": "fused", "n100M_b27": "fused",
         "b8": "unfused", "b9": "fused", "b27_odd": "fused", "b32": "fused", "mixed_lengths": "fused",
         "mixed_lengths_lsd": "fused_lsd", "dense_b9": "unfused", "heavy_big_r12": "fused",
         "heavy_lsd_r13": "fused_lsd", "in_order": "unfused", "wide": "unfused", "empty": "unfused"}


def _bitlen(x):
    return int(x).bit_length()


def has_hist(col):
    return len(col) >= MSD_MIN_N and 9 <= _bitlen(col.max()) <= 32


def expected(col, env):
    """(route, {tag: launches}) of qce_build_sorted_tuples_base on `col` under the switches in `env`."""
    n = len(col)
    top = int(col.max()) if n else 0
    kb = max(1, _bitlen(top))
    in_order = bool(np.all(col[1:] >= col[:-1]))
    run = {"kind": "built", "n": n, "key_bits": kb, "key_min": 0, "key_max": top, "wide": kb > 32, "built": True,
           "hist_arg": None, "in_order": in_order}
    route, tags, _ = plan(run, col, env)
    tags = dict(tags)
    fused = (env.get("QCE_FUSED_BUILD_SORT", "1") != "0" and has_hist(col) and not in_order
             and partition_bits(n, top) is not None)
    # the build's histogram and the column's are the same counts: the sort launches do not change
    tags["build_tuples"] = 0 if fused or n == 0 else 1
    if not fused:
        return "unfused", tags
    return ("fused_lsd" if route == "msd_lsd_fallback" else "fused"), tags


def _launches(e):
    prof = e.profile_read()
    return {t: prof[t]["launches"] for t in TAGS if t in prof and prof[t]["launches"]}


def _skewed(e, t, probe):
    """The run's skewed flag, read from the join route: a skewed side keeps the join off k_join_fused."""
    e.profile(True)
    oR, oS = e.merge_join(t, probe)
    prof = e.profile_read()
    e.profile(False)
    e.rowids_free(oR)
    e.rowids_free(oS)
    return "join_fused" not in prof


def run_cases(names):
    import qce_b200
    e = qce_b200.Engine()
    env = dict(os.environ)
    probe = e.tuples_from_host(np.array([1, 5], dtype=U64), np.array([0, 1], dtype=U64))
    e.sort_tuples(probe)
    fails = []
    for name in names:
        try:
            col = column(name)
            want_route, want = expected(col, env)
            if env.get("QCE_FUSED_BUILD_SORT") != "0":
                assert want_route == CASES[name], "stale label: planned %s" % want_route
            e.upload_column(7, 1, col)
            bins, kb = e.column_histogram(7, 1)
            if has_hist(col):
                b = _bitlen(col.max())
                assert kb == b, (kb, b)
                np.testing.assert_array_equal(bins, np.bincount((col >> U64(b - 8)).astype(np.int64), minlength=256))
            else:
                assert kb == 0 and bins is None, kb
            t0 = e.build_tuples(7, 1)
            e.sort_tuples(t0)
            k0, p0 = e.tuples_to_host(t0)
            skew0 = _skewed(e, t0, probe) if len(col) else False
            e.tuples_free(t0)
            e.profile(True)
            t = e.build_sorted_tuples(7, 1)
            got = _launches(e)
            e.profile(False)
            assert got == {k: v for k, v in want.items() if v}, "launches %s, planned %s" % (got, want)
            assert e.is_sorted(t)
            k, p = e.tuples_to_host(t)
            skew = _skewed(e, t, probe) if len(col) else False
            e.tuples_free(t)
            np.testing.assert_array_equal(k, k0)
            o, o0 = np.lexsort((p, k)), np.lexsort((p0, k0))  # the (key, row id) multisets
            np.testing.assert_array_equal(p[o], p0[o0])
            if len(col):
                np.testing.assert_array_equal(np.sort(k), np.sort(col))
                np.testing.assert_array_equal(np.sort(p), np.arange(len(col), dtype=U64))
            assert skew == skew0, (skew, skew0)
            print("ok %s %s %s skewed=%s" % (name, want_route, json.dumps(got), skew), flush=True)
        except Exception as ex:  # noqa: BLE001 -- every case runs; the parent reports them all
            fails.append("%s: %s" % (name, str(ex)[:1500]))
            print("FAIL " + fails[-1], flush=True)
    e.tuples_free(probe)
    return fails


def run_cache_and_reupload():
    """The same column twice in one batch: the second call borrows the cached run and launches nothing.
    A re-upload of the same shape with other keys replaces the column's histogram."""
    import qce_b200
    e = qce_b200.Engine()
    rng = np.random.default_rng(11)
    col = _uniform(rng, N_ODD, 27)
    e.upload_column(9, 0, col)
    assert e.lib.qce_batch_begin() == 0
    t1 = e.build_sorted_tuples(9, 0)
    k1, p1 = e.tuples_to_host(t1)
    e.profile(True)
    t2 = e.build_sorted_tuples(9, 0)
    prof = e.profile_read()
    e.profile(False)
    assert not any(v["launches"] for v in prof.values() if isinstance(v, dict) and "launches" in v), prof
    k2, p2 = e.tuples_to_host(t2)
    np.testing.assert_array_equal(k2, k1)
    np.testing.assert_array_equal(p2, p1)
    e.tuples_free(t1)
    e.tuples_free(t2)
    assert e.lib.qce_batch_end() == 0
    other = _uniform(rng, N_ODD, 25)
    other[:1000] = 7
    e.upload_column(9, 0, other)
    bins, kb = e.column_histogram(9, 0)
    assert kb == 25
    np.testing.assert_array_equal(bins, np.bincount((other >> U64(17)).astype(np.int64), minlength=256))
    e.upload_column(9, 0, _uniform(rng, 1000, 25))  # too short for a histogram
    assert e.column_histogram(9, 0) == (None, 0)
    t = e.build_sorted_tuples(9, 0)
    assert e.tuples_count(t) == 1000 and e.is_sorted(t)
    e.tuples_free(t)
    print("ok cache", flush=True)
    return []


_CHILD = r"""
import json, sys
sys.path.insert(0, %r)
from tests.test_gpu_build_sorted import run_cases, run_cache_and_reupload
arg = json.loads(sys.argv[1])
fails = run_cache_and_reupload() if arg == "cache" else run_cases(arg)
print("ok" if not fails else "%%d failed" %% len(fails))
"""


def _child(arg, env):
    base = {k: v for k, v in os.environ.items() if not k.startswith("QCE_")}
    p = subprocess.run([sys.executable, "-c", _CHILD % ROOT, json.dumps(arg)], env=dict(base, **env),
                       capture_output=True, text=True, timeout=1500)
    out = p.stdout.strip().splitlines()
    assert p.returncode == 0 and out and out[-1] == "ok", \
        "\n".join([l for l in out if not l.startswith("ok ")] + [p.stderr[-3000:]])


def test_cases_plan_to_their_labels():
    """The planner sends every case the way its label says (without a GPU)."""
    for name, label in CASES.items():
        if name == "n100M_b27":
            continue  # 100 M keys: planned in the GPU run only
        col = column(name)
        assert expected(col, {})[0] == label, name
        assert expected(col, {"QCE_FUSED_BUILD_SORT": "0"})[0] == "unfused", name


def test_host_layer_binds_the_engine_entry():
    """src/join.c references qce_build_sorted_tuples_base weakly, so that the host layer also links against the
    plain-C stand-in engine of its CPU tests.  Linked against the engine library, the reference must bind to it:
    otherwise every sorted base side would quietly be built, then sorted."""
    exe = os.path.join(PKG, "build", "queries")
    p = subprocess.run([exe], input=b"", env=dict(os.environ, LD_DEBUG="bindings"), capture_output=True, timeout=60)
    assert re.search(rb"binding file \S*queries \S* to \S*libqce_b200\.so \S*: normal symbol `qce_build_sorted_tuples_base'",
                     p.stderr), p.stderr[-2000:]


@pytest.mark.gpu
def test_build_sorted_matches_build_then_sort():
    """Every case, under the default switches, in a fresh process."""
    _child(list(CASES), {})


@pytest.mark.gpu
def test_build_sorted_switched_off():
    """QCE_FUSED_BUILD_SORT=0: every run is built, then sorted."""
    _child([c for c in CASES if c != "n100M_b27"], {"QCE_FUSED_BUILD_SORT": "0"})


@pytest.mark.gpu
def test_build_sorted_cache_and_reupload():
    _child("cache", {})
