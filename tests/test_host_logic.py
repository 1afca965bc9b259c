"""CPU: the C host layer's parser/arranger against the reference's recorded
orders, and the C-ABI library's exported symbols against include/qce_b200.h."""
import os
import re
import subprocess

import pytest

from tests.helpers import HOST_PROBE, ROOT, load_json


def _build():
    import __graft_entry__
    __graft_entry__.build()


@pytest.fixture(scope="module", autouse=True)
def built():
    if not os.path.exists(HOST_PROBE):
        _build()


def _probe(lines):
    out = subprocess.run([HOST_PROBE], input="".join(lines).encode(), stdout=subprocess.PIPE, check=True).stdout.decode()
    rows = out.splitlines()
    return rows[0::2], rows[1::2]


def test_host_arranger_matches_reference():
    recs = load_json("arrange.json")
    orders, _ = _probe([f"0 1 2 3|{r['written']}|0.0\n" for r in recs])
    assert len(orders) == len(recs)
    for got, rec in zip(orders, recs):
        assert got == rec["executed"], rec["written"]


def test_host_parser_sections():
    orders, meta = _probe(["F\n", "3 0 1|0.2=1.0&0.1=2.0&0.2>3499|1.2 0.1\n", "\n", "0|0.1=4294967297|0.0\n"])
    assert orders == ["0.2>3499 0.2=1.0 0.1=2.0", "0.1=1"]
    assert meta[0] == "#rels=3 sels=2 r3 r0 r1 s1.2 s0.1"
    assert meta[1] == "#rels=1 sels=1 r0 s0.0"


def test_malformed_lines_are_skipped_not_executed():
    """Parser hardening (SURVEY 8f-4): an unparsable predicate element or a binding index outside the
    relation list is refused with a diagnostic; the well-formed lines around it are unaffected.
    (The reference sizes its arrays by separator counts and executes whatever sscanf left there.)"""
    lines = ["0 1|0.1=1.1|0.0\n",
             "9999999999|9999999999|9999999999\n",        # no predicate at all in the predicate section
             "0 1|0.1=1.1&0.2|0.0\n",                    # second element has no operator
             "0 1|0.1=2.1|0.0\n",                        # binding 2 of a 2-relation query
             "0 1|0.1=1.1|2.0\n",                        # select on binding 2
             "0 1|0.1=1.1&&0.2<5|0.0\n",                 # empty element
             "0|0.2<5|0.0\n"]
    p = subprocess.run([HOST_PROBE], input="".join(lines).encode(), stdout=subprocess.PIPE, stderr=subprocess.PIPE, check=True)
    rows = p.stdout.decode().splitlines()
    assert rows[0::2] == ["0.1=1.1", "0.2<5"]
    assert p.stderr.decode().count("malformed query line skipped") == 5


def test_loader_rejects_implausible_headers(tmp_path):
    """The relation file header is untrusted (src/utilities.c:105-121 trusts it): a rows x columns
    product that wraps around, or more cells than the file holds, fails before anything is uploaded."""
    import numpy as np
    from tests.helpers import QUERIES_BIN, REFMAIN_BIN
    # our driver and, where it was built, the reference's unchanged main: both call read_relations
    # before anything touches the device
    binaries = [QUERIES_BIN] + ([REFMAIN_BIN] if os.path.exists(REFMAIN_BIN) else [])
    cases = {"wrap": np.array([1 << 61, 8, 1, 2, 3], dtype=np.uint64),       # 2^61 * 8 wraps to 0
             "trunc": np.array([1000, 3, 1, 2, 3], dtype=np.uint64),
             "huge_rows": np.array([1 << 33, 1, 5], dtype=np.uint64),
             "short": np.array([7], dtype=np.uint64)}
    for binary in binaries:
        for name, words in cases.items():
            path = tmp_path / name
            words.tofile(path)
            p = subprocess.run([binary], input=f"{path}\nDone\n".encode(), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            err = p.stderr.decode()
            assert p.stdout == b"", (binary, name)
            assert ("implausible relation header" in err or "truncated" in err or "too short" in err), (binary, name, err)


def test_library_exports_every_declared_symbol():
    import qce_b200
    header = open(os.path.join(ROOT, "include", "qce_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(qce_[a-z0-9_]+)\s*\(", header)))
    assert declared == sorted(qce_b200.SYMBOLS)
    lib = qce_b200.load_library()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.qce_abi_version() >= 1


def test_engine_refuses_to_run_without_a_gpu():
    import torch
    import qce_b200
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(qce_b200.EngineError, match="no CPU path"):
        qce_b200.Engine()


def test_hbm_arena_free_list_on_cpu(tmp_path):
    """The engine's HBM arena (csrc/qce_arena.hpp: best-fit free list over large slabs, coalescing, and the
    shrink that trims a join output sized by a guess) compiled with malloc-backed slabs and driven with random
    alloc / free / shrink traffic under ASan + UBSan: live and free blocks tile every slab, free neighbours are
    always merged, everything comes back, and the steady single-pass-join loop reuses the same addresses."""
    exe = str(tmp_path / "arena_test")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-o", exe,
                    os.path.join(ROOT, "tests", "c", "arena_test.cpp")], check=True)
    p = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120)
    assert p.returncode == 0 and p.stdout.decode().strip() == "arena ok", p.stderr.decode()[-2000:]


_SEARCH_HARNESS = r"""
#include <stdio.h>
#include <stdlib.h>
#include <stddef.h>
#include <algorithm>
#include <random>
#include <vector>
typedef unsigned long long u64;
typedef unsigned int u32;
#define __device__
#define __forceinline__ inline
struct TupleView { const u64 *a; const u32 *ids; };
template <bool WIDE> u64 tv_key(const TupleView &t, size_t i) { return WIDE ? t.a[i] : (t.a[i] >> 32); }
%s
int main()
{
    std::mt19937_64 rng(3);
    long checked = 0;
    for (int round = 0; round < 400; round++) {
        const u32 n = 1 + (u32)(rng() %% (round %% 7 == 0 ? 40000 : 300));
        const u64 domain = 1 + rng() %% (round %% 3 == 0 ? 5 : (round %% 3 == 1 ? n : 4ull * n));
        std::vector<u64> keys(n), packed(n);
        for (auto &k : keys) k = rng() %% domain;
        std::sort(keys.begin(), keys.end());
        for (u32 i = 0; i < n; i++) packed[i] = (keys[i] << 32) | i;
        TupleView wide{keys.data(), nullptr}, pk{packed.data(), nullptr};
        for (int q = 0; q < 300; q++) {
            u32 lo = (u32)(rng() %% n), hi = lo + (u32)(rng() %% (n - lo + 1));
            if (q %% 5 == 0) { lo = 0; hi = n; }
            const u64 key = q %% 11 == 0 ? domain + 3 : rng() %% (domain + 1);
            u32 g = lo;
            if (hi > lo) g = q %% 4 == 0 ? lo : (q %% 4 == 1 ? hi - 1 : lo + (u32)(rng() %% (hi - lo)));
            const u32 wl = (u32)(std::lower_bound(keys.begin() + lo, keys.begin() + hi, key) - keys.begin());
            const u32 wu = (u32)(std::upper_bound(keys.begin() + lo, keys.begin() + hi, key) - keys.begin());
            if (bound_from_guess<true, false>(wide, lo, hi, g, key) != wl || bound_from_guess<true, true>(wide, lo, hi, g, key) != wu ||
                bound_from_guess<false, false>(pk, lo, hi, g, key) != wl || bound_from_guess<false, true>(pk, lo, hi, g, key) != wu) {
                fprintf(stderr, "mismatch: n %%u lo %%u hi %%u g %%u key %%llu\n", n, lo, hi, g, key);
                return 1;
            }
            // the way the kernels chain the two: the upper bound starts at the lower bound
            if (hi > lo && bound_from_guess<true, true>(wide, wl, hi, std::min(wl, hi - 1), key) != wu) return 2;
            checked++;
        }
    }
    printf("search ok %%ld\n", checked);
    return 0;
}
"""


def test_guess_and_gallop_search_on_cpu(tmp_path):
    """bound_from_guess (csrc/k_join.cuh: the join's search over windows too large to stage -- start at an
    interpolated guess, gallop until the answer is bracketed, bisect) is lifted from the shipped source as it
    stands and held to std::lower_bound / std::upper_bound on random sorted runs: duplicates, sub-ranges, guesses at
    both ends, keys outside the run, packed and wide tuples."""
    src = open(os.path.join(ROOT, "query-compiler-executor_b200", "csrc", "k_join.cuh")).read()
    m = re.search(r"template <bool WIDE, bool UPPER>\n__device__ __forceinline__ u32 bound_from_guess.*?\n    return lo;\n}\n", src, re.S)
    assert m, "bound_from_guess not found in k_join.cuh"
    cpp = tmp_path / "search_test.cpp"
    cpp.write_text(_SEARCH_HARNESS % m.group(0))
    exe = str(tmp_path / "search_test")
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-o", exe, str(cpp)], check=True)
    p = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120)
    assert p.returncode == 0 and p.stdout.decode().startswith("search ok"), (p.stdout.decode(), p.stderr.decode()[-2000:])
