"""Runs of 2^30 to 2^31 - 1 tuples: the tuple sort, the joins, distinct pairs, the re-join and the host layer.

The reference indexes a run with `int` (src/utilities.c:20), so it sorts and joins runs of up to 2^31 - 1 tuples; so
does the engine.  Above 2^30 tuples the LSD one-sweep passes sort every run (msd_plan sends such runs there), and the
inclusive prefix of a digit that holds most of the run passes 2^30 inside the look-back of k_onesweep.

Every check here is exact and linear in the run's length, with no host sort.  Keys are a closed form of the row index
(tools/benchkit.mix_t on the device, mix_np to check), so a sorted run of a whole base column is exactly the stable
sort of its input when: it holds n tuples, every row id is below n, every key is gen(row id), and (key, row id) is
strictly increasing.  Joins against a primary-key side arange(K) are checked against closed-form checksums.

Every test runs its cases in a fresh process, so the tens of GB each one holds on the device go back when it ends.
Each case prints its time."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N30, N31 = 1 << 30, (1 << 31) - 1
SKIP_RC = 3  # a child's exit code: the device cannot hold the case (the message says why)
GB = 1 << 30

# key families: (bits kept of mix(i, seed), bits forced on); every one is a closed form of the row index
KEYS = {
    "u32": (0xFFFFFFFF, 0),                    # uniform 32-bit keys: 4 passes
    "lowbyte": (0xFFFFFF00, 0x5A),             # constant low byte: pass 0 puts every tuple in one digit
    "b9": (0x1FF, 0),                          # 9-bit keys: 16 or more tuples per possible key, skewed
    "wide": ((1 << 40) - 1, 1 << 32),          # keys >= 2^32: the key / row-id sort (k_onesweep<true>), 5 passes
}
SEED = 11


def gen_np(i, kind):
    from tools import benchkit as bk
    keep, on = KEYS[kind]
    return (bk.mix_np(i, SEED) & np.uint64(keep)) | np.uint64(on)


def dev_column(torch, n, fn, step=1 << 27):
    """int64 device tensor x[i] = fn(arange), generated in slices so that the temporaries stay small"""
    out = torch.empty(n, dtype=torch.int64, device="cuda")
    for a in range(0, n, step):
        b = min(n, a + step)
        out[a:b] = fn(torch.arange(a, b, dtype=torch.int64, device="cuda"))
    return out


def gen_t(torch, kind):
    from tools import benchkit as bk
    keep, on = KEYS[kind]
    return lambda i: (bk.mix_t(torch, i, SEED) & keep) | on


def upload(e, torch, rel, col, n, fn):
    t = dev_column(torch, n, fn)
    torch.cuda.synchronize()
    e.upload_column_device(rel, col, t.data_ptr(), n)
    e.sync()
    del t
    torch.cuda.empty_cache()


def need_device(torch, nbytes, what):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        print("SKIP %s needs about %.0f GB of device memory, %.0f GB are free" % (what, nbytes / GB, free / GB))
        sys.exit(SKIP_RC)


def check_sorted_run(k, p, n, kind, step=1 << 27):
    """The sorted run (k, p) of a whole base column of n rows is the stable sort of (gen(i), i): n tuples, row ids
    below n, key == gen(row id), (key, row id) strictly increasing (which also makes the row ids a permutation)."""
    import torch
    assert len(k) == n and len(p) == n, (len(k), len(p), n)
    keep, on = KEYS[kind]
    gen = gen_t(torch, kind)
    kt, pt = torch.from_numpy(k.view(np.int64)), torch.from_numpy(p.view(np.int64))  # every value is below 2^63
    for a in range(0, n, step):
        b = min(n, a + step)
        lo = max(a - 1, 0)  # the slices overlap by one: the order also holds across their seams
        kc, pc = kt[lo:b], pt[lo:b]
        assert bool((pc < n).all()), "row id out of range in [%d, %d)" % (lo, b)
        assert bool((kc == gen(pc)).all()), "key != gen(row id) in [%d, %d)" % (lo, b)
        inc = (kc[1:] > kc[:-1]) | ((kc[1:] == kc[:-1]) & (pc[1:] > pc[:-1]))
        assert bool(inc.all()), "(key, row id) not strictly increasing in [%d, %d)" % (lo, b)
    # a spot check of the same closed form through numpy, independent of torch
    idx = np.linspace(0, n - 1, 4097).astype(np.int64)
    np.testing.assert_array_equal(k[idx], gen_np(p[idx], kind))


WATCH = ("block_sort", "radix_hist", "onesweep_k", "onesweep_kv", "msd_hist", "msd_partition", "msd_count_sort",
         "msd_local_sort", "msd_big_partition")


def launches(prof):
    return {t: v["launches"] for t, v in prof.items() if v.get("launches")}


def expected_launches(n, kind, kmax):
    """the sort's launch profile: below 2^30 the route planner of test_gpu_sort_routes; from 2^30 on the LSD passes
    alone -- one digit histogram and one one-sweep pass per digit, no MSD kernel"""
    key_bits = max(1, int(kmax).bit_length())
    npass = -(-key_bits // 8)
    if kind == "wide":
        return {"radix_hist": 1, "onesweep_kv": npass}
    if n < N30:
        from tests.test_gpu_sort_routes import plan
        run = {"kind": "built", "n": n, "key_bits": key_bits, "key_min": 0, "key_max": kmax, "wide": False,
               "built": True, "hist_arg": None, "in_order": False}
        # `keys` is only read once a partition-bit count is found, which no run of this size and width gets
        route, want, _ = plan(run, None, dict(os.environ))
        assert route == "lsd", route
        return want
    return {"radix_hist": 1, "onesweep_k": npass}


def skewed(e, t):
    """the run's skewed flag, read from the join route: a skewed side keeps the join off k_join_fused"""
    probe = e.tuples_from_host(np.array([1, 5], dtype=np.uint64), np.array([0, 1], dtype=np.uint64))
    e.sort_tuples(probe)
    e.profile(True)
    oR, oS = e.merge_join(t, probe)
    prof = e.profile_read()
    e.profile(False)
    for h in (oR, oS):
        e.rowids_free(h)
    e.tuples_free(probe)
    return "join_fused" not in prof


# ---- children ---------------------------------------------------------------------------------------------------
def child_sort(kind, sizes):
    """Build a whole base column of n rows of `kind` keys, sort it, check the launch profile and the run."""
    import torch
    import qce_b200
    e = qce_b200.Engine()
    per = 28 if kind == "wide" else 24  # column + run + its sort buffer (+ ids) bytes per row, + 2 GB of status
    need_device(torch, max(sizes) * per + 2 * GB, "%s sort of %d tuples" % (kind, max(sizes)))
    for n in sizes:
        t0 = time.time()
        upload(e, torch, 70, 0, n, gen_t(torch, kind))
        _, kmax = e.column_info(70, 0)
        want = expected_launches(n, kind, kmax)
        t = e.build_tuples(70, 0)
        e.profile(True)
        t1 = time.time()
        e.sort_tuples(t)
        e.sync()
        t_sort = time.time() - t1
        prof = e.profile_read()
        e.profile(False)
        got = {k: v for k, v in launches(prof).items() if k in WATCH}
        assert got == want, (kind, n, got, want)
        assert not [k for k in launches(prof) if k.startswith("msd_")], (kind, n, launches(prof))
        skew = skewed(e, t) if kind == "b9" else None
        if kind == "b9":
            assert skew, "a run of 9-bit keys with %d tuples is not flagged skewed" % n
        k, p = e.tuples_to_host(t)
        e.tuples_free(t)
        e.drop_relations()
        check_sorted_run(k, p, n, kind)
        del k, p
        print("case sort %s n=%d passes=%s sort %.3f s (wall, incl. launch profile), case %.1f s%s" % (
            kind, n, want.get("onesweep_k", want.get("onesweep_kv")), t_sort, time.time() - t0,
            "" if skew is None else " skewed=%s" % skew), flush=True)


def child_join(nfk, K):
    """FK side of nfk rows, fk = gen(i) mod K, against a PK side arange(K): merge join, merge join with stats, and for
    the wide key range distinct pairs and the re-join on the join's output."""
    import ctypes as C
    import torch
    import qce_b200
    from tools import benchkit as bk
    e = qce_b200.Engine()
    need_device(torch, nfk * 60 + 8 * GB, "join of %d tuples" % nfk)
    t0 = time.time()
    fk = lambda i: bk.mix_t(torch, i, SEED) & (K - 1)  # noqa: E731
    upload(e, torch, 60, 0, nfk, fk)                   # FK keys
    upload(e, torch, 60, 1, nfk, lambda i: i)          # row index: sum over a join output = n(n-1)/2
    upload(e, torch, 61, 0, K, lambda i: i)            # PK keys arange(K), stored in order
    sum_fk = int(dev_column(torch, nfk, fk).sum().item())
    sum_i = nfk * (nfk - 1) // 2
    L = e.build_tuples(60, 0)
    R = e.build_tuples(61, 0)
    e.sort_tuples(L)
    e.sort_tuples(R)
    assert e.is_sorted(L)
    skew = skewed(e, L)
    assert skew == (nfk // K >= 16), (skew, nfk, K)
    t1 = time.time()
    e.profile(True)
    oL, oR = e.merge_join(L, R)
    e.sync()
    t_join = time.time() - t1
    prof = launches(e.profile_read())
    e.profile(False)
    assert ("join_fused" in prof) == (not skew), prof
    assert e.rowids_count(oL) == nfk and e.rowids_count(oR) == nfk
    assert e.checksum(oL, 60, [1])[0] == sum_i            # every FK row exactly once
    assert e.checksum(oL, 60, [0])[0] == sum_fk           # the FK keys that matched
    assert e.checksum(oR, 61, [0])[0] == sum_fk           # == the PK keys they met
    # merge join with stats: every FK row meets exactly one PK row
    sR, sS, mn, mx = C.c_void_p(), C.c_void_p(), C.c_uint32(), C.c_uint32()
    e._ck(e.lib.qce_merge_join_stats(L, R, C.byref(sR), C.byref(sS), C.byref(mn), C.byref(mx)))
    assert e.rowids_count(sR.value) == nfk and e.rowids_count(sS.value) == nfk
    assert (mn.value, mx.value) == (1, 1), (mn.value, mx.value)
    assert e.checksum(sR.value, 60, [1])[0] == sum_i and e.checksum(sS.value, 61, [0])[0] == sum_fk
    e.rowids_free(sR.value)
    e.rowids_free(sS.value)
    print("case join nfk=%d K=%d skewed=%s route=%s join %.3f s (wall, incl. launch profile)" % (
        nfk, K, skew, "single-pass" if "join_fused" in prof else "two-phase", t_join), flush=True)
    e.tuples_free(L)
    e.tuples_free(R)
    if not skew:
        # distinct pairs of the join output: all nfk pairs are distinct
        t1 = time.time()
        dL, dR = e.distinct_pairs(oL, oR)
        e.sync()
        t_dist = time.time() - t1
        assert e.rowids_count(dL) == nfk and e.rowids_count(dR) == nfk
        assert e.checksum(dL, 60, [1])[0] == sum_i and e.checksum(dR, 61, [0])[0] == sum_fk
        e.rowids_free(dL)
        e.rowids_free(dR)
        # re-join a bystander: `last` = every FK row, `edit` = the PK row each FK row points at (its fk value);
        # driven by the join's FK side, the re-joined bystander is fk[oL[j]], whose PK keys sum to sum(fk)
        e.rowids_free(oR)
        last = e.rowids_iota(0, nfk, nfk)
        edit = e.column_gather_u32(60, 0, last)
        t1 = time.time()
        out = e.rejoin(oL, last, edit)
        e.sync()
        t_rejoin = time.time() - t1
        assert e.rowids_count(out) == nfk
        assert e.checksum(out, 61, [0])[0] == sum_fk
        for h in (out, last, edit):
            e.rowids_free(h)
        print("case distinct_pairs n=%d %.3f s, rejoin n=%d %.3f s" % (nfk, t_dist, nfk, t_rejoin), flush=True)
    else:
        e.rowids_free(oR)
    e.rowids_free(oL)
    print("case join total %.1f s" % (time.time() - t0), flush=True)


# relation 0: N0 rows (values, FK into relation 1 and 2, row index for the filter); relations 1 and 2: PK arange(K)
E2E_N0, E2E_K, E2E_C = 1_200_000_000, 1 << 27, 100_000_000
E2E_QUERIES = ["0 1|0.1=1.0&0.2>%d|0.0 1.1\n" % E2E_C,
               "0 1 2|0.1=1.0&0.1=2.0&0.2>%d|0.0 1.1 2.1\n" % E2E_C]


def e2e_columns(torch):
    from tools import benchkit as bk
    return {
        (0, 0): (E2E_N0, lambda i: bk.mix_t(torch, i, 5) & 0xFFFFFFFF),
        (0, 1): (E2E_N0, lambda i: bk.mix_t(torch, i, 6) & (E2E_K - 1)),
        (0, 2): (E2E_N0, lambda i: i),
        (1, 0): (E2E_K, lambda i: i),
        (1, 1): (E2E_K, lambda i: bk.mix_t(torch, i, 7) & 0xFFFFFF),
        (2, 0): (E2E_K, lambda i: i),
        (2, 1): (E2E_K, lambda i: bk.mix_t(torch, i, 8) & 0xFFFFFF),
    }


def e2e_expected(torch, cols):
    """the lines the queries print, from closed forms on the device: the rows of relation 0 past the filter, each
    with the one row of relations 1 and 2 its FK points at"""
    r1 = dev_column(torch, E2E_K, cols[(1, 1)][1])
    r2 = dev_column(torch, E2E_K, cols[(2, 1)][1])
    s0 = s1 = s2 = 0
    step = 1 << 27
    for a in range(E2E_C + 1, E2E_N0, step):
        i = torch.arange(a, min(E2E_N0, a + step), dtype=torch.int64, device="cuda")
        fk = cols[(0, 1)][1](i)
        s0 += int(cols[(0, 0)][1](i).sum().item())
        s1 += int(r1[fk].sum().item())
        s2 += int(r2[fk].sum().item())
    m = (1 << 64) - 1
    return ["%d %d \n" % (s0 & m, s1 & m), "%d %d %d \n" % (s0 & m, s1 & m, s2 & m)]


def child_e2e(which):
    """The host layer's batch entry (qce_host_run_batch) through bench.Rig, columns generated on the device."""
    import torch
    import bench
    rig = bench.Rig(torch, None, 0, 1, 0)
    need_device(torch, 75 * GB, "the end-to-end queries")
    cols = e2e_columns(torch)
    for (rel, col), (rows, fn) in cols.items():
        rig.upload_fn(rel, col, rows, lambda b, c, fn=fn: dev_column(torch, c, lambda i: fn(i + b)))
    torch.cuda.empty_cache()
    want = e2e_expected(torch, cols)
    torch.cuda.empty_cache()
    for q, w in zip(E2E_QUERIES, want):
        if which == "faithful" and q.startswith("0 1|"):
            continue  # the faithful replay only changes the query with a bystander
        t1 = time.time()
        got = rig.run(q)
        dt = time.time() - t1
        assert got == w, (q, got, w)
        print("case e2e %s %r %.3f s (wall, first run)" % (which, q.strip(), dt), flush=True)


def child_limit():
    """A base column of exactly 2^31 rows builds; its sort is refused with the limit's message; a small join after
    that still gives the right answer."""
    import torch
    import qce_b200
    e = qce_b200.Engine()
    n = 1 << 31
    need_device(torch, n * 16 + 2 * GB, "the 2^31-row column")
    upload(e, torch, 70, 0, n, gen_t(torch, "u32"))
    t = e.build_tuples(70, 0)
    assert e.tuples_count(t) == n
    try:
        e.sort_tuples(t)
    except qce_b200.EngineError as ex:
        msg = str(ex)
    else:
        raise AssertionError("a sort of 2^31 tuples was not refused")
    assert "2147483648 tuples" in msg and "2^31 - 1" in msg, msg
    e.tuples_free(t)
    e.drop_relations()
    # a small join afterwards
    rng = np.random.default_rng(5)
    m = 100_000
    pk = rng.permutation(m).astype(np.uint64)
    fk = rng.integers(0, m, 3 * m, dtype=np.uint64)
    e.upload_column(80, 0, fk)
    e.upload_column(81, 0, pk)
    L, R = e.build_tuples(80, 0), e.build_tuples(81, 0)
    e.sort_tuples(L)
    e.sort_tuples(R)
    oL, oR = e.merge_join(L, R)
    assert e.rowids_count(oL) == 3 * m
    assert e.checksum(oR, 81, [0])[0] == int(fk.sum())
    print("case limit: %s; a join afterwards is right" % msg, flush=True)


CHILDREN = {"sort": child_sort, "join": child_join, "e2e": child_e2e, "limit": child_limit}

_CHILD = r"""
import json, sys
sys.path.insert(0, %r)
from tests.test_gpu_big_runs import CHILDREN
name, args = sys.argv[1], json.loads(sys.argv[2])
CHILDREN[name](*args)
print("ok")
"""


def run_child(name, *args, env=None, timeout=1500):
    import json
    t0 = time.time()
    p = subprocess.run([sys.executable, "-c", _CHILD % ROOT, name, json.dumps(args)], capture_output=True, text=True,
                       timeout=timeout, env=dict(os.environ, **(env or {})))
    out = p.stdout.strip().splitlines()
    for line in out:
        print(line)
    print("%s%s: %.1f s" % (name, args, time.time() - t0))
    if p.returncode == SKIP_RC:
        pytest.skip(" ".join(l for l in out if l.startswith("SKIP")))
    assert p.returncode == 0 and out and out[-1] == "ok", "\n".join(out[-20:] + [p.stderr[-3000:]])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u32", "lowbyte"])
def test_packed_sort(kind):
    """Packed sort at 2^30 - 1, 2^30, 2^30 + 1 and 2^31 - 1 tuples: exactly the stable sort, and the launches the
    route planner predicts below 2^30 / the LSD passes alone from 2^30 on."""
    run_child("sort", kind, [N30 - 1, N30, N30 + 1, N31])


@pytest.mark.gpu
def test_packed_sort_9bit_is_skewed():
    """9-bit keys at 2^30 + 1 tuples (2^21 tuples per key): sorted exactly, and flagged skewed."""
    run_child("sort", "b9", [N30 + 1])


@pytest.mark.gpu
def test_wide_sort():
    """Keys >= 2^32 (the key / row-id one-sweep) at 2^30 + 1 tuples: exactly the stable sort."""
    run_child("sort", "wide", [N30 + 1])


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1 << 27, 1 << 9])
def test_join_of_big_runs(K):
    """An FK side of 1.2 G rows against a PK side arange(K): both joins give one pair per FK row with the closed-form
    checksums; K = 2^27 takes the single-pass join and also checks distinct pairs and the re-join on its 1.2 G pairs,
    K = 2^9 (skewed) takes the two-phase join."""
    run_child("join", 1_200_000_000, K)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["elide", "faithful"])
def test_end_to_end(which):
    """qce_host_run_batch over a 1.2 G-row relation with a filter keeping 1.1 G rows: a 2-way join, and a 3-binding
    query whose bystander is re-aligned by elision (default) or by the faithful re-joins (QCE_ELIDE=0), which sort
    pair words of 1.1 G tuples."""
    run_child("e2e", which, env={"QCE_ELIDE": "1" if which == "elide" else "0"})


@pytest.mark.gpu
def test_sort_limit():
    """2^31 tuples: the sort is refused with the limit's message, and the engine stays usable."""
    run_child("limit")
