#!/usr/bin/env python
"""bench.py -- the reference's headline workloads on B200.

Metric (BASELINE.json): join input rows/s (and queries/s for the batch config).

  python bench.py [--gpus N --steps K --warmup W]     headline = config 2 (BASELINE.json configs[1]):
      single 2-way equi-join + range filter over 2 x 100M-row relations of 3 uint64 columns, query
      `0 1|0.1=1.1&0.2>500000|0.0 1.0 1.2` (SURVEY.md 8d).  The same line carries, under "configs",
      runs of configs 3, 4 and 5 at their BASELINE sizes: the 4-way chain at 62.5M rows per relation
      per GPU (500M over 8 GPUs), the Zipf(1.2) 3-way join at 100M rows per relation per GPU, and the
      1000-query batch over 14 relations of 10^6..10^9 rows.  Every config (and every leg of config 2)
      runs --warmup untimed steps, then --steps timed ones; a config-5 step is ~6 s on one GPU.
  python bench.py --config c3|c4|c5 ...                that config alone, at full size, as the line's workload
  python bench.py --impl reference ...                 the reference's own CPU binary (oracle/_ref/queries)
                                                       on the config-2 scaled twin

Every step goes through the reference-facing boundary: query text -> libqce_host.so (parse, arrange,
execute_filter / execute_join / print_sums -- the host operator layer of src/) -> libqce_b200.so
(C-ABI, CUDA).  With N > 1 (torchrun, one process per GPU) nothing changes above the C-ABI: the
ranks meet through qce_comm_attach and the SAME host layer runs SPMD; the operators exchange tuples
over NVLink peer windows (csrc/qce_shard.cuh).  torch is used for device RNG, pinned host buffers,
the independent checkers and the max-over-ranks reduction of the timings -- never inside a step.

Every config is self-verifying (the line's "parity" block):
  twin_vs_reference   a scaled twin of the workload (same generator family) runs through the product
                      path -- sharded over the N ranks when N > 1 -- and its stdout is compared byte for
                      byte with the unmodified reference binary's (oracle/_ref/queries) on the same files
  full_vs_checker     the full-size result is compared with an independent linear-time checker
                      (tools/benchkit.py: bincount closed form for config 2, index maps for 3/4/5 --
                      no sort, no merge, no code shared with the engine)

  value     rows/s with the base columns already resident in HBM
  e2e       headline only: every step first copies the referenced columns from pinned host memory
  roofline  per-kernel live CUDA-event times against the measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline  the reference binary on the config-2 scaled twin, on this box's host cores

  --dump-outputs DIR  after the timed steps, writes what the last timed step of every config returned
                      (the checksum lines the host layer prints) as DIR/<config>.npy; see dump_outputs
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = os.path.join(ROOT, "query-compiler-executor_b200")
METRIC = "join_input_rows_per_s"
QUERY = "0 1|0.1=1.1&0.2>{thr}|0.0 1.0 1.2\n"
REF_SAMPLE_ROWS = 1_000_000  # per relation: ~2-3 s of the (output-quadratic) CPU reference per step
M64 = (1 << 64) - 1


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  In-process
    NVML (a `nvidia-smi -lms 100` child perturbed the CUDA driver enough to cost
    ~25 % of a 10 ms step); nvidia-smi at 200 ms is the fallback."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period=0.05):
        self.index, self.period, self.sm, self.reasons, self.max_mhz = index, period, [], set(), None
        self._stop, self._thr, self._smi = threading.Event(), None, None

    def start(self):
        if self.period <= 0:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for name, bit in self.BAD.items():
                            if r & bit:
                                self.reasons.add(name)
                    except Exception:
                        pass
                    self._stop.wait(self.period)
            self._thr = threading.Thread(target=loop, daemon=True)
            self._thr.start()
        except Exception:
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            try:
                self._smi = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                              "--format=csv,noheader,nounits", "-lms", "200"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self._smi = None

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1.0)
        if self._smi:
            time.sleep(0.25)
            self._smi.terminate()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for line in self._smi.stdout.read().splitlines():
                f = [x.strip() for x in line.split(",")]
                try:
                    self.sm.append(float(f[0])); self.max_mhz = float(f[1])
                except Exception:
                    continue
                for nme, v in zip(names, f[2:6]):
                    if v == "Active":
                        self.reasons.add(nme)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ------------------------------------------------------------------ config 2 data (numpy default_rng family)
def gen_relation(rows, seed, key_domain, row_base=0):
    rng = np.random.default_rng(seed)
    return [np.arange(row_base, row_base + rows, dtype=np.uint64),
            rng.integers(0, key_domain, rows, dtype=np.uint64),
            rng.integers(0, 10 ** 6, rows, dtype=np.uint64)]


# ------------------------------------------------------------------ CPU reference arm
def time_reference(rows, steps, warmup):
    """The unmodified reference binary (single-threaded C) on a scaled twin of the
    workload; per step: whole-process wall time minus a load-only run."""
    from oracle import workload as wl
    if not wl.have_reference():
        return None
    db = [gen_relation(rows, 1, rows), gen_relation(rows, 2, rows)]
    d = tempfile.mkdtemp(prefix="qce_ref_")
    paths = wl.write_db(d, db)
    q = QUERY.format(thr=500000)
    t = time.time(); wl.run_reference(paths, ""); load_s = time.time() - t
    times, out = [], ""
    for i in range(warmup + steps):
        t = time.time()
        out, err, rc = wl.run_reference(paths, q)
        dt = time.time() - t
        if rc != 0:
            raise RuntimeError("reference failed: " + err)
        if i >= warmup:
            times.append(max(dt - load_s, 1e-9))
    for p in paths:
        os.unlink(p)
    sec = float(np.mean(times))
    return {"rows_per_s": 2 * rows / sec, "sec_per_step": sec, "load_s": load_s, "stdout": out.strip()}


def dump_outputs(outdir, outputs):
    """outputs: config name -> stdout text of its last timed step.  Every value printed there (a uint64
    checksum, a count, or NULL) becomes one row (line, high 32 bits, low 32 bits) of a float64 array, exact
    (NULL = NaN in both halves), so two builds can be compared output for output with numpy:
    np.array_equal(a, b, equal_nan=True).  The reference arm (--impl reference) writes reference_c2_twin."""
    os.makedirs(outdir, exist_ok=True)
    for name, text in outputs.items():
        rows = []
        for ln, line in enumerate(text.splitlines()):
            for tok in line.split():
                if tok == "NULL":
                    rows.append((ln, np.nan, np.nan))
                else:
                    v = int(tok)
                    rows.append((ln, float(v >> 32), float(v & 0xFFFFFFFF)))
        np.save(os.path.join(outdir, name + ".npy"), np.array(rows, dtype=np.float64).reshape(-1, 3))


# ------------------------------------------------------------------ the engine as bench.py sees it
class Rig:
    """The product as an embedder sees it: libqce_b200.so (C-ABI) + libqce_host.so (the host operator
    layer's batch entry).  One per process / rank."""

    def __init__(self, torch, dist, rank, world, local_rank):
        import qce_b200
        self.torch, self.dist, self.rank, self.world = torch, dist, rank, world
        self.lib = qce_b200.load_library()
        if world > 1:
            # the ranks of the node meet in /dev/shm (no torch inside the engine); rank 0's random
            # token tells this run's segment from a stale one
            tok = torch.randint(1, 1 << 62, (1,), dtype=torch.int64, device="cuda")
            dist.broadcast(tok, 0)
            name = "qce_bench_%s" % os.environ.get("MASTER_PORT", "0")
            if self.lib.qce_comm_attach(name.encode(), rank, world, int(tok.item())) != 0:
                raise RuntimeError(self.lib.qce_last_error().decode())
        self.eng = qce_b200.Engine(local_rank)
        C.CDLL(os.path.join(PKG, "libqce_b200.so"), mode=C.RTLD_GLOBAL)
        self.host = C.CDLL(os.path.join(PKG, "libqce_host.so"))
        self.host.qce_host_run_batch.restype = C.c_long
        self.host.qce_host_run_batch.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_int)]
        self._buf = C.create_string_buffer(1 << 20)

    def ck(self, rc):
        if rc != 0:
            raise RuntimeError(self.lib.qce_last_error().decode())

    def run(self, text):
        """query text -> the bytes the reference would print (every rank gets the sharded queries' lines,
        rank 0 everything)"""
        failed = C.c_int(0)
        n = self.host.qce_host_run_batch(text.encode(), self._buf, len(self._buf), C.byref(failed))
        if n < 0 or failed.value:
            raise RuntimeError("host layer failed %d queries: %s" % (failed.value, self.lib.qce_last_error().decode()))
        return self._buf.value.decode()

    def arena(self):
        """(reserved, in use) bytes of the engine's HBM arena, or None"""
        try:
            return self.eng.mempool_stats()
        except Exception:
            return None

    def share(self, rows):
        b, c = C.c_uint64(), C.c_uint64()
        self.ck(self.lib.qce_row_share(rows, self.rank, self.world, C.byref(b), C.byref(c)))
        return b.value, c.value

    def whole(self, rows):
        return self.world == 1 or self.lib.qce_column_would_be_whole(rows) == 1

    def upload_fn(self, rel, col, rows, make):
        """make(begin, count) -> device int64 tensor of those rows; the engine keeps its own copy"""
        if self.whole(rows):
            t = make(0, rows)
            self.torch.cuda.synchronize()
            self.ck(self.lib.qce_upload_column_device(rel, col, t.data_ptr(), rows))
        else:
            b, c = self.share(rows)
            t = make(b, c)
            self.torch.cuda.synchronize()
            self.ck(self.lib.qce_upload_column_window_device(rel, col, t.data_ptr() if c else 0, b, c, rows))
        self.eng.sync()
        del t

    def upload_host(self, rel, col, arr):
        """a whole numpy column (every rank holds it: the twins)"""
        a = np.ascontiguousarray(arr, dtype=np.uint64)
        self.ck(self.lib.qce_upload_column(rel, col, a.ctypes.data, len(a)))

    def sync_all(self):
        self.eng.sync()
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    def verdict_of_rank0(self, ok):
        """rank 0 holds the whole batch's stdout: its verdict is everybody's"""
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int64, device="cuda")
        self.dist.broadcast(t, 0)
        return bool(int(t[0]))

    def sum_over_ranks(self, vals):
        """uint64 sums mod 2^64 over the ranks"""
        if self.world == 1:
            return [int(v) & M64 for v in vals]
        t = self.torch.tensor([v - (1 << 64) if v >> 63 else v for v in vals], dtype=self.torch.int64, device="cuda")
        self.dist.all_reduce(t)
        return [int(x) & M64 for x in t.tolist()]

    def timed(self, text, steps, warmup, want=None):
        """K timed steps: device time (CUDA events on the engine stream, each step ends with its results
        on the host), max over ranks.  Returns (ms_per_step, launches_per_step, last_output)."""
        out = None
        for _ in range(warmup):
            out = self.run(text)
        self.sync_all()
        arena0 = self.arena()
        self.eng.timer_reset()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = self.run(text)
        ms, launches = self.eng.timer_read()
        wall = 1e3 * (time.perf_counter() - t0)
        arena1 = self.arena()
        # steady state allocates nothing new: the engine's HBM arena (this rank's main context) must not have
        # grown inside the timed region, and every temporary must be back (a leak shows here long before it
        # costs a cudaMalloc in the middle of a run)
        self.last_arena = None
        if arena0 is not None and arena1 is not None:
            self.last_arena = {"reserved_mb": round(arena1[0] / 1e6, 1), "grew_during_timed_steps": arena1[0] != arena0[0],
                               "in_use_mb_after_last_step": round(arena1[1] / 1e6, 1)}
        if want is not None and self.rank == 0:
            assert out == want, (out[:200], want[:200])
        return self.max_over_ranks(ms) / steps, launches // max(steps, 1), out, self.max_over_ranks(wall) / steps


# ------------------------------------------------------------------ twin vs the reference binary
def twin_parity(rig, w, rel_offset, first=None):
    """The scaled twin `w` through the product path (row-sharded over all ranks when N > 1) against the
    unmodified reference binary on the same relation files.  Returns (ok or None, seconds of the reference)."""
    from oracle import workload as wl
    cols = w.referenced() if first is None else None
    db = [[w.column_np(r, c) for c in range(len(w.relations[r][1]))] for r in range(len(w.relations))]
    if rig.world > 1:
        rig.ck(rig.lib.qce_set_replicate_bytes(0))  # force the exchange path: nothing replicated
    try:
        for r, cs in enumerate(db):
            for c, a in enumerate(cs):
                if cols is None or (r, c) in cols:
                    rig.upload_host(rel_offset + r, c, a)
        got = rig.run(w.text(rel_offset, first))
    finally:
        if rig.world > 1:
            rig.ck(rig.lib.qce_set_replicate_bytes(2 << 30))
    ok, ref_s = None, None
    if rig.rank == 0 and wl.have_reference():
        d = tempfile.mkdtemp(prefix="qce_twin_")
        paths = wl.write_db(d, db)
        t = time.time()
        want, err, rc = wl.run_reference(paths, w.text(0, first))
        ref_s = time.time() - t
        for p in paths:
            os.unlink(p)
        ok = bool(rc == 0 and got == want)
        if not ok:
            sys.stderr.write("twin mismatch (%s): reference rc=%d\n got  %r\n want %r\n" % (w.name, rc, got[:300], want[:300]))
    return ok, ref_s


# ------------------------------------------------------------------ configs 3, 4, 5
def run_generated(rig, name, w, twin, check, rel_offset, steps, warmup, twin_first=None, sampler=None):
    """Generic config runner: twin parity, device-generated columns, full-size check, timing."""
    torch = rig.torch
    t0 = time.time()
    twin_ok, ref_s = twin_parity(rig, twin, 100 + rel_offset, twin_first)
    twin_s = time.time() - t0
    t0 = time.time()
    placement = {}
    if rig.world > 1:
        # replicate what fits (smallest relations first, 45 % of HBM), row-shard the rest: the engine's planner
        rows = np.array([w.rows(r) for (r, c) in w.referenced()], dtype=np.uint64)
        cap = C.c_uint64()
        rig.ck(rig.lib.qce_placement_cap(rows.ctypes.data, len(rows), C.byref(cap)))
        rig.ck(rig.lib.qce_set_replicate_bytes(cap.value))
    for (r, c) in w.referenced():
        rows = w.rows(r)
        rig.upload_fn(rel_offset + r, c, rows, lambda b, n, r=r, c=c: w.column_t(torch, r, c, b, n))
        placement[r] = "whole" if rig.whole(rows) else "row-sharded"
    torch.cuda.empty_cache()
    load_s = time.time() - t0
    text = w.text(rel_offset)
    got = rig.run(text)  # cold run = the result every timed step must reproduce
    full_ok = check(got)
    if sampler:
        sampler.start()
    ms, launches, out, wall_ms = rig.timed(text, steps, warmup, want=got)
    rig.last_output = out
    clocks = sampler.stop() if sampler else None
    rows_in = w.join_input_rows()
    res = {
        "workload": "%s: %s" % (name.upper(), w.describe), "ms_per_step": ms, "wall_ms_per_step": wall_ms,
        "value": rows_in / (ms / 1e3), "unit": "rows/s", "join_input_rows_per_step": rows_in,
        "queries_per_step": len(w.queries), "queries_per_s": len(w.queries) / (ms / 1e3),
        "steps": steps, "warmup": warmup, "gpu_launches_per_step_main_stream": int(launches),
        "parity": {"twin_vs_reference": twin_ok, "full_vs_checker": full_ok,
                   "twin": "%s; reference binary %.1f s" % (twin.describe, ref_s or 0.0)},
        "placement": sorted(set(placement.values())), "load_s": round(load_s, 2), "twin_s": round(twin_s, 2),
    }
    if clocks:
        res["clocks"] = clocks
    if getattr(rig, "last_arena", None):
        res["arena"] = rig.last_arena
    if len(w.queries) == 1:
        res["result"] = got.strip()
    return res


def config_c3(rig, rows_per_gpu, steps, warmup, sampler=None):
    from tools import benchkit as bk
    w = bk.c3_workload(rows_per_gpu * rig.world)
    twin = bk.c3_workload(60_000)

    def check(got):
        b, n = rig.share(w.rows(0)) if rig.world > 1 else (0, w.rows(0))
        pairs, sums = bk.c3_check(rig.torch, w, b, n)
        tot = rig.sum_over_ranks([pairs] + sums)
        return rig.verdict_of_rank0(got == bk.format_line(tot[0], tot[1:]))
    res = run_generated(rig, "c3", w, twin, check, 10, steps, warmup, sampler=sampler)
    res["scaling"] = "weak (%d rows per relation per GPU; BASELINE config 3 = 500M rows per relation over 8 GPUs)" % rows_per_gpu
    return res


def config_c4(rig, rows_per_gpu, steps, warmup, sampler=None):
    from tools import benchkit as bk
    w = bk.c4_workload(rows_per_gpu * rig.world)
    twin = bk.c4_workload(100_000)

    def check(got):
        b, n = rig.share(w.rows(0)) if rig.world > 1 else (0, w.rows(0))
        pairs, sums = bk.c4_check(rig.torch, w, b, n)
        tot = rig.sum_over_ranks([pairs] + sums)
        return rig.verdict_of_rank0(got == bk.format_line(tot[0], tot[1:]))
    res = run_generated(rig, "c4", w, twin, check, 20, steps, warmup, sampler=sampler)
    res["scaling"] = "weak (%d rows per relation per GPU)" % rows_per_gpu
    return res


def config_c5(rig, scale, nqueries, steps, warmup, check_queries=48, sampler=None):
    from tools import benchkit as bk
    w = bk.c5_workload(scale=scale, nqueries=nqueries)
    twin = bk.c5_workload(scale=1.0 / 8000, nqueries=nqueries)

    def check(got):
        # a spread of the batch (every len/check_queries-th query, always including those over the largest
        # relations) against the index-map checker.  Every rank evaluates its row share of every picked
        # query (the same collectives on every rank); rank 0, which holds the whole batch's stdout, locates
        # each query's lines by replaying the batch's line structure (filter-only queries print a count line).
        by_size = sorted(range(len(w.queries)), key=lambda k: -sum(w.rows(r) for r in w.plans[k][0]))
        pick = sorted(set(by_size[:check_queries // 4] + list(range(0, len(w.queries), max(1, len(w.queries) // check_queries)))))
        wants = {}
        for k in pick:
            r0 = w.plans[k][0][0]
            per = -(-w.rows(r0) // rig.world)
            b = min(rig.rank * per, w.rows(r0))
            n = min(per, w.rows(r0) - b)
            first, pairs, sums = bk.c5_check_query(rig.torch, w, k, b, n)
            tot = rig.sum_over_ranks([pairs, first or 0] + sums)
            wants[k] = ("%d\n" % tot[1] if first is not None else "") + bk.format_line(tot[0], tot[2:])
        lines = got.splitlines(keepends=True)
        at, where = 0, []
        for k in range(len(w.queries)):
            n = 2 if not w.plans[k][1] else 1
            where.append((at, n))
            at += n
        ok = at == len(lines) and all("".join(lines[where[k][0]:where[k][0] + where[k][1]]) == wants[k] for k in pick)
        return rig.verdict_of_rank0(ok)
    res = run_generated(rig, "c5", w, twin, check, 30, steps, warmup, twin_first=100, sampler=sampler)
    res["scaling"] = "strong (the same batch on every N)"
    res["relation_rows"] = bk.c5_sizes(scale)
    hits, misses = C.c_uint64(), C.c_uint64()
    rig.lib.qce_batch_cache_stats(C.byref(hits), C.byref(misses))
    res["sorted_run_cache"] = {"hits": hits.value, "misses": misses.value}
    return res


# ------------------------------------------------------------------ config 2 (headline)
C2_MODELS = {
    # algorithmic HBM bytes per STEP of every kernel (DESIGN.md section 3): packed 8-byte tuples,
    # 4-byte row ids, 8-byte column values
    "msd_partition": lambda s: (16.0 * s["sort"] * 2, "16 B per tuple per level (8 read + 8 written), two partition levels"),
    "msd_count_sort": lambda s: (16.0 * s["sort"], "16 B per tuple (8 read + 8 written)"),
    "msd_hist": lambda s: (8.0 * s["sort"], "8 B per tuple (level B; level A rides on the build kernel)"),
    "onesweep_k": lambda s: (16.0 * s["sort"] * s["passes"], "16 B per tuple per pass"),
    "checksum": lambda s: (12.0 * s["pairs"] * 3, "4 B row id + 8 B value per row per projected column"),
    "join_bounds": lambda s: (8.0 * s["sort"] + 8.0 * s["lhs"], "8 B per input tuple + 8 B (lb,cnt) per lhs tuple"),
    "join_fused": lambda s: (8.0 * s["sort"] + 8.0 * s["pairs"], "8 B per input tuple (both runs, read once) + 8 B per pair written"),
    "join_write": lambda s: (16.0 * s["lhs"] + 8.0 * (s["sort"] - s["lhs"]) + 8.0 * s["pairs"],
                             "8 B (lb,cnt) + 8 B tuple per lhs tuple, the rhs run's 8 B tuples (row ids of the matches), 8 B per pair written"),
    "build_tuples": lambda s: (8.0 * s["rows"] + 12.0 * s["lhs"] + 8.0 * s["sort"], "8 B key (+4 B id) in, 8 B packed tuple out"),
    "filter_scan": lambda s: (8.0 * s["rows"] + s["rows"] / 8.0, "8 B per row in + 1 bit per row out"),
    "push_tuples": lambda s: (16.0 * s["sort"], "8 B read + 8 B stored (locally or over NVLink) per tuple"),
    "push_rowids": lambda s: (8.0 * s["pairs"] * 2, "4 B read + 4 B stored per row id"),
}
# which kernels form a stage; the dominant STAGE is reported (deterministic: a 3 % wobble between two
# kernels no longer flips the headline kernel)
C2_STAGES = {"sort": ["msd_partition", "msd_count_sort", "msd_hist", "onesweep_k", "radix_hist", "msd_tiles", "msd_max"],
             "projection": ["checksum", "hist_u32", "partition_u32", "join_write", "push_rowids", "hist_ids"],
             "join": ["join_fused", "join_bounds", "join_partition"], "build": ["build_tuples", "filter_scan", "compact_ids"],
             "exchange": ["push_tuples", "radix_hist"]}


def config_c2(rig, rows, steps, warmup, args, local_rank):
    """Config 2; N > 1: weak scaling, every rank owns a `rows`-row window of two relations of N x rows rows
    (row-sharded, nothing replicated)."""
    torch, dist, world, rank = rig.torch, rig.dist, rig.world, rig.rank
    from tools import benchkit as bk
    pk, pk_src = peaks()
    nproc = os.cpu_count() or 1
    q = QUERY.format(thr=500000)

    # ---- (a) the scaled twin (the reference arm's workload) through the product path, vs the reference
    class Twin:
        name, describe = "c2", "2 x %d rows, same generator family (seeds 1/2)" % REF_SAMPLE_ROWS
        relations = [(REF_SAMPLE_ROWS, [None] * 3)] * 2
        queries = [q.strip()]
        _db = [gen_relation(REF_SAMPLE_ROWS, 1, REF_SAMPLE_ROWS), gen_relation(REF_SAMPLE_ROWS, 2, REF_SAMPLE_ROWS)]

        def column_np(self, r, c):
            return self._db[r][c]

        def referenced(self):
            return [(r, c) for r in range(2) for c in range(3)]

        def text(self, off=0, first=None):
            return "%d %d|%s" % (off, off + 1, q.split("|", 1)[1])
    twin = Twin()
    twin_ok, ref_s = twin_parity(rig, twin, 100)
    # the GPU arm on the very workload the reference arm times (vs_reference's same-config leg)
    if world > 1:
        rig.ck(rig.lib.qce_set_replicate_bytes(0))
    twin_ms, _, _, _ = rig.timed(twin.text(100), steps, warmup)
    twin_leg = {"rows_per_relation": REF_SAMPLE_ROWS, "ms_per_step": twin_ms, "value": 2 * REF_SAMPLE_ROWS / (twin_ms / 1e3),
                "unit": "rows/s", "note": "the reference arm's workload (config-2 scaled twin) through the same product path"}

    # ---- (b) full size
    if world > 1:
        rows = rows // 4096 * 4096  # equal, vector-aligned row windows on every rank (qce_row_share)
    n = world * rows
    gen_s = time.time()
    host_cols = {}
    if world == 1:
        for r, seed in enumerate((1, 2)):
            for c, col in enumerate(gen_relation(rows, seed, rows)):
                host_cols[(r, c)] = torch.from_numpy(col.view(np.int64)).pin_memory()
        begin = 0

        def upload_all():
            for (r, c), t in host_cols.items():
                rig.ck(rig.lib.qce_upload_column(r, c, t.data_ptr(), rows))
        upload_all()
        dev_cols = None
    else:
        begin, count = rig.share(n)
        assert (begin, count) == (rank * rows, rows), (begin, count, rows)
        g = torch.Generator(device="cuda")
        dev_cols = {}
        for r, seed in enumerate((1, 2)):
            g.manual_seed(1000 + 64 * seed + rank)
            dev_cols[(r, 0)] = torch.arange(begin, begin + rows, dtype=torch.int64, device="cuda")
            dev_cols[(r, 1)] = torch.randint(0, n, (rows,), dtype=torch.int64, device="cuda", generator=g)
            dev_cols[(r, 2)] = torch.randint(0, 10 ** 6, (rows,), dtype=torch.int64, device="cuda", generator=g)
        torch.cuda.synchronize()
        for (r, c), t in dev_cols.items():
            rig.ck(rig.lib.qce_upload_column_window_device(r, c, t.data_ptr(), begin, rows, n))
        host_cols = {k: v.cpu().pin_memory() for k, v in dev_cols.items()}

        def upload_all():
            for (r, c), t in host_cols.items():
                rig.ck(rig.lib.qce_upload_column_window(r, c, t.data_ptr(), begin, rows, n))
    gen_s = time.time() - gen_s
    col_bytes = rows * 8
    want = rig.run(q)

    # ---- independent full-size check: multiplicities by bincount over the key domain
    if dev_cols is None:
        dc = {k: v.cuda(non_blocking=True) for k, v in host_cols.items()}
    else:
        dc = dev_cols
    lhs, pairs, sums = bk.c2_check(torch, dist if world > 1 else None, dc[(0, 1)], dc[(0, 2)], dc[(0, 0)],
                                   dc[(1, 1)], dc[(1, 0)], dc[(1, 2)], n, 500000)
    full_ok = want == bk.format_line(pairs, sums)
    del dc
    dev_cols = None
    torch.cuda.empty_cache()

    sampler = ClockSampler(local_rank, period=float(os.environ.get("QCE_BENCH_CLOCK_PERIOD", "0.05")))
    # ---- value: columns resident in HBM
    for _ in range(warmup):
        assert rig.run(q) == want
    rig.sync_all()
    sampler.start()
    ms_per_step, launches, out, wall_ms = rig.timed(q, steps, 0, want=want)
    rig.last_output = out
    arena_c2 = getattr(rig, "last_arena", None)
    value = 2 * n / (ms_per_step / 1e3)
    # the same K steps again with CUDA events around every kernel launch (adds ~1.5 % to a step, so it is
    # kept out of `value`): per-kernel times for the roofline
    rig.eng.profile(True)
    rig.eng.timer_reset()
    for _ in range(steps):
        out = rig.run(q)
    ms_prof, _ = rig.eng.timer_read()
    prof_all = rig.eng.profile_read()
    prof = {k: v for k, v in prof_all.items() if not k.startswith("gap_before")}
    rig.eng.profile(False)

    # ---- e2e: host buffers in, checksums out, every step
    for _ in range(warmup):
        upload_all(); rig.run(q)
    rig.sync_all()
    rig.eng.timer_reset()
    for _ in range(steps):
        upload_all()
        out = rig.run(q)
    ms_e2e, _ = rig.eng.timer_read()
    ms_e2e = rig.max_over_ranks(ms_e2e)
    clocks = sampler.stop()
    assert rank != 0 or out == want
    e2e_value = 2 * n / (ms_e2e / steps / 1e3)

    line = {"metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64"}
    if rank != 0:
        return line
    # ---- roofline, per kernel and per stage (rank 0's share of the work)
    key_bits = max(1, int(n - 1).bit_length())
    sizes = {"rows": rows, "lhs": lhs / world, "pairs": pairs / world, "sort": (lhs + n) / world, "passes": (key_bits + 7) // 8}
    kms = {k: v["ms"] / steps for k, v in prof.items()}
    kfrac = {}
    for k, ms_k in kms.items():
        if k in C2_MODELS and ms_k > 0:
            kfrac[k] = round(C2_MODELS[k](sizes)[0] / (ms_k / 1e3) / 1e9 / pk["hbm_gbs"], 3)
    stage_ms = {s: sum(kms.get(k, 0.0) for k in ks) for s, ks in C2_STAGES.items()}
    dom_stage = max(sorted(stage_ms), key=lambda s: stage_ms[s])
    dom = max((k for k in C2_STAGES[dom_stage] if k in C2_MODELS and k in kms), key=lambda k: kms[k])
    alg_launch = C2_MODELS[dom](sizes)[0] / max(1, prof[dom]["launches"] // steps)
    avg_launch_ms = prof[dom]["ms"] / max(1, prof[dom]["launches"])
    achieved = alg_launch / (avg_launch_ms / 1e3) / 1e9
    traffic = None  # DRAM bytes per launch from the committed ncu --set full capture of this kernel
    try:
        tr_db = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        if dom in tr_db:
            traffic = tr_db[dom]["dram_bytes_per_tuple"] / tr_db[dom]["algorithmic_bytes_per_tuple"] * alg_launch
    except Exception:
        pass
    passes = sizes["passes"]
    lhs_r, pairs_r = lhs / world, pairs / world
    # whole-query algorithmic bytes in SURVEY 8d's terms (uint64 SoA, 16-byte tuples), this rank's share
    alg_query = (8 * rows + 8 * lhs_r) + (32 * lhs_r + 24 * rows) + (lhs_r + rows) * (8 + passes * 32) \
        + 16 * (lhs_r + rows) + 16 * pairs_r + 3 * 16 * pairs_r
    total_kernel_ms = sum(kms.values())
    roofline = {"bound": "hbm", "kernel": dom, "stage": dom_stage, "achieved": achieved, "peak": pk["hbm_gbs"], "peak_source": pk_src,
                "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "traffic": traffic,
                "algorithmic_bytes_per_launch": alg_launch, "launches": prof[dom]["launches"],
                "avg_launch_ms": avg_launch_ms, "share_of_kernel_time": kms[dom] / total_kernel_ms if total_kernel_ms else None,
                "algorithmic_bytes": C2_MODELS[dom](sizes)[1],
                "stages_ms_per_step": {k: round(v, 4) for k, v in stage_ms.items()},
                "kernels_ms_per_step": {k: round(v, 4) for k, v in sorted(kms.items(), key=lambda kv: -kv[1])},
                "stream_gaps_ms_per_step": {k[len("gap_before:"):]: round(v["ms"] / steps, 4)
                                            for k, v in sorted(prof_all.items(), key=lambda kv: -kv[1]["ms"])
                                            if k.startswith("gap_before") and v["ms"] / steps >= 0.01},
                "kernels_frac_of_peak": kfrac,
                "whole_query": {"algorithmic_gb_survey_8d": alg_query / 1e9, "lhs_rows": lhs, "pairs": pairs,
                                "frac_of_peak": (alg_query / 1e9) / (ms_per_step / 1e3) / pk["hbm_gbs"]},
                "note": "rank 0's kernels" if world > 1 else None}
    cpu = None
    if not args.no_cpu_baseline:
        try:
            r = time_reference(REF_SAMPLE_ROWS, 2, 0)
            if r:
                cpu = {"value": r["rows_per_s"], "unit": "rows/s", "cores": 1, "kind": "reference",
                       "sample": "oracle/_ref/queries (unmodified reference, gcc -O2) on the C2 scaled twin: 2 x %d rows, "
                                 "mean of 2 runs, process wall minus load-only run; host has %d cores, the reference "
                                 "uses 1" % (REF_SAMPLE_ROWS, nproc)}
                twin_leg["speedup_vs_cpu_reference_same_workload"] = twin_leg["value"] / r["rows_per_s"]
        except Exception as e:  # the baseline is reported, never required
            cpu = {"value": None, "unit": "rows/s", "cores": 1, "kind": "reference", "sample": "failed: %r" % (e,)}
    line.update({
        "data": "synthetic (%s, generated in %.1f s)" % ("numpy default_rng seeds 1/2" if world == 1 else "torch device RNG, one window per rank", gen_s),
        "config": {"workload": "C2: single 2-way equi-join + range filter, 2 x %d-row uint64 relations x 3 columns%s, "
                               "query %s" % (n, "" if world == 1 else " (%d rows per GPU per relation, ROW-SHARDED over %d ranks: "
                                             "histogram all-gather, partition+push kernel over NVLink peer windows, row ids pushed "
                                             "to their owners for the checksums)" % (rows, world), q.strip()),
                   "rows_per_relation": n, "l2": "inputs larger than L2: %.1f GB of columns and >= 1.2 GB of tuples touched per step per GPU" % (6 * col_bytes / 1e9),
                   "result": want.strip(), "queries_per_s": 1e3 / ms_per_step,
                   "boundary": "query text -> libqce_host.so (src/*.c host operator layer) -> libqce_b200.so (C-ABI); no Python between the operators"},
        "parity": {"twin_vs_reference": twin_ok, "full_vs_checker": full_ok,
                   "twin": "%s; reference binary %.1f s" % (twin.describe, ref_s or 0.0),
                   "checker": "torch.bincount closed form over the key domain%s" % (" (all-reduced over the ranks)" if world > 1 else "")},
        "same_workload_as_reference_arm": twin_leg,
        "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": 6 * col_bytes, "d2h_bytes_per_step": 3 * 8 + 5 * 16,
                "ms_per_step": ms_e2e / steps, "note": "per rank: its six column windows from pinned host memory, statistics recomputed"},
        "gpu_launches": int(launches) * steps, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "wall_ms_per_step": wall_ms, "ms_per_step_with_kernel_events": ms_prof / steps, "arena": arena_c2,
    })
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every config (and of the reference arm)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="all", choices=["all", "c2", "c3", "c4", "c5"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="config 2/4: rows per relation per GPU")
    ap.add_argument("--c3-rows", type=int, default=62_500_000, help="config 3: rows per relation per GPU (500M / 8)")
    ap.add_argument("--c5-scale", type=float, default=None, help="config 5: relation sizes = 10^6..10^9 rows x scale")
    ap.add_argument("--c5-queries", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write each config's output of its last timed step to DIR/<config>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    nproc = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return 0
        steps, warm = args.steps, args.warmup
        r = time_reference(REF_SAMPLE_ROWS, steps, warm)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/queries not built"}))
            return 0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"reference_c2_twin": r["stdout"]})
        line = {
            "impl": "reference", "metric": METRIC, "value": r["rows_per_s"], "unit": "rows/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * r["sec_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "C2 scaled twin: 2-way equi-join + range filter, 2 x %d-row uint64 relations, "
                                   "3 checksums (the CPU reference is quadratic in join output, full size is infeasible); "
                                   "the GPU arm reports the same workload under same_workload_as_reference_arm"
                                   % REF_SAMPLE_ROWS, "rows_per_relation": REF_SAMPLE_ROWS},
            "cpu_baseline": {"value": r["rows_per_s"], "unit": "rows/s", "cores": 1, "kind": "reference",
                             "sample": "2 x %d rows, process wall time minus load-only run (%.2f s), host has %d cores, "
                                       "reference is single-threaded" % (REF_SAMPLE_ROWS, r["load_s"], nproc)},
            "e2e": {"value": r["rows_per_s"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rig = Rig(torch, dist, rank, world, local_rank)
    outputs = {}

    def drop():
        rig.sync_all()
        rig.ck(rig.lib.qce_drop_relations())
        torch.cuda.empty_cache()

    if args.config in ("all", "c2"):
        line = config_c2(rig, args.rows, args.steps, args.warmup, args, local_rank)
        outputs["c2"] = rig.last_output
        others = {}
        if args.config == "all":
            drop()
            for name, fn in (("c3", lambda: config_c3(rig, args.c3_rows, args.steps, args.warmup)),
                             ("c4", lambda: config_c4(rig, args.rows, args.steps, args.warmup)),
                             ("c5", lambda: config_c5(rig, args.c5_scale or 1.0, args.c5_queries, args.steps, args.warmup))):
                try:
                    others[name] = fn()
                    outputs[name] = rig.last_output
                    drop()
                except Exception as e:  # a side config never takes the headline down
                    others[name] = {"error": repr(e)[:400]}
                    if world > 1:
                        # the ranks are out of step after a failure: keep the headline, skip the rest, and do
                        # not wait for peers that may be gone
                        rig.lib.qce_comm_abort()
                        line["configs"] = others
                        if rank == 0:
                            if args.dump_outputs:
                                dump_outputs(args.dump_outputs, outputs)
                            print(json.dumps(line), flush=True)
                        os._exit(0 if rank == 0 else 1)
                    drop()
            line["configs"] = others
    else:
        sampler = ClockSampler(local_rank, period=float(os.environ.get("QCE_BENCH_CLOCK_PERIOD", "0.05")))
        if args.config == "c3":
            res = config_c3(rig, args.c3_rows, args.steps, args.warmup, sampler)
        elif args.config == "c4":
            res = config_c4(rig, args.rows, args.steps, args.warmup, sampler)
        else:
            res = config_c5(rig, args.c5_scale or 1.0, args.c5_queries, args.steps, args.warmup, sampler=sampler)
        outputs[args.config] = rig.last_output
        line = {"metric": METRIC if args.config != "c5" else "queries_per_s", "value": res["value"] if args.config != "c5" else res["queries_per_s"],
                "unit": "rows/s" if args.config != "c5" else "queries/s", "n_gpus": world, "steps": res["steps"], "warmup": res["warmup"],
                "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                "scaling": "strong" if args.config == "c5" else "weak", "vs_baseline": None, "dtype": "u64",
                "data": "synthetic (tools/benchkit.py: every column a function of the row index, generated on the device)",
                "config": {"workload": res["workload"]}, "parity": res["parity"], "clocks": res.get("clocks"),
                "gpu_launches": res["gpu_launches_per_step_main_stream"] * res["steps"], "detail": res}
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
