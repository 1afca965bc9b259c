"""ctypes binding of libqce_b200.so (the C-ABI in include/qce_b200.h).

This is harness plumbing for tests and bench.py: the product is the C library
and the C host layer in src/.  Nothing here computes anything -- every method
is one C-ABI call, and a missing library or a missing GPU raises immediately
(there is no CPU path to fall back to).
"""
from __future__ import annotations

import ctypes as C
import json
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libqce_b200.so")

# every symbol include/qce_b200.h declares (tests check the library exports them all)
SYMBOLS = [
    "qce_init", "qce_shutdown", "qce_last_error", "qce_abi_version", "qce_timer_reset", "qce_timer_read",
    "qce_sync", "qce_mempool_stats", "qce_profile_enable", "qce_profile_json", "qce_upload_column", "qce_upload_column_device",
    "qce_adopt_column_device", "qce_column_info", "qce_drop_relations", "qce_filter_scan", "qce_filter_scan_range",
    "qce_build_tuples_base_range", "qce_filter_refine",
    "qce_build_tuples_base", "qce_build_tuples_rowids", "qce_sort_tuples", "qce_tuples_is_sorted",
    "qce_merge_join", "qce_merge_join_walk", "qce_distinct_pairs", "qce_scan_join", "qce_scan_join_base", "qce_rejoin", "qce_checksum", "qce_rowids_count",
    "qce_rowids_from_host", "qce_rowids_to_host", "qce_rowids_clone", "qce_rowids_free", "qce_tuples_count",
    "qce_tuples_from_host", "qce_tuples_to_host", "qce_tuples_free", "qce_partition_tuples",
    "qce_tuples_from_device_packed", "qce_tuples_adopt_device_packed", "qce_exchange_release", "qce_key_histogram",
    "qce_xwin_create", "qce_xwin_attach", "qce_xwin_loopback", "qce_xwin_info", "qce_xwin_destroy", "qce_push_tuples",
    "qce_push_u32_by_slot", "qce_push_tuples_cols", "qce_rowids_bin_histogram", "qce_push_rowids", "qce_tuples_from_window", "qce_rowids_from_window",
    "qce_rowids_gather", "qce_adopt_column_window", "qce_column_max_device", "qce_column_window_u32", "qce_rowids_iota",
    "qce_tuples_from_u32", "qce_column_gather_u32", "qce_exchange_plan", "qce_rowid_push_plan",
    "qce_ctx_create", "qce_ctx_bind", "qce_ctx_destroy", "qce_ctx_solo", "qce_batch_begin", "qce_batch_end",
    "qce_batch_cache_stats", "qce_comm_fork", "qce_comm_attach", "qce_comm_rank", "qce_comm_world", "qce_comm_is_child",
    "qce_comm_barrier", "qce_comm_allreduce_sum_u64", "qce_comm_allreduce_max_u64", "qce_comm_gatherv", "qce_comm_abort",
    "qce_comm_finish", "qce_upload_column_window", "qce_upload_column_window_device", "qce_row_share",
    "qce_set_replicate_bytes", "qce_column_would_be_whole", "qce_column_is_whole", "qce_rowids_count_local", "qce_xwin_unmap_peers", "qce_build_tuples_positions", "qce_merge_join_stats",
    "qce_elision_supported", "qce_tuples_attach", "qce_placement_cap",
    "qce_key_histogram_wide", "qce_push_tuples_wide", "qce_tuples_from_window_wide",
    "qce_build_sorted_tuples_base", "qce_column_histogram",
]


class EngineError(RuntimeError):
    pass


def load_library(path: str = LIB_PATH) -> C.CDLL:
    if not os.path.exists(path):
        raise EngineError(f"{path} is missing: build it with `make -C {HERE} engine` "
                          "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(path)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    P = C.POINTER
    sig = {
        "qce_init": (i32, [i32]), "qce_shutdown": (None, []), "qce_last_error": (C.c_char_p, []),
        "qce_abi_version": (i32, []), "qce_timer_reset": (i32, []),
        "qce_timer_read": (i32, [P(C.c_double), P(u64)]), "qce_sync": (i32, []),
        "qce_mempool_stats": (i32, [P(u64), P(u64)]), "qce_profile_enable": (i32, [i32]), "qce_profile_json": (C.c_char_p, []),
        "qce_upload_column": (i32, [u32, u32, vp, u64]), "qce_upload_column_device": (i32, [u32, u32, vp, u64]),
        "qce_adopt_column_device": (i32, [u32, u32, vp, u64]),
        "qce_column_info": (i32, [u32, u32, P(u64), P(u64)]), "qce_drop_relations": (i32, []),
        "qce_filter_scan": (i32, [u32, u32, C.c_char, u64, P(vp)]),
        "qce_filter_scan_range": (i32, [u32, u32, C.c_char, u64, u64, u64, P(vp)]),
        "qce_build_tuples_base_range": (i32, [u32, u32, u64, u64, P(vp)]),
        "qce_filter_refine": (i32, [vp, u32, u32, C.c_char, u64, P(u64)]),
        "qce_build_tuples_base": (i32, [u32, u32, P(vp)]), "qce_build_tuples_rowids": (i32, [u32, u32, vp, P(vp)]),
        "qce_sort_tuples": (i32, [vp]), "qce_tuples_is_sorted": (i32, [vp, P(i32)]),
        "qce_build_sorted_tuples_base": (i32, [u32, u32, P(vp)]),
        "qce_column_histogram": (i32, [u32, u32, vp, P(i32)]),
        "qce_merge_join": (i32, [vp, vp, P(vp), P(vp), P(vp), P(vp)]),
        "qce_merge_join_walk": (i32, [vp, vp, P(vp), P(vp)]),
        "qce_distinct_pairs": (i32, [vp, vp, P(vp), P(vp)]),
        "qce_scan_join": (i32, [u32, u32, vp, u32, u32, vp, P(vp), P(vp)]),
        "qce_scan_join_base": (i32, [u32, u32, u32, u32, P(vp), P(vp)]),
        "qce_rejoin": (i32, [vp, vp, vp, P(vp)]), "qce_checksum": (i32, [vp, u32, P(u32), u32, P(u64)]),
        "qce_rowids_count": (u64, [vp]), "qce_rowids_from_host": (i32, [vp, u64, P(vp)]),
        "qce_rowids_to_host": (i32, [vp, vp]), "qce_rowids_clone": (i32, [vp, P(vp)]),
        "qce_rowids_free": (None, [vp]), "qce_tuples_count": (u64, [vp]),
        "qce_tuples_from_host": (i32, [vp, vp, u64, P(vp)]), "qce_tuples_to_host": (i32, [vp, vp, vp]),
        "qce_tuples_free": (None, [vp]), "qce_partition_tuples": (i32, [vp, u32, vp, u32, P(u64), P(vp)]),
        "qce_tuples_from_device_packed": (i32, [vp, u64, u32, u32, u64, u64, P(vp)]),
        "qce_tuples_adopt_device_packed": (i32, [vp, u64, u32, u32, u64, u64, P(vp)]), "qce_exchange_release": (i32, [vp]),
        "qce_key_histogram": (i32, [vp, u32, P(u64)]),
        "qce_xwin_create": (i32, [u64, vp]), "qce_xwin_attach": (i32, [u32, u32, vp]), "qce_xwin_loopback": (i32, [u32]),
        "qce_xwin_info": (i32, [P(u64), P(vp)]), "qce_xwin_destroy": (i32, []),
        "qce_push_tuples": (i32, [vp, u32, vp, u32, vp, vp, P(vp)]),
        "qce_push_u32_by_slot": (i32, [vp, vp, u32, vp]),
        "qce_push_tuples_cols": (i32, [vp, u32, vp, u32, vp, vp, u32, vp, vp]),
        "qce_rowids_bin_histogram": (i32, [vp, u32, u32, u32, u32, vp]),
        "qce_push_rowids": (i32, [vp, u32, u32, u32, u32, vp]),
        "qce_column_window_u32": (i32, [u32, u32, u64, u64, P(vp)]), "qce_rowids_iota": (i32, [u64, u64, u32, P(vp)]),
        "qce_tuples_from_u32": (i32, [vp, u32, P(vp)]), "qce_column_gather_u32": (i32, [u32, u32, vp, P(vp)]),
        "qce_tuples_from_window": (i32, [u64, u64, u32, u32, u64, u64, P(vp)]),
        "qce_rowids_from_window": (i32, [u64, u64, u32, u32, i32, P(vp)]), "qce_rowids_gather": (i32, [vp, vp, P(vp)]),
        "qce_adopt_column_window": (i32, [u32, u32, vp, u64, u64, u64, u64]),
        "qce_column_max_device": (i32, [vp, u64, P(u64)]),
        "qce_exchange_plan": (i32, [vp, u32, u32, u32, vp, u32, vp, vp, vp, vp, vp, P(u64), vp]),
        "qce_rowid_push_plan": (i32, [vp, u32, u32, u32, u32, vp, vp, vp, P(u64), vp]),
        "qce_ctx_create": (vp, []), "qce_ctx_bind": (i32, [vp]), "qce_ctx_destroy": (None, [vp]), "qce_ctx_solo": (i32, [i32]),
        "qce_batch_begin": (i32, []), "qce_batch_end": (i32, []), "qce_batch_cache_stats": (i32, [P(u64), P(u64)]),
        "qce_comm_fork": (i32, [u32]), "qce_comm_attach": (i32, [C.c_char_p, u32, u32, u64]),
        "qce_comm_rank": (u32, []), "qce_comm_world": (u32, []), "qce_comm_is_child": (i32, []), "qce_comm_barrier": (i32, []),
        "qce_comm_allreduce_sum_u64": (i32, [vp, u32]), "qce_comm_allreduce_max_u64": (i32, [vp, u32]),
        "qce_comm_gatherv": (i32, [vp, u64, P(vp), vp]), "qce_comm_abort": (None, []), "qce_comm_finish": (i32, [i32]),
        "qce_upload_column_window": (i32, [u32, u32, vp, u64, u64, u64]),
        "qce_upload_column_window_device": (i32, [u32, u32, vp, u64, u64, u64]),
        "qce_row_share": (i32, [u64, u32, u32, P(u64), P(u64)]), "qce_set_replicate_bytes": (i32, [u64]),
        "qce_column_would_be_whole": (i32, [u64]), "qce_column_is_whole": (i32, [u32, u32]),
        "qce_rowids_count_local": (u64, [vp]), "qce_xwin_unmap_peers": (i32, []),
        "qce_build_tuples_positions": (i32, [u32, u32, vp, P(vp)]),
        "qce_merge_join_stats": (i32, [vp, vp, P(vp), P(vp), P(u32), P(u32)]), "qce_elision_supported": (i32, []), "qce_tuples_attach": (i32, [vp, u32, vp]), "qce_placement_cap": (i32, [vp, u32, P(u64)]),
        "qce_key_histogram_wide": (i32, [vp, u64, u32, P(u64)]),
        "qce_push_tuples_wide": (i32, [vp, u64, u32, vp, u32, vp, vp]),
        "qce_tuples_from_window_wide": (i32, [u64, u64, u64, u32, u64, u64, P(vp)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


def exchange_plan(lib, hists: np.ndarray, world: int, rank: int, ncols: Sequence[int], key_bits: int):
    """qce_exchange_plan (host arithmetic only: works without a device)."""
    h = np.ascontiguousarray(hists, dtype=np.uint64)
    nsides = len(ncols)
    nc = np.ascontiguousarray(ncols, dtype=np.uint32)
    splitters = np.zeros(max(world - 1, 1), dtype=np.uint64)
    recv, before, run_off = (np.zeros((nsides, world), dtype=np.uint64) for _ in range(3))
    col_off = np.zeros((max(int(nc.sum()), 1), world), dtype=np.uint64)
    sent = np.zeros(nsides, dtype=np.uint64)
    need = C.c_uint64()
    if lib.qce_exchange_plan(h.ctypes.data, world, rank, nsides, nc.ctypes.data, key_bits, splitters.ctypes.data,
                             recv.ctypes.data, before.ctypes.data, run_off.ctypes.data, col_off.ctypes.data,
                             C.byref(need), sent.ctypes.data) != 0:
        raise EngineError(lib.qce_last_error().decode())
    return [int(x) for x in splitters[:world - 1]], recv, before, run_off, col_off, need.value, sent


def rowid_push_plan(lib, hists: np.ndarray, world: int, rank: int, nbind: int, bins_per_rank: int):
    """qce_rowid_push_plan (host arithmetic only)."""
    h = np.ascontiguousarray(hists, dtype=np.uint64)
    nb = bins_per_rank * world
    offs = np.zeros((nbind, nb), dtype=np.uint64)
    view_off, view_cnt, sent = (np.zeros(nbind, dtype=np.uint64) for _ in range(3))
    need = C.c_uint64()
    if lib.qce_rowid_push_plan(h.ctypes.data, world, rank, nbind, bins_per_rank, offs.ctypes.data, view_off.ctypes.data,
                               view_cnt.ctypes.data, C.byref(need), sent.ctypes.data) != 0:
        raise EngineError(lib.qce_last_error().decode())
    return offs, view_off, view_cnt, need.value, sent


class Engine:
    """One engine per process / per GPU."""

    def __init__(self, device: int = -1):
        self.lib = load_library()
        self._ck(self.lib.qce_init(device))

    # ---- plumbing
    def _ck(self, rc: int) -> None:
        if rc != 0:
            raise EngineError(self.lib.qce_last_error().decode())

    def sync(self) -> None:
        self._ck(self.lib.qce_sync())

    def timer_reset(self) -> None:
        self._ck(self.lib.qce_timer_reset())

    def timer_read(self) -> Tuple[float, int]:
        ms, n = C.c_double(), C.c_uint64()
        self._ck(self.lib.qce_timer_read(C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def mempool_stats(self) -> Tuple[int, int]:
        r, u = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.qce_mempool_stats(C.byref(r), C.byref(u)))
        return r.value, u.value

    def profile(self, on: bool) -> None:
        self._ck(self.lib.qce_profile_enable(1 if on else 0))

    def profile_read(self) -> dict:
        return json.loads(self.lib.qce_profile_json().decode())

    # ---- relations
    def upload_column(self, rel: int, col: int, values) -> None:
        v = _u64(values)
        self._ck(self.lib.qce_upload_column(rel, col, v.ctypes.data, len(v)))

    def upload_column_device(self, rel: int, col: int, dev_ptr: int, n: int, adopt: bool = False) -> None:
        fn = self.lib.qce_adopt_column_device if adopt else self.lib.qce_upload_column_device
        self._ck(fn(rel, col, dev_ptr, n))

    def upload_db(self, db: Sequence[Sequence[np.ndarray]]) -> None:
        for r, cols in enumerate(db):
            for c, v in enumerate(cols):
                self.upload_column(r, c, v)

    def column_info(self, rel: int, col: int) -> Tuple[int, int]:
        n, mx = C.c_uint64(), C.c_uint64()
        self._ck(self.lib.qce_column_info(rel, col, C.byref(n), C.byref(mx)))
        return n.value, mx.value

    def column_histogram(self, rel: int, col: int) -> Tuple[Optional[np.ndarray], int]:
        """(bins of key >> (key_bits - 8), key_bits) taken at upload, or (None, 0) when the column has none."""
        bins = np.zeros(256, dtype=np.uint32)
        kb = C.c_int()
        self._ck(self.lib.qce_column_histogram(rel, col, bins.ctypes.data, C.byref(kb)))
        return (bins if kb.value else None), kb.value

    def drop_relations(self) -> None:
        self._ck(self.lib.qce_drop_relations())

    # ---- handles
    def rowids_from_host(self, ids) -> int:
        v = _u64(ids)
        h = C.c_void_p()
        self._ck(self.lib.qce_rowids_from_host(v.ctypes.data, len(v), C.byref(h)))
        return h.value

    def rowids_to_host(self, h: int) -> np.ndarray:
        n = self.lib.qce_rowids_count(h)
        out = np.empty(n, dtype=np.uint64)
        self._ck(self.lib.qce_rowids_to_host(h, out.ctypes.data))
        return out

    def rowids_count(self, h: int) -> int:
        return self.lib.qce_rowids_count(h)

    def rowids_free(self, h: Optional[int]) -> None:
        if h:
            self.lib.qce_rowids_free(h)

    def tuples_from_host(self, keys, rowids) -> int:
        k, r = _u64(keys), _u64(rowids)
        h = C.c_void_p()
        self._ck(self.lib.qce_tuples_from_host(k.ctypes.data, r.ctypes.data, len(k), C.byref(h)))
        return h.value

    def tuples_to_host(self, h: int) -> Tuple[np.ndarray, np.ndarray]:
        n = self.lib.qce_tuples_count(h)
        k, r = np.empty(n, dtype=np.uint64), np.empty(n, dtype=np.uint64)
        self._ck(self.lib.qce_tuples_to_host(h, k.ctypes.data, r.ctypes.data))
        return k, r

    def tuples_count(self, h: int) -> int:
        return self.lib.qce_tuples_count(h)

    def tuples_free(self, h: Optional[int]) -> None:
        if h:
            self.lib.qce_tuples_free(h)

    # ---- operators
    def filter_scan(self, rel: int, col: int, op: str, c: int, rows: Optional[Tuple[int, int]] = None) -> int:
        h = C.c_void_p()
        if rows is None:
            self._ck(self.lib.qce_filter_scan(rel, col, op.encode(), c, C.byref(h)))
        else:
            self._ck(self.lib.qce_filter_scan_range(rel, col, op.encode(), c, rows[0], rows[1], C.byref(h)))
        return h.value

    def filter_refine(self, h: int, rel: int, col: int, op: str, c: int) -> int:
        n = C.c_uint64()
        self._ck(self.lib.qce_filter_refine(h, rel, col, op.encode(), c, C.byref(n)))
        return n.value

    def build_tuples(self, rel: int, col: int, rowids: Optional[int] = None,
                     rows: Optional[Tuple[int, int]] = None) -> int:
        h = C.c_void_p()
        if rows is not None:
            self._ck(self.lib.qce_build_tuples_base_range(rel, col, rows[0], rows[1], C.byref(h)))
        elif rowids is None:
            self._ck(self.lib.qce_build_tuples_base(rel, col, C.byref(h)))
        else:
            self._ck(self.lib.qce_build_tuples_rowids(rel, col, rowids, C.byref(h)))
        return h.value

    def sort_tuples(self, h: int) -> None:
        self._ck(self.lib.qce_sort_tuples(h))

    def build_sorted_tuples(self, rel: int, col: int) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_build_sorted_tuples_base(rel, col, C.byref(h)))
        return h.value

    def is_sorted(self, h: int) -> bool:
        s = C.c_int()
        self._ck(self.lib.qce_tuples_is_sorted(h, C.byref(s)))
        return bool(s.value)

    def merge_join(self, R: int, S: int, distinct: bool = False):
        oR, oS, dR, dS = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._ck(self.lib.qce_merge_join(R, S, C.byref(oR), C.byref(oS),
                                         C.byref(dR) if distinct else None, C.byref(dS) if distinct else None))
        return (oR.value, oS.value, dR.value, dS.value) if distinct else (oR.value, oS.value)

    def merge_join_walk(self, R: int, S: int):
        oR, oS = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.qce_merge_join_walk(R, S, C.byref(oR), C.byref(oS)))
        return oR.value, oS.value

    def distinct_pairs(self, pR: int, pS: int):
        dR, dS = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.qce_distinct_pairs(pR, pS, C.byref(dR), C.byref(dS)))
        return dR.value, dS.value

    def scan_join(self, relR, colR, idsR, relS, colS, idsS):
        oR, oS = C.c_void_p(), C.c_void_p()
        if idsR is None and idsS is None:
            self._ck(self.lib.qce_scan_join_base(relR, colR, relS, colS, C.byref(oR), C.byref(oS)))
        else:
            self._ck(self.lib.qce_scan_join(relR, colR, idsR, relS, colS, idsS, C.byref(oR), C.byref(oS)))
        return oR.value, oS.value

    def rejoin(self, driver: int, last: int, edit: int) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_rejoin(driver, last, edit, C.byref(h)))
        return h.value

    def checksum(self, ids: int, rel: int, cols: Sequence[int]) -> List[int]:
        n = len(cols)
        ca = (C.c_uint32 * n)(*cols)
        out = (C.c_uint64 * n)()
        self._ck(self.lib.qce_checksum(ids, rel, ca, n, out))
        return [int(x) for x in out]

    # ---- exchange
    def key_histogram(self, t: int, key_bits: int) -> np.ndarray:
        out = np.zeros(256, dtype=np.uint64)
        self._ck(self.lib.qce_key_histogram(t, key_bits, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def key_histogram_wide(self, t: int, base: int, width: int) -> np.ndarray:
        out = np.zeros(256, dtype=np.uint64)
        self._ck(self.lib.qce_key_histogram_wide(t, base, width, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def partition_tuples(self, t: int, key_bits: int, splitters, nparts: int):
        sp = _u64(splitters if len(splitters) else [0])
        counts = (C.c_uint64 * nparts)()
        buf = C.c_void_p()
        self._ck(self.lib.qce_partition_tuples(t, key_bits, sp.ctypes.data, nparts, counts, C.byref(buf)))
        return [int(x) for x in counts], buf.value

    def tuples_from_device_packed(self, dev_ptr: int, n: int, key_bits: int, id_bound: int = 0,
                                  key_lo: int = 0, key_hi: int = 0, adopt: bool = False) -> int:
        h = C.c_void_p()
        fn = self.lib.qce_tuples_adopt_device_packed if adopt else self.lib.qce_tuples_from_device_packed
        self._ck(fn(dev_ptr, n, key_bits, id_bound, key_lo, key_hi, C.byref(h)))
        return h.value

    def exchange_release(self, buf: Optional[int]) -> None:
        if buf:
            self._ck(self.lib.qce_exchange_release(buf))

    # ---- peer-memory exchange (partition + push over NVLink)
    def xwin_create(self, nbytes: int) -> bytes:
        h = (C.c_ubyte * 64)()
        self._ck(self.lib.qce_xwin_create(nbytes, h))
        return bytes(h)

    def xwin_attach(self, world: int, rank: int, handles: bytes) -> None:
        buf = (C.c_ubyte * (64 * world)).from_buffer_copy(handles)
        self._ck(self.lib.qce_xwin_attach(world, rank, buf))

    def xwin_loopback(self, world: int) -> None:
        self._ck(self.lib.qce_xwin_loopback(world))

    def xwin_info(self) -> Tuple[int, int]:
        n, p = C.c_uint64(), C.c_void_p()
        self._ck(self.lib.qce_xwin_info(C.byref(n), C.byref(p)))
        return n.value, p.value or 0

    def xwin_destroy(self) -> None:
        self._ck(self.lib.qce_xwin_destroy())

    def push_tuples(self, t: int, key_bits: int, splitters, nparts: int, dst_word_offset,
                    dst_run_index=None, want_slots: bool = False) -> Optional[int]:
        sp = _u64(splitters if len(splitters) else [0])
        off = _u64(dst_word_offset)
        ri = np.ascontiguousarray(dst_run_index, dtype=np.uint32) if dst_run_index is not None else None
        slots = C.c_void_p()
        self._ck(self.lib.qce_push_tuples(t, key_bits, sp.ctypes.data, nparts, off.ctypes.data,
                                          ri.ctypes.data if ri is not None else None,
                                          C.byref(slots) if want_slots else None))
        return slots.value if want_slots else None

    def push_tuples_cols(self, t: int, key_bits: int, splitters, nparts: int, dst_word_offset, dst_run_index,
                         cols: Sequence[int], col_u32_offset) -> None:
        sp = _u64(splitters if len(splitters) else [0])
        off = _u64(dst_word_offset)
        ri = np.ascontiguousarray(dst_run_index, dtype=np.uint32)
        ca = (C.c_void_p * max(1, len(cols)))(*cols)
        co = _u64(np.asarray(col_u32_offset).reshape(-1) if len(cols) else [0])
        self._ck(self.lib.qce_push_tuples_cols(t, key_bits, sp.ctypes.data, nparts, off.ctypes.data, ri.ctypes.data,
                                               len(cols), ca, co.ctypes.data))

    def push_tuples_wide(self, t: int, base: int, width: int, splitters, nparts: int, dst_word_offset,
                         dst_id_offset) -> None:
        sp = _u64(splitters if len(splitters) else [0])
        off, ido = _u64(dst_word_offset), _u64(dst_id_offset)
        self._ck(self.lib.qce_push_tuples_wide(t, base, width, sp.ctypes.data, nparts, off.ctypes.data, ido.ctypes.data))

    def push_u32_by_slot(self, vals: int, slots: int, nparts: int, dst_u32_offset) -> None:
        off = _u64(dst_u32_offset)
        self._ck(self.lib.qce_push_u32_by_slot(vals, slots, nparts, off.ctypes.data))

    def rowids_bin_histogram(self, ids: int, rows_per_rank: int, bin_width: int, bins_per_rank: int, nranks: int) -> np.ndarray:
        out = np.zeros(bins_per_rank * nranks, dtype=np.uint64)
        self._ck(self.lib.qce_rowids_bin_histogram(ids, rows_per_rank, bin_width, bins_per_rank, nranks, out.ctypes.data))
        return out

    def push_rowids(self, ids: int, rows_per_rank: int, bin_width: int, bins_per_rank: int, nranks: int,
                    bin_u32_offset) -> None:
        off = _u64(bin_u32_offset)
        self._ck(self.lib.qce_push_rowids(ids, rows_per_rank, bin_width, bins_per_rank, nranks, off.ctypes.data))

    def column_window_u32(self, rel: int, col: int, begin: int, count: int) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_column_window_u32(rel, col, begin, count, C.byref(h)))
        return h.value

    def column_gather_u32(self, rel: int, col: int, ids: int) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_column_gather_u32(rel, col, ids, C.byref(h)))
        return h.value

    def rowids_iota(self, begin: int, count: int, id_bound: int = 0) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_rowids_iota(begin, count, id_bound, C.byref(h)))
        return h.value

    def tuples_from_u32(self, keys: int, key_bits: int) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_tuples_from_u32(keys, key_bits, C.byref(h)))
        return h.value

    def tuples_from_window(self, word_offset: int, n: int, key_bits: int, id_bound: int = 0,
                           key_lo: int = 0, key_hi: int = 0) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_tuples_from_window(word_offset, n, key_bits, id_bound, key_lo, key_hi, C.byref(h)))
        return h.value

    def tuples_from_window_wide(self, word_offset: int, id_u32_offset: int, n: int, id_bound: int = 0,
                                key_lo: int = 0, key_hi: int = 0) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_tuples_from_window_wide(word_offset, id_u32_offset, n, id_bound, key_lo, key_hi, C.byref(h)))
        return h.value

    def rowids_from_window(self, u32_offset: int, n: int, id_bound: int = 0, bucketed: bool = False, id_min: int = 0) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_rowids_from_window(u32_offset, n, id_min, id_bound, 1 if bucketed else 0, C.byref(h)))
        return h.value

    def rowids_gather(self, src: int, index: int) -> int:
        h = C.c_void_p()
        self._ck(self.lib.qce_rowids_gather(src, index, C.byref(h)))
        return h.value

    def adopt_column_window(self, rel: int, col: int, dev_ptr: int, row_begin: int, row_count: int,
                            rows_global: int, max_value_global: int) -> None:
        self._ck(self.lib.qce_adopt_column_window(rel, col, dev_ptr, row_begin, row_count, rows_global, max_value_global))

    def column_max_device(self, dev_ptr: int, n: int) -> int:
        m = C.c_uint64()
        self._ck(self.lib.qce_column_max_device(dev_ptr, n, C.byref(m)))
        return m.value
