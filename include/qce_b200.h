/*
 * qce_b200.h -- C-ABI of the B200 execution engine (libqce_b200.so).
 *
 * This is the drop-in boundary: plain C, opaque handles, raw pointers and
 * sizes, `int` status (0 ok / -1 error, text via qce_last_error()).  The
 * host-side operator layer (query-compiler-executor_b200/src/filter.c, join.c,
 * utilities.c -- same entry points as the reference's filter.h / join.h /
 * utilities.h) calls nothing else.  Every entry point cites the reference code
 * it replaces as path:line relative to /root/reference.
 *
 * Data model on the device (all resident in HBM, SoA):
 *   base column   uint64_t[n]            one per (relation, column), uploaded once
 *   row-id column uint32_t[m]            a mid_result's `payloads` (the reference
 *                                        keeps a DArray of calloc'ed uint64_t*)
 *   tuple run     packed uint64_t[m]     (key << 32 | rowid) when every key of the
 *                                        source column is < 2^32, otherwise
 *                 uint64_t keys[m] + uint32_t ids[m]
 * Row ids are 32-bit on the device because the reference itself caps a relation
 * below 2^31 tuples (`int start,size`, src/utilities.c:20; int32 histogram,
 * src/histogram.h:5).  At the ABI they are widened to uint64_t.
 *
 * Several ranks (one process per GPU; "ranks of the node" below): a handle is THIS
 * RANK'S SHARE of a distributed object -- base columns are replicated or split by
 * row range, filter outputs follow the row windows, join outputs follow the key
 * ranges of the exchange -- while every count the host layer sees
 * (qce_rowids_count, qce_tuples_count, the survivors of a refine) and every
 * checksum is global and identical on all ranks.  The host layer is the same code
 * on one GPU and on eight.
 *
 * There is no CPU fallback: every compute entry point fails with -1 when no
 * CUDA device is usable.
 */
#ifndef QCE_B200_H
#define QCE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct qce_rowids qce_rowids; /* device row-id column                   */
typedef struct qce_tuples qce_tuples; /* device (key,rowid) run, maybe sorted   */

/* ---- engine lifetime ---------------------------------------------------- */

/* Bind the calling process to CUDA device `device` (one process per GPU; -1: LOCAL_RANK or
 * the rank inside the node, modulo the visible devices) and create the main context.
 * Idempotent; every entry point does it on first use.  No reference counterpart. */
int qce_init(int device);
void qce_shutdown(void);
/* Last error text of the calling thread ("" when none). */
const char *qce_last_error(void);
/* ABI version, bumped on any signature change. */
int qce_abi_version(void);
/* Device-side time (ms) spent in engine kernels since the last reset, measured
 * with CUDA events on the engine stream; used by the bench, not by the host. */
int qce_timer_reset(void);
int qce_timer_read(double *ms, uint64_t *kernel_launches);
/* Block until all queued engine work is done. */
int qce_sync(void);
/* Bytes the engine's HBM arena currently holds (slabs) / has handed out. */
int qce_mempool_stats(uint64_t *reserved_bytes, uint64_t *used_bytes);
/* Per-kernel device times: CUDA events around every launch while enabled.
 * qce_profile_json() returns {"tag": {"launches": n, "ms": total}, ...} for
 * everything recorded since qce_profile_enable(1). */
int qce_profile_enable(int on);
const char *qce_profile_json(void);

/* ---- engine contexts (SURVEY.md 8f-3) ------------------------------------
 * The reference runs one query at a time on one thread (execute_queries,
 * src/utilities.c:289-300).  A context is a stream with its own scratch and HBM
 * arena; the host layer's batch scheduler binds one per worker thread so that
 * independent small queries overlap on the device.  Calls made by a thread that
 * never bound a context use the main one.  A bound context is `solo`: it runs
 * whole queries on this rank alone (never the sharded operators). */
void *qce_ctx_create(void);
int qce_ctx_bind(void *ctx); /* NULL: back to the main context */
void qce_ctx_destroy(void *ctx);
int qce_ctx_solo(int on);    /* the calling thread's context */
/* One batch = one execute_queries call: sorted runs of whole base columns are kept
 * between its queries (the same rel.col is sorted again and again, 8f-3) and dropped
 * at its end. */
int qce_batch_begin(void);
int qce_batch_end(void);
int qce_batch_cache_stats(uint64_t *hits, uint64_t *misses);

/* ---- ranks of the node (SURVEY.md 8e) --------------------------------------
 * One process per GPU, SPMD: every rank runs the same host operator layer over its
 * share of the data.  Small host vectors (histograms, counts, checksums) are agreed
 * through a shared-memory segment; tuples and row ids move GPU to GPU over NVLink,
 * stored by the pushing kernels into the peers' CUDA-IPC-mapped windows.  With more
 * than one rank every operator below works on distributed objects: a handle is this
 * rank's share, counts are global, results are identical on every rank.
 * qce_comm_fork: the calling process becomes rank 0 and forks ranks 1..world-1; must
 * run before the process touches CUDA (the host layer does it in execute_queries when
 * QCE_GPUS=n).  Returns the rank, or -1.  qce_comm_attach: independently started
 * processes (torchrun) meet in /dev/shm/<name>; `token` tells a stale segment apart. */
int qce_comm_fork(uint32_t world);
int qce_comm_attach(const char *name, uint32_t rank, uint32_t world, uint64_t token);
uint32_t qce_comm_rank(void);
uint32_t qce_comm_world(void);
int qce_comm_is_child(void);
int qce_comm_barrier(void);
int qce_comm_allreduce_sum_u64(uint64_t *v, uint32_t n);
int qce_comm_allreduce_max_u64(uint64_t *v, uint32_t n);
/* blobs to rank 0: *out (malloc'ed, rank 0 only; may be NULL) = the ranks' blobs back to back,
 * lens[r] (every rank) = rank r's length */
int qce_comm_gatherv(const void *mine, uint64_t bytes, char **out, uint64_t *lens);
void qce_comm_abort(void);
/* fork mode: a child exits here with `status`; rank 0 waits for the children and returns
 * how many of them failed */
int qce_comm_finish(int status);

/* ---- base relations ------------------------------------------------------
 * Replaces fill_data()/read_relations(), src/utilities.c:105-162: the column
 * is uploaded as-is (SoA uint64), the row id stays implicit (= index); the
 * reference's AoS tuple{key,payload=i} copy is never materialised.
 * Also records max(column) so the sort knows its significant bits. */
int qce_upload_column(uint32_t rel, uint32_t col, const uint64_t *host, uint64_t n);
/* With several ranks the column is placed by size: up to qce_set_replicate_bytes (default
 * 2 GB) every rank holds all rows, larger columns are ROW-SHARDED -- rank r keeps rows
 * [r * rpr, (r+1) * rpr), rpr = ceil(n / world) rounded up to 4096 (qce_row_share) -- and
 * the peers' windows are mapped so that a gather of a foreign row is an NVLink load.
 * Collective: every rank makes the same call. `host` pointers of pageable memory (the
 * mapped relation file) are staged through pinned chunks by a small thread pool. */
int qce_upload_column_device(uint32_t rel, uint32_t col, const void *dev, uint64_t n);
/* The caller holds only rows [row_begin, row_begin + row_count): at least its share. */
int qce_upload_column_window(uint32_t rel, uint32_t col, const uint64_t *host, uint64_t row_begin,
                             uint64_t row_count, uint64_t rows_global);
int qce_upload_column_window_device(uint32_t rel, uint32_t col, const void *dev, uint64_t row_begin,
                                    uint64_t row_count, uint64_t rows_global);
int qce_row_share(uint64_t rows_global, uint32_t rank, uint32_t world, uint64_t *row_begin, uint64_t *row_count);
int qce_set_replicate_bytes(uint64_t bytes);
/* Plan a batch: the largest column size that still fits replicated when the batch's columns (rows of
 * each) are taken smallest first into QCE_REPLICATE_FRACTION (0.45) of the device memory. */
int qce_placement_cap(const uint64_t *col_rows, uint32_t ncols, uint64_t *cap_bytes);
int qce_column_would_be_whole(uint64_t rows);
int qce_column_is_whole(uint32_t rel, uint32_t col); /* 1 whole / 0 row-sharded / -1 unknown */
/* Adopt a device buffer without copying (caller keeps ownership, must outlive use). */
int qce_adopt_column_device(uint32_t rel, uint32_t col, const void *dev, uint64_t n);
int qce_column_info(uint32_t rel, uint32_t col, uint64_t *n, uint64_t *max_value);
/* The histogram of key >> (*key_bits - 8) over a whole column, *key_bits = bit length of its maximum,
 * counted with the statistics the upload takes; bins[256].  *key_bits = 0 (bins untouched) when the
 * column has none: row windows, fewer than 2^20 rows, or a maximum outside [2^8, 2^32). */
int qce_column_histogram(uint32_t rel, uint32_t col, uint32_t *bins, int *key_bits);
int qce_drop_relations(void);

/* ---- filter operator -----------------------------------------------------
 * `op` is the reference's operator character: '=', '>' or '<' (unsigned
 * compare); any other character is an error ("Wrong operator",
 * src/filter.c:28,58). */

/* exec_filter_rel_no_exists, src/filter.c:37-64: all i with col[i] OP c, in
 * ascending i. */
int qce_filter_scan(uint32_t rel, uint32_t col, char op, uint64_t c, qce_rowids **out);
/* Same over the row window [row_begin, row_begin + row_count) only (row ids stay
 * relation-global): one rank's share of the scan when a join is sharded by row
 * range across GPUs (SURVEY 8e).  row_begin must be even. */
int qce_filter_scan_range(uint32_t rel, uint32_t col, char op, uint64_t c, uint64_t row_begin,
                          uint64_t row_count, qce_rowids **out);
/* exec_filter_rel_exists, src/filter.c:3-35: order-preserving subset of an
 * existing row-id column, in place; *survivors = the count the reference
 * prints at src/filter.c:32. */
int qce_filter_refine(qce_rowids *ids, uint32_t rel, uint32_t col, char op, uint64_t c,
                      uint64_t *survivors);

/* ---- join operator primitives ------------------------------------------ */

/* allocate_relation, src/join.c:122-142: (key = col[i], rowid = i), all i. */
int qce_build_tuples_base(uint32_t rel, uint32_t col, qce_tuples **out);
/* Same over a row window (row ids relation-global), for row-range sharding. */
int qce_build_tuples_base_range(uint32_t rel, uint32_t col, uint64_t row_begin, uint64_t row_count,
                                qce_tuples **out);
/* allocate_relation_mid_results, src/join.c:96-120: (key = col[id], rowid = id)
 * for each id of the row-id column, in column order. */
int qce_build_tuples_rowids(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_tuples **out);
/* iterative_sort, src/join.c:5-94 (+ build_histogram/build_psum/
 * build_reordered_array, src/utilities.c:20-70; random_quicksort,
 * src/quicksort.c:54-64): ascending by key.  The order among equal keys is
 * unspecified, as in the reference (its quicksort is rand()-driven): runs below
 * 2^20 tuples are sorted stably, larger ones may take the MSD partition path. */
int qce_sort_tuples(qce_tuples *t);
/* qce_build_tuples_base followed by qce_sort_tuples, in one call: the same run, sorted, with the same
 * unspecified order among equal keys.  A large whole column whose run takes the MSD route is never
 * stored unsorted: the first partition level reads the column and forms the tuples on the fly, which
 * saves one write and one read of the whole run.  Every other run (several ranks, keys of 2^32 or
 * more, a column stored in key order, a small or dense one) is built, then sorted.  Like
 * qce_sort_tuples, it takes a sorted run from the batch's cache and leaves one there. */
int qce_build_sorted_tuples_base(uint32_t rel, uint32_t col, qce_tuples **out);
/* 1 if keys are non-decreasing (the reference never checks; the host layer
 * uses it to refuse JOIN_SORT_* merges over unsorted input, SURVEY 8a-10). */
int qce_tuples_is_sorted(const qce_tuples *t, int *sorted);

/* join_relations, src/join.c:325-392: sort-merge equi-join of two key-sorted
 * runs.  outR/outS = aligned row-id columns of all matching pairs, R-major
 * (for each R tuple in order, each equal-key S tuple in order).
 * distinctR/distinctS (may be NULL) = the R / S side of the distinct
 * (rowid_R,rowid_S) pairs (`non_duplicates`, src/join.c:358-367); their order
 * is (rowid_R,rowid_S)-ascending, the reference's is first-seen -- consumers
 * (join_payloads) sort them first, so only the multiset matters. */
int qce_merge_join(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS,
                   qce_rowids **distinctR, qce_rowids **distinctS);
/* join_relations run over an outer run R that is NOT sorted (S sorted): the
 * result of the reference's serial pointer walk, src/join.c:342-377, which it
 * executes when build_relations wrongly assumes R is in key order
 * (JOIN_SORT_RHS via src/join.c:253-267).  An R tuple yields its full match
 * range iff its key >= every earlier R key, nothing otherwise; output R-major. */
int qce_merge_join_walk(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR,
                        qce_rowids **outS);
/* The non_duplicates of join_relations computed on their own (Hashmap dedup,
 * src/join.c:358-367), so the host layer can skip the pass when no bystander
 * column consumes them. */
int qce_distinct_pairs(const qce_rowids *pairsR, const qce_rowids *pairsS, qce_rowids **distinctR,
                       qce_rowids **distinctS);
/* scan_join, src/join.c:395-423: positional filter keyR[i]==keyS[i] for
 * i < min(nR,nS), keys gathered through the two row-id columns. */
int qce_scan_join(uint32_t relR, uint32_t colR, const qce_rowids *idsR, uint32_t relS,
                  uint32_t colS, const qce_rowids *idsS, qce_rowids **outR, qce_rowids **outS);
/* Same with both sides read from base columns (ids = 0..n-1), the
 * `lhs_index == -1 && rhs_index == -1` SCAN_JOIN of src/join.c:270-284. */
int qce_scan_join_base(uint32_t relR, uint32_t colR, uint32_t relS, uint32_t colS,
                       qce_rowids **outR, qce_rowids **outS);
/* join_payloads, src/join.c:426-484: bystander re-join.  R' = (key=last[i],
 * payload=edit[i]) for i < len(last); S' = driver; both sorted by key; emit
 * edit[i] once per equal driver entry, in R'-sorted order. Fails (-1) when
 * len(edit) < len(last) (the reference reads past the array there). */
int qce_rejoin(const qce_rowids *driver, const qce_rowids *last, const qce_rowids *edit,
               qce_rowids **out);

/* ---- projection ----------------------------------------------------------
 * print_sums, src/utilities.c:215-219: sums[k] = sum over ids of
 * column (rel, cols[k])[id], modulo 2^64.  Up to 8 columns per call share one
 * read of the row-id column. */
int qce_checksum(const qce_rowids *ids, uint32_t rel, const uint32_t *cols, uint32_t ncols,
                 uint64_t *sums);

/* ---- handles -------------------------------------------------------------*/
uint64_t qce_rowids_count(const qce_rowids *ids);       /* over all ranks */
uint64_t qce_rowids_count_local(const qce_rowids *ids); /* this rank's share */
int qce_rowids_from_host(const uint64_t *host, uint64_t n, qce_rowids **out);
int qce_rowids_to_host(const qce_rowids *ids, uint64_t *host);
int qce_rowids_clone(const qce_rowids *ids, qce_rowids **out);
void qce_rowids_free(qce_rowids *ids);

uint64_t qce_tuples_count(const qce_tuples *t);
/* Build a run from host (key,payload) arrays -- test entry point. */
int qce_tuples_from_host(const uint64_t *keys, const uint64_t *rowids, uint64_t n,
                         qce_tuples **out);
int qce_tuples_to_host(const qce_tuples *t, uint64_t *keys, uint64_t *rowids);
void qce_tuples_free(qce_tuples *t);

/* ---- multi-GPU exchange step (SURVEY 8e) --------------------------------
 * Splits a tuple run by key range into `nparts` destination runs:
 * part(key) = number of splitters <= key (splitters ascending, nparts-1 of
 * them, each a multiple of 2^(key_bits-8): a boundary of the 256-bin histogram
 * qce_key_histogram returns).  counts[p] = tuples for rank p.  The packed 8-byte
 * words of part p are contiguous in *sendbuf (device pointer owned by the
 * engine until qce_exchange_release) at element offset sum(counts[0..p)); the
 * order inside a part is unspecified (the receiver sorts it).  The collective itself (all-to-all over NVLink) is done
 * by the caller's communicator (torch.distributed / NCCL) on those pointers. */
int qce_partition_tuples(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters,
                         uint32_t nparts, uint64_t *counts, void **sendbuf);
/* Wrap `n` received packed words (device pointer, copied) as a tuple run.
 * id_bound = exclusive upper bound of the row ids they carry (0 = unknown);
 * [key_lo, key_hi] = the key range this rank received (its splitter interval;
 * key_hi = 0 when unknown) -- it sizes the buckets of the local sort. */
int qce_tuples_from_device_packed(const void *dev_words, uint64_t n, uint32_t key_bits,
                                  uint32_t id_bound, uint64_t key_lo, uint64_t key_hi,
                                  qce_tuples **out);
/* Same without the copy: the run is sorted/joined in the caller's buffer, which
 * must be complete (its stream synchronised), 16-byte aligned and outlive the run. */
int qce_tuples_adopt_device_packed(void *dev_words, uint64_t n, uint32_t key_bits,
                                   uint32_t id_bound, uint64_t key_lo, uint64_t key_hi,
                                   qce_tuples **out);
int qce_exchange_release(void *sendbuf);
/* 256-bin histogram of the top 8 significant key bits of a run (for splitter
 * selection from an all-reduced global histogram).  hist = 256 uint64 on host. */
int qce_key_histogram(const qce_tuples *t, uint32_t key_bits, uint64_t *hist);
/* Wide runs (keys >= 2^32): the same over the key's offset from `base`, bin(key) =
 * (key - base) >> max(width - 8, 0), width 1..64.  Every key must lie in
 * [base, base + 2^width): the exchange takes base = the smallest key of all ranks and
 * width = bitlen(largest - base), so keys clustered at a high offset (64-bit ids,
 * timestamps) still spread over the bins.  Cached on the run like the packed histogram.  An
 * empty run of either kind counts as an empty wide run (also for qce_push_tuples_wide). */
int qce_key_histogram_wide(const qce_tuples *t, uint64_t base, uint32_t width, uint64_t *hist);

/* ---- peer-memory exchange: partition + push over NVLink (SURVEY 8e) --------
 * The multi-GPU half of the reference's radix partitioning (build_histogram /
 * build_psum / build_reordered_array, src/utilities.c:20-70): the scatter pass of
 * the top digit stores every tuple directly into the receive window of the GPU
 * that owns its key range (P2P stores through CUDA-IPC-mapped windows), so the
 * partition pass IS the transfer -- no send buffer, no separate all-to-all.
 * One process per GPU; the caller (any communicator: torch.distributed here)
 * only all-gathers the 64-byte IPC handles once and the 256-bin histograms per
 * exchange, and provides a barrier after the pushing kernels have completed. */
int qce_xwin_create(uint64_t bytes, unsigned char *ipc_handle_out /* 64 bytes, may be NULL */);
int qce_xwin_attach(uint32_t world, uint32_t rank, const unsigned char *handles /* world x 64 bytes */);
/* single process: present the local window as `world` ranks (rank r = bytes from r * window/world) */
int qce_xwin_loopback(uint32_t world);
int qce_xwin_info(uint64_t *bytes, void **local_base);
int qce_xwin_destroy(void);
/* first half of a collective re-creation: unmap the peers' windows (then barrier, then destroy) */
int qce_xwin_unmap_peers(void);
/* Scatter a packed run by key range (same splitter rules as qce_partition_tuples) into
 * the destination windows: the tuples for rank p are stored from 8-byte word offset
 * dst_word_offset[p] of p's window on (order inside unspecified).  Asynchronous on the
 * engine stream.  dst_run_index != NULL: the payload of every tuple is replaced by
 * dst_run_index[p] + its position inside this rank's segment, i.e. its index in the
 * receiver's run when the caller lays the segments out in that order; slots_out != NULL
 * receives, per input tuple, (p << 28 | position inside the segment) for
 * qce_push_u32_by_slot (bystander columns of the same entity, join.c:486-505). */
int qce_push_tuples(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                    const uint64_t *dst_word_offset, const uint32_t *dst_run_index, qce_rowids **slots_out);
/* Same with the run's bystander columns fused into the same kernel (requires dst_run_index):
 * column c of input tuple i is stored at 4-byte element col_u32_offset[c * nparts + p] +
 * (position of the tuple inside this rank's segment) of rank p's window; every column
 * leaves in the same coalesced per-destination runs as the tuples.  ncols <= 6. */
int qce_push_tuples_cols(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                         const uint64_t *dst_word_offset, const uint32_t *dst_run_index, uint32_t ncols,
                         const qce_rowids *const *cols, const uint64_t *col_u32_offset);
/* Scatter a wide run by the key range of key - base (qce_key_histogram_wide's bins; splitters
 * as qce_exchange_plan returns them at that width): the keys for rank p are stored unchanged
 * from 8-byte word dst_word_offset[p] of p's window on, their row ids in the same order from
 * 4-byte element dst_id_offset[p] on.  Asynchronous on the engine stream. */
int qce_push_tuples_wide(const qce_tuples *t, uint64_t base, uint32_t width, const uint64_t *splitters,
                         uint32_t nparts, const uint64_t *dst_word_offset, const uint64_t *dst_id_offset);
/* vals[i] -> 4-byte element dst_u32_offset[p] + position of rank p's window, (p, position) = slots[i] */
int qce_push_u32_by_slot(const qce_rowids *vals, const qce_rowids *slots, uint32_t nparts,
                         const uint64_t *dst_u32_offset);
/* Row ids by owner: owner(id) = min(id / rows_per_rank, nranks-1); inside the owner's rows
 * bins_per_rank equal-width bins (bin_width rows each, the last one open-ended);
 * bin(id) = owner * bins_per_rank + local bin.  hist = nranks * bins_per_rank uint64 on the
 * host.  qce_push_rowids stores the ids of bin b from 4-byte element offset
 * bin_u32_offset[b] of the owner's window on: the owner receives its ids grouped by row
 * region, which is what print_sums' gathers (src/utilities.c:215-219) want. */
int qce_rowids_bin_histogram(const qce_rowids *ids, uint32_t rows_per_rank, uint32_t bin_width,
                             uint32_t bins_per_rank, uint32_t nranks, uint64_t *hist);
int qce_push_rowids(const qce_rowids *ids, uint32_t rows_per_rank, uint32_t bin_width,
                    uint32_t bins_per_rank, uint32_t nranks, const uint64_t *bin_u32_offset);
/* Carried join-key columns of the sharded executor: the low 32 bits of a base column's row
 * window as a 4-byte device column; row ids begin..begin+count-1; a packed run
 * (keys[i] << 32 | i) over such a column (allocate_relation_mid_results, src/join.c:96-120,
 * with the key already at hand). */
int qce_column_window_u32(uint32_t rel, uint32_t col, uint64_t row_begin, uint64_t row_count,
                          qce_rowids **out);
int qce_column_gather_u32(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_rowids **out);
int qce_rowids_iota(uint64_t begin, uint64_t count, uint32_t id_bound, qce_rowids **out);
int qce_tuples_from_u32(const qce_rowids *keys, uint32_t key_bits, qce_tuples **out);
/* Views into this rank's own window (no copy; valid until the window is reused). */
int qce_tuples_from_window(uint64_t word_offset, uint64_t n, uint32_t key_bits, uint32_t id_bound,
                           uint64_t key_lo, uint64_t key_hi, qce_tuples **out);
/* A wide run received by qce_push_tuples_wide: n keys from 8-byte word word_offset, their ids
 * from 4-byte element id_u32_offset (both 16-byte aligned).  Every key lies in [key_lo, key_hi],
 * so the keys agree above bit bitlen(key_lo ^ key_hi) and its sort passes cover only the bits
 * below. */
int qce_tuples_from_window_wide(uint64_t word_offset, uint64_t id_u32_offset, uint64_t n, uint32_t id_bound,
                                uint64_t key_lo, uint64_t key_hi, qce_tuples **out);
/* [id_min, id_bound) = range of the received ids (the owner's row window); bucketed != 0:
 * they arrived grouped by L2-sized row regions, the checksum needs no bucketing pass. */
int qce_rowids_from_window(uint64_t u32_offset, uint64_t n, uint32_t id_min, uint32_t id_bound,
                           int bucketed, qce_rowids **out);
/* Bystander re-join elision (SURVEY 8f-2), used by the host layer's join operator when it can show
 * that the reference's join_payloads (src/join.c:426-484) yields the same multisets:
 * qce_build_tuples_positions: (key = col[ids[i]], payload = i) instead of payload = ids[i];
 * qce_merge_join_stats: qce_merge_join + min / max matches per outer tuple (uniform multiplicity
 * test); qce_rowids_gather re-aligns every column of the entity with the positions the merge
 * returned.  qce_elision_supported: 1 unless QCE_ELIDE=0. */
int qce_build_tuples_positions(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_tuples **out);
/* the row-id columns aligned with the run's positions (<= 6): with several ranks they travel with the
 * tuples when the join exchanges the run, and qce_rowids_gather reads the received copies */
int qce_tuples_attach(qce_tuples *t, uint32_t ncols, const qce_rowids *const *cols);
int qce_merge_join_stats(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS,
                         uint32_t *min_matches, uint32_t *max_matches);
int qce_elision_supported(void);
/* out[i] = src[index[i]] (re-align a bystander row-id column with a join output whose
 * payloads are positions; SURVEY 8f-2, replaces join_payloads src/join.c:426-484 inside PDQ-T). */
int qce_rowids_gather(const qce_rowids *src, const qce_rowids *index, qce_rowids **out);
/* Row-sharded base column: this rank holds rows [row_begin, row_begin + row_count) of a
 * relation of rows_global rows (device buffer of row_count uint64, adopted).  Row ids stay
 * relation-global everywhere; operators may only touch resident rows (checked for windows,
 * by construction for gathers: ids are routed to their owner with qce_push_rowids). */
int qce_adopt_column_window(uint32_t rel, uint32_t col, const void *dev, uint64_t row_begin,
                            uint64_t row_count, uint64_t rows_global, uint64_t max_value_global);
int qce_column_max_device(const void *dev, uint64_t n, uint64_t *max_value);

/* Exchange bookkeeping, identical on every rank (pure host arithmetic, no device needed):
 * from the all-gathered histograms (hists[world][nsides][256]) derive the world-1 splitters,
 * per (side, destination) the tuples the destination receives (recv), the tuples earlier
 * ranks put before this rank's segment (before = dst_run_index), the byte offset of the
 * side's run in the destination's window (run_off) and of each of its ncols[side] columns
 * (col_off[column][dst], columns numbered side-major), the window bytes the largest receiver
 * needs, and the tuples this rank sends off-rank per side.  key_bits 1..64 (above 32: the width
 * of a wide exchange; a wide side lays out its ids as one column, ncols = 1).  The splitter
 * cutting before bin b is b << (key_bits - 8), except that a cut past the last bin at 64 bits
 * (2^64) is returned as UINT64_MAX: it lies past every key. */
int qce_exchange_plan(const uint64_t *hists, uint32_t world, uint32_t rank, uint32_t nsides,
                      const uint32_t *ncols, uint32_t key_bits, uint64_t *splitters, uint64_t *recv,
                      uint64_t *before, uint64_t *run_off, uint64_t *col_off, uint64_t *window_bytes,
                      uint64_t *sent_tuples);
/* The same for qce_push_rowids: hists[world][nbind][bins_per_rank * world] -> per binding the
 * 4-byte element offset of this rank's ids of every bin in the owner's window, and the view
 * (offset, count) of the ids this rank receives. */
int qce_rowid_push_plan(const uint64_t *hists, uint32_t world, uint32_t rank, uint32_t nbind,
                        uint32_t bins_per_rank, uint64_t *bin_u32_offset, uint64_t *view_u32_offset,
                        uint64_t *view_count, uint64_t *window_bytes, uint64_t *sent_ids);

#ifdef __cplusplus
}
#endif
#endif /* QCE_B200_H */
