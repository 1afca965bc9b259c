// qce_engine.cu -- libqce_b200.so: the C-ABI of include/qce_b200.h on top of
// the sm_100a kernels in k_filter.cuh / k_radix.cuh / k_join.cuh.
//
// One process drives one GPU.  All work is queued on one engine stream;
// temporaries come from the engine's own HBM arena (no cudaMalloc / cudaFree on
// the hot path once the slabs exist); the only host synchronisations are the result
// sizes the host-side operator layer needs to size the next step (filter
// count, join pair count) and the final checksums.
//
// There is deliberately no CPU path: if the CUDA runtime reports no usable
// device every entry point returns -1 and qce_last_error() says why.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <map>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "../../include/qce_b200.h"
#include "k_filter.cuh"
#include "k_join.cuh"
#include <memory>
#include "k_radix.cuh"
#include "k_exchange.cuh"
#include "qce_comm.cuh"
#include "qce_arena.hpp"

#define QCE_ABI_VERSION 3

// ------------------------------------------------------------------ handles
// How the elements of a column / run are spread over the ranks of the node (SURVEY.md 8e).
// The global order is always "rank 0's elements, then rank 1's, ...": a filter output
// (ascending row ids, each rank its own row window) and a join output (key order, each rank
// its key range) both keep the order the reference's serial loops produce.
struct Dist {
    enum Kind : int { LOCAL = 0, ROWS, KEYS, ANY };
    int kind = LOCAL;        // LOCAL: one rank holds everything (world 1 / a solo context)
    u32 rel = 0, col = 0;    // ROWS: ids are rows of this rank's window of `rel`; KEYS: sorted by (rel, col)
    int key_bits = 0;        // KEYS: the exchange's key width (splitters sit on its 256-bin boundaries)
    std::vector<uint64_t> split;  // KEYS: world-1 ascending splitters, rank r holds keys in [split[r-1], split[r])
    bool wide = false;       // KEYS of a wide exchange: the splitters and key_bits are those of key - base
    u64 base = 0;            // (a splitter of ~0 lies past every key: the cut 2^64 at width 64)
    bool from_split = false; // output of a join whose exchange cut inside a key: one key's pairs on several ranks
};
struct qce_rowids {
    u32 *d;        // device row ids (this rank's share)
    u64 n;
    u32 id_bound;  // exclusive upper bound of the ids (rows of the source relation), 0 = unknown
    bool bucketed = false; // already grouped by row region (received through qce_push_rowids)
    u32 id_min = 0;        // inclusive lower bound of the ids (a row-sharded owner sees only its window)
    u64 n_others = 0;      // elements held by the other ranks (0 on one GPU): count = n + n_others
    Dist dist;
    u64 attach_gen = 0;    // positions into the columns that travelled with the exchange of that generation
};
struct qce_tuples {
    u64 *a;        // packed words (key << 32 | rowid), or keys when wide
    u32 *ids;      // wide only
    u64 n;
    bool wide;
    int key_bits;  // significant bits of the largest possible key
    u64 key_min;   // smallest / largest possible key (column statistics, or the rank's key
    u64 key_max;   // range after an exchange); they size the MSD buckets
    u32 id_bound;
    bool sorted;
    bool in_order = false;  // built from a whole base column that is stored in ascending order (Column::in_order)
    bool skewed = false;    // the sort met a heavy key (a sub-bucket over the finish tile): joins take the two-phase route
    u32 *hist256 = nullptr; // device: 256-bin histogram of the top 8 of hist_key_bits key bits (taken by the build
    int hist_key_bits = 0;  // kernels, or by qce_key_histogram); valid while the run is unsorted and unmodified
    u64 hist_base = 0;      // wide runs (qce_key_histogram_wide): the bins are those of key - hist_base
    std::vector<unsigned int> hist_host; // the same 256 counts on the host
    bool range_sort = false; // wide run received from an exchange: its keys lie in [key_min, key_max], so
                             // they agree above bit bitlen(key_min ^ key_max) and only the bits below are sorted
    u64 n_others = 0;         // tuples held by the other ranks
    Dist dist;
    bool sort_pending = false; // sharded: qce_sort_tuples is deferred to the join, which first moves
                               // every tuple to the rank that owns its key range
    bool borrowed = false;     // `a` belongs to the batch's sorted-run cache
    u32 src_rel = 0, src_col = 0; // the base column a whole-column run was built from
    bool whole_base = false;
    // elided re-joins (SURVEY.md 8f-2): the payloads are positions, and these row-id columns are
    // aligned with them -- when the run is exchanged between ranks they travel with the tuples
    bool positions = false;
    std::vector<const qce_rowids *> attached;
};

namespace {

struct Column {
    const u64 *d = nullptr; // row-sharded column: VIRTUAL base (window pointer - win_begin), rows outside the
    u64 n = 0;              // window are not resident; n stays the relation's global row count
    u64 maxv = 0;
    bool in_order = false;  // the whole column is resident and stored in ascending order (seen when it was loaded)
    bool owned = false;
    bool windowed = false;
    u64 win_begin = 0, win_count = 0;
    // sharded over the ranks of the node: every rank's window mapped through CUDA IPC
    bool peer_mapped = false;
    u32 rpr = 0, last_rank = 0;        // rows per rank; world - 1
    const u64 *vb[QCE_MAX_RANKS] = {}; // virtual bases: row id r of rank q's window lives at vb[q][r]
    void *alloc = nullptr;             // the cudaMalloc behind d (reused by a re-upload of the same shape)
    u64 alloc_bytes = 0;
    std::vector<void *> opened;        // the peers' mappings (cudaIpcCloseMemHandle on drop)
    // whole columns of 2^20 rows or more with 9 <= hist_bits = bitlen(maxv) <= 32: the 256-bin histogram of
    // key >> (hist_bits - 8), MSD level A of a run built from the column (taken with the load-time statistics)
    u32 *hist = nullptr;               // device, cudaMalloc'ed; kept for a re-upload, freed on drop
    int hist_bits = 0;                 // 0: hist holds nothing
};
ColRef ref_of(const Column *c)
{
    ColRef r;
    memset(&r, 0, sizeof r);
    r.d = c->d;
    if (c->peer_mapped) {
        r.rpr = c->rpr;
        r.last = c->last_rank;
        r.inv = 1.0f / (float)c->rpr;
        // rounded down: the owner estimate may only err low (corrected upwards in ColRef::owner)
        r.inv = nextafterf(r.inv, 0.0f);
        for (int q = 0; q < QCE_MAX_RANKS; q++) r.vb[q] = c->vb[q];
    }
    return r;
}

struct ProfRec {
    const char *tag;
    cudaEvent_t e0, e1;
};

// Per host thread that drives the engine: its own stream, scalar scratch, timers and HBM arena.
// The main context serves the classic one-thread host loop; the batch scheduler
// (src/utilities.c: execute_queries) creates more with qce_ctx_create and binds one per worker
// thread, so independent small queries overlap on the device (SURVEY.md 8f-3).
class Arena;
struct Ctx;
struct Global {
    bool inited = false;
    int device = -1;
    int sms = 148;
    std::map<u64, Column> cols;  // read-mostly: written by uploads (main thread, before a batch runs)
    // peer-memory exchange: this rank's receive window + the peers' windows mapped through CUDA IPC
    unsigned char *xwin = nullptr;
    u64 xwin_bytes = 0;
    u32 xworld = 0, xrank = 0;
    PeerWindows peers;
    std::vector<void *> xopened;
    u32 world = 1, rank = 0;     // ranks of the node (qce_comm.cuh); 1 / 0 on a single GPU
    u64 replicate_bytes = 2ull << 30; // columns up to this size are held whole by every rank
    bool replicate_forced = false;    // QCE_REPLICATE_BYTES was given: the batch planner leaves it alone
    std::mutex mu;               // guards cols / run cache when worker contexts are live
    // sorted base runs of the running batch, keyed by (relation, column): the same column is
    // sorted again and again across the ~1000 queries of a batch (SURVEY.md 8f-3)
    struct CachedRun {
        u64 *a; u64 n; int key_bits; u64 key_min, key_max; u32 id_bound;
        cudaEvent_t ready;      // recorded on the producer's stream after the sort
        class Arena *owner;
        bool skewed = false;
    };
    std::map<u64, CachedRun> run_cache;
    bool cache_on = false;
    u64 cache_bytes = 0, cache_budget = 0, cache_hits = 0, cache_misses = 0;
    std::vector<Ctx *> workers;
};
Global G;
thread_local char g_err[512] = "";

int fail(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return -1;
}

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            (void)cudaGetLastError(); /* a non-sticky failure must not poison the next launch check */ \
            return fail("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
        }                                                                                     \
    } while (0)
#define NEED_INIT()                                                                 \
    do {                                                                            \
        if (!G.inited && qce_init(-1) != 0) return -1;                              \
    } while (0)

inline int bitlen(u64 v)
{
    int b = 0;
    while (v) { b++; v >>= 1; }
    return b;
}
inline u64 ceil_div(u64 a, u64 b) { return (a + b - 1) / b; }
// Exchange splitters sit on the boundaries of the 256-bin histogram of the top 8 of key_bits bits
// (shift = key_bits - 8): the cut before bin b is the key b << shift.  At 64 bits the cut past the
// last bin would be 2^64, which wraps to 0; it is stored as ~0 instead, a value no other cut takes
// (they are multiples of 2^56) and that is read back as bin 256 -- past every key.
inline u64 cut_key(u32 bin, int shift) { return (bin >= 256 && shift >= 56) ? ~0ull : (u64)bin << shift; }
inline u32 cut_bin(u64 split, int shift) { return split == ~0ull ? 256u : (u32)std::min<u64>(256, split >> shift); }
inline bool on_bin_boundary(u64 split, int shift) { return split == ~0ull || (split & ((1ull << shift) - 1)) == 0; }
inline u64 col_key(u32 rel, u32 col) { return ((u64)rel << 32) | col; }
void row_share(u64 n, u32 rank, u32 world, u64 *begin, u64 *count, u64 *per_out = nullptr)
{
    u64 per = ceil_div(n ? n : 1, world);
    per = ceil_div(per, 4096) * 4096;
    const u64 b = std::min<u64>((u64)rank * per, n);
    *begin = b;
    *count = std::min<u64>(per, n - b);
    if (per_out) *per_out = per;
}

// ---- HBM arena (qce_arena.hpp) ------------------------------------------------------------
// Large slabs from cudaMalloc, a best-fit free list with coalescing on the host: no cudaMalloc / cudaFree on
// the hot path once the slabs exist.
static void *arena_slab_alloc(u64 bytes)
{
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return p;
}
static void arena_slab_free(void *p) { cudaFree(p); }
static void arena_grow_hook(const QceArena *self, u64 grew_by, u64 need, bool failed)
{
    if (failed)
        fail("out of device memory: %llu bytes requested, %llu reserved", (unsigned long long)need,
             (unsigned long long)self->reserved());
    else if (getenv("QCE_TRACE"))
        fprintf(stderr, "[qce] arena %p grows by %.1f MB (need %.1f MB, reserved %.1f MB)\n", (const void *)self, grew_by / 1e6,
                need / 1e6, self->reserved() / 1e6);
}
class Arena : public QceArena {
  public:
    Arena() : QceArena(arena_slab_alloc, arena_slab_free, arena_grow_hook) {}
};

struct Ctx {
    cudaStream_t stream = nullptr;
    u64 *d_scalars = nullptr; // 16 u64 of device scratch for totals
    u64 *h_scalars = nullptr; // pinned mirror
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    u64 launches = 0;
    bool profile = false;
    std::vector<ProfRec> prof;
    std::vector<cudaEvent_t> ev_pool; // recycled profiling events
    std::string prof_json;
    Arena arena;
    bool solo = false; // a worker context: whole queries on this rank alone, never the sharded path
    // columns that travelled with the last exchange: caller's handle -> view of the received copy
    u64 attach_gen = 0;
    std::vector<std::pair<const qce_rowids *, qce_rowids *>> recv_cols;
    // exchange overlap: the first received run is sorted on `aux` while the second side's push is
    // still crossing NVLink on `stream`; scratch the in-flight push reads is freed after it
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_side[2] = {nullptr, nullptr}, ev_aux = nullptr;
    bool defer_frees = false;
    std::vector<void *> deferred;
};
Ctx g_main;
thread_local Ctx *tl_ctx = nullptr;
inline Ctx &cx() { return tl_ctx ? *tl_ctx : g_main; }

template <typename T> int dalloc(T **p, u64 count)
{
    *p = nullptr;
    return cx().arena.alloc((void **)p, (count ? count : 1) * sizeof(T));
}
template <typename T> void dfree(T *p) { cx().arena.free((void *)p); }
// scratch of a kernel that may still be in flight while another stream of this context allocates
template <typename T> void dfree_after_push(T *p)
{
    if (cx().defer_frees) cx().deferred.push_back((void *)p);
    else cx().arena.free((void *)p);
}
inline void release_deferred()
{
    for (void *p : cx().deferred) cx().arena.free(p);
    cx().deferred.clear();
}
// Scratch buffers of one operator: whatever path the function leaves by (every `return -1` of a
// failed allocation or launch included) they go back to the arena -- an out-of-memory error used
// to leave the arena permanently smaller.  Buffers that outlive the call are allocated with dalloc.
struct Scratch {
    std::vector<void *> owned;
    ~Scratch() { for (void *p : owned) cx().arena.free(p); }
    template <typename T> int get(T **p, u64 count)
    {
        if (dalloc(p, count) != 0) return -1;
        owned.push_back((void *)*p);
        return 0;
    }
};

void prof_begin(const char *tag)
{
    if (!cx().profile) return;
    ProfRec r;
    r.tag = tag;
    cudaEvent_t *ev[2] = {&r.e0, &r.e1};
    for (auto e : ev) {
        if (!cx().ev_pool.empty()) { *e = cx().ev_pool.back(); cx().ev_pool.pop_back(); }
        else cudaEventCreate(e);
    }
    cudaEventRecord(r.e0, cx().stream);
    cx().prof.push_back(r);
}
void prof_end()
{
    if (!cx().profile) return;
    cudaEventRecord(cx().prof.back().e1, cx().stream);
}

#define LAUNCH(tag, kern, grid, block, smem, ...)                         \
    do {                                                                  \
        prof_begin(tag);                                                  \
        (kern)<<<(grid), (block), (smem), cx().stream>>>(__VA_ARGS__);       \
        prof_end();                                                       \
        cx().launches++;                                                     \
        CK(cudaGetLastError());                                           \
    } while (0)

// read `k` device scalars (d_scalars[0..k)) back; the one sync point of an op
int read_scalars(int k)
{
    CK(cudaMemcpyAsync(cx().h_scalars, cx().d_scalars, k * sizeof(u64), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    return 0;
}

// Row-sharded columns hold only [win_begin, win_begin + win_count) of the relation.
bool window_resident(const struct Column *cl, u64 begin, u64 count);
int get_column(u32 rel, u32 col, const Column **out)
{
    std::lock_guard<std::mutex> lk(G.mu); // map nodes are stable: the pointer outlives the lock
    auto it = G.cols.find(col_key(rel, col));
    if (it == G.cols.end()) return fail("relation %u column %u was never uploaded", rel, col);
    *out = &it->second;
    return 0;
}

bool window_resident(const Column *cl, u64 begin, u64 count)
{
    if (!cl->windowed || count == 0) return true;
    return begin >= cl->win_begin && begin + count <= cl->win_begin + cl->win_count;
}

int op_code(char op, int *code)
{
    switch (op) {
    case '=': *code = QCE_OP_EQ; return 0;
    case '>': *code = QCE_OP_GT; return 0;
    case '<': *code = QCE_OP_LT; return 0;
    }
    return fail("Wrong operator '%c'", op);
}

int new_rowids(u64 n, u32 id_bound, qce_rowids **out)
{
    qce_rowids *r = new qce_rowids();
    r->n = n;
    r->id_bound = id_bound;
    if (dalloc(&r->d, n) != 0) { delete r; return -1; }
    *out = r;
    return 0;
}

int grid_for(u64 items_per_block, u64 n, int waves = 8)
{
    u64 blocks = ceil_div(n ? n : 1, items_per_block);
    u64 cap = (u64)G.sms * waves;
    return (int)(blocks < cap ? blocks : cap);
}

// mask + per-tile counts -> compacted outputs (pass 2 of every filter-like op)
int compact_from_mask(int layout, int mode, const u32 *mask, const u32 *tile_count, u64 ntiles,
                      const void *src0, const u32 *src1, u32 id_bound0, u32 id_bound1,
                      qce_rowids **out0, qce_rowids **out1, u32 id_base = 0)
{
    Scratch sc;
    u32 *tile_off = nullptr;
    if (sc.get(&tile_off, ntiles) != 0) return -1;
    if (ntiles <= 512)
        LAUNCH("scan_tiles", (k_scan_excl_warp<u32, u32>), 1, 32, 0, tile_count, tile_off, ntiles, cx().d_scalars);
    else
        LAUNCH("scan_tiles", (k_scan_excl<u32, u32>), 1, 1024, 0, tile_count, tile_off, ntiles, cx().d_scalars);
    if (read_scalars(1) != 0) return -1;
    const u64 m = cx().h_scalars[0];
    if (new_rowids(m, id_bound0, out0) != 0) return -1;
    if (out1 && new_rowids(m, id_bound1, out1) != 0) return -1;
    u32 *o0 = (*out0)->d, *o1 = out1 ? (*out1)->d : nullptr;
    if (m > 0) {
        const int grid = (int)ntiles;
        if (layout == QCE_LAYOUT_PAIR && mode == QCE_EMIT_INDEX)
            LAUNCH("compact_ids", (k_compact<QCE_LAYOUT_PAIR, QCE_EMIT_INDEX>), grid, QCE_FTHREADS, 0,
                   mask, tile_off, tile_count, src0, src1, o0, o1, id_base);
        else if (layout == QCE_LAYOUT_NATURAL && mode == QCE_EMIT_SRC)
            LAUNCH("compact_src", (k_compact<QCE_LAYOUT_NATURAL, QCE_EMIT_SRC>), grid, QCE_FTHREADS, 0,
                   mask, tile_off, tile_count, src0, src1, o0, o1, id_base);
        else if (layout == QCE_LAYOUT_NATURAL && mode == QCE_EMIT_SRC2)
            LAUNCH("compact_src2", (k_compact<QCE_LAYOUT_NATURAL, QCE_EMIT_SRC2>), grid, QCE_FTHREADS, 0,
                   mask, tile_off, tile_count, src0, src1, o0, o1, id_base);
        else if (layout == QCE_LAYOUT_NATURAL && mode == QCE_EMIT_PACKED)
            LAUNCH("compact_packed", (k_compact<QCE_LAYOUT_NATURAL, QCE_EMIT_PACKED>), grid, QCE_FTHREADS, 0,
                   mask, tile_off, tile_count, src0, src1, o0, o1, id_base);
        else
            return fail("internal: unsupported compaction layout/mode %d/%d", layout, mode);
    }
    return 0;
}

// ---- radix sort driver -------------------------------------------------------
// One digit pass of the LSD sort (k_onesweep).
// BIG: the status-word decode for runs of 2^30 tuples or more (k_radix.cuh).
template <bool HAS_VALS, bool BIG, typename DigitOp>
int launch_onesweep(const u64 *kin, u64 *kout, const u32 *vin, u32 *vout, u32 n, DigitOp dop, const u32 *gbase,
                    u32 *status, u32 *counter)
{
    auto kern = k_onesweep<HAS_VALS, DigitOp, BIG>;
    const size_t smem = sizeof(OnesweepSmem) + (HAS_VALS ? QCE_OS_TILE * sizeof(u32) : 0);
    static bool attr_set = false; // per instantiation
    if (!attr_set) {
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    const u32 ntiles = (u32)ceil_div(n, QCE_OS_TILE);
    LAUNCH(HAS_VALS ? "onesweep_kv" : "onesweep_k", kern, ntiles, QCE_OS_THREADS, smem, kin, kout, vin, vout, n, dop, gbase,
           status, counter);
    return 0;
}

constexpr int BS_THREADS = 512, BS_ITEMS = 8, BS_TILE = BS_THREADS * BS_ITEMS; // block sort: runs <= 4096 tuples

// Sort words (and optional 32-bit values) by the digits listed in rs, least
// significant first.  *keys / *vals are replaced by the sorted buffers.
int radix_sort(u64 **keys, u32 **vals, u64 n, const RadixShifts &rs)
{
    if (n <= 1 || rs.npass == 0) return 0;
    // the reference's runs are indexed by int (src/utilities.c:20), and the one-sweep status word holds prefixes below 2^31
    if (n >= (1ull << 31))
        return fail("sort of %llu tuples exceeds the per-run limit of 2^31 - 1 tuples", (unsigned long long)n);
    if (n <= BS_TILE) {
        // small run: the whole sort in one CTA (k_block_sort), in place
        const size_t smem = BS_TILE * sizeof(u64) + (vals ? BS_TILE * sizeof(u32) : 0) +
                            ((BS_THREADS / 32) * 256 + 256 + 33) * sizeof(u32);
        static bool attr_k = false, attr_kv = false;
        if (vals) {
            if (!attr_kv) {
                CK(cudaFuncSetAttribute(k_block_sort<BS_THREADS, BS_ITEMS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                attr_kv = true;
            }
            LAUNCH("block_sort", (k_block_sort<BS_THREADS, BS_ITEMS, true>), 1, BS_THREADS, smem, *keys, *vals, (u32)n, rs);
        } else {
            if (!attr_k) {
                CK(cudaFuncSetAttribute(k_block_sort<BS_THREADS, BS_ITEMS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                attr_k = true;
            }
            LAUNCH("block_sort", (k_block_sort<BS_THREADS, BS_ITEMS, false>), 1, BS_THREADS, smem, *keys, (u32 *)nullptr, (u32)n, rs);
        }
        return 0;
    }
    const u32 bins = QCE_RADIX_BINS;
    const u32 ntiles = (u32)ceil_div(n, QCE_OS_TILE);
    u64 *alt_k = nullptr;
    u32 *alt_v = nullptr, *ghist = nullptr, *gbase = nullptr, *status = nullptr, *counters = nullptr;
    Scratch sc; // the ping-pong buffers change hands with *keys / *vals and are released by hand
    if (sc.get(&ghist, (u64)rs.npass * bins) != 0 || sc.get(&gbase, (u64)rs.npass * bins) != 0 ||
        sc.get(&status, (u64)rs.npass * ntiles * bins) != 0 || sc.get(&counters, (u64)rs.npass) != 0)
        return -1;
    if (dalloc(&alt_k, n) != 0) return -1;
    if (vals && dalloc(&alt_v, n) != 0) { dfree(alt_k); return -1; }
    CK(cudaMemsetAsync(ghist, 0, (u64)rs.npass * bins * sizeof(u32), cx().stream));
    CK(cudaMemsetAsync(status, 0, (u64)rs.npass * ntiles * bins * sizeof(u32), cx().stream));
    CK(cudaMemsetAsync(counters, 0, (u64)rs.npass * sizeof(u32), cx().stream));
    LAUNCH("radix_hist", k_radix_hist, grid_for(1024, n, 4), 512, 0, *keys, n, rs, bins, ghist);
    LAUNCH("radix_bases", k_radix_bases, rs.npass, bins, 0, ghist, gbase);

    u64 *kin = *keys, *kout = alt_k;
    u32 *vin = vals ? *vals : nullptr, *vout = alt_v;
    for (int p = 0; p < rs.npass; p++) {
        DigitShift dop{rs.shift[p]};
        DigitShiftHi dhi{rs.shift[p] - 32};
        u32 *gb = gbase + p * bins, *st = status + (u64)p * ntiles * bins;
        const u32 m = (u32)n;
        int rc;
        if (n >= (1ull << 30)) {
            if (vals)
                rc = launch_onesweep<true, true>(kin, kout, vin, vout, m, dop, gb, st, counters + p);
            else
                rc = rs.shift[p] >= 32 ? launch_onesweep<false, true>(kin, kout, vin, vout, m, dhi, gb, st, counters + p)
                                       : launch_onesweep<false, true>(kin, kout, vin, vout, m, dop, gb, st, counters + p);
        } else if (vals)
            rc = launch_onesweep<true, false>(kin, kout, vin, vout, m, dop, gb, st, counters + p);
        else
            rc = rs.shift[p] >= 32 ? launch_onesweep<false, false>(kin, kout, vin, vout, m, dhi, gb, st, counters + p)
                                   : launch_onesweep<false, false>(kin, kout, vin, vout, m, dop, gb, st, counters + p);
        if (rc != 0) return -1;
        std::swap(kin, kout);
        std::swap(vin, vout);
    }
    // kin/vin now hold the sorted data
    dfree(kout);
    if (vals) dfree(vout);
    *keys = kin;
    if (vals) *vals = vin;
    return 0;
}

// Digit plan for `bits` significant key bits starting at word bit `base_shift`: 8-bit
// digits; the last digit may cover bits above the key, which are zero.
RadixShifts shifts_for(int base_shift, int bits)
{
    RadixShifts rs;
    rs.npass = 0;
    for (int b = 0; b < bits && rs.npass < QCE_MAX_PASSES; b += QCE_RADIX_BITS) rs.shift[rs.npass++] = base_shift + b;
    for (int i = rs.npass; i < QCE_MAX_PASSES; i++) rs.shift[i] = 0;
    return rs;
}

// ---- MSD partition + shared-memory finish (k_radix.cuh) --------------------------
constexpr u32 MSD_LOCAL_CAP = 256 * 16; // tuples the largest k_msd_local_sort shape can hold
thread_local bool tl_sort_skewed = false; // set by msd_sort: some sub-bucket holds more than the finish tile (a heavy key)
// The sort runs in three stages: msd_plan decides from the run's length and key range alone whether
// the MSD route applies; msd_level_a scatters the run by its top 8 key bits, from the packed tuples
// or straight from a base column (qce_build_sorted_tuples_base); msd_after_level_a does the rest.
struct MsdPlan {
    u64 n, base;       // the kernels work on key - key_min: base = key_min << 32
    int key_bits, P, R, shiftA, shiftB;
    u32 nbA, nbB, nsub, ntiles0;
};

// Dynamic shared memory of the MSD kernels that need more than the default 48 KB.
constexpr size_t CS_SMEM = 512 * 8 * sizeof(u64) + 4096 * sizeof(u32) + 33 * sizeof(u32); // k_msd_count_sort<512, 8, 3>
constexpr size_t CSB_TILE = (256 * 12 + 2) * sizeof(u64) * 2; // k_msd_count_sort_bulk<256, 12, MAXB>: + MAXB counters
constexpr size_t BIG_SMEM = QCE_MSD_TILE * sizeof(u64) + 3 * 4096 * sizeof(u32); // k_big_partition<4096>
int msd_set_smem_attrs()
{
    static bool set = false;
    if (set) return 0;
    const cudaFuncAttribute a = cudaFuncAttributeMaxDynamicSharedMemorySize;
    CK(cudaFuncSetAttribute(k_msd_partition_bulk<false>, a, (int)QCE_MSDB_SMEM));
    CK(cudaFuncSetAttribute(k_msd_partition_bulk<true>, a, (int)QCE_MSDB_SMEM));
    CK(cudaFuncSetAttribute(k_msd_count_sort<512, 8, 3>, a, (int)CS_SMEM));
    CK(cudaFuncSetAttribute(k_msd_count_sort_bulk<256, 12, 1024>, a, (int)(CSB_TILE + 1024 * sizeof(u32))));
    CK(cudaFuncSetAttribute(k_msd_count_sort_bulk<256, 12, 2048>, a, (int)(CSB_TILE + 2048 * sizeof(u32))));
    CK(cudaFuncSetAttribute(k_msd_count_sort_bulk<256, 12, 4096>, a, (int)(CSB_TILE + 4096 * sizeof(u32))));
    CK(cudaFuncSetAttribute(k_big_partition<4096>, a, (int)BIG_SMEM));
    set = true;
    return 0;
}

// 1: the MSD route applies; 0: the LSD passes sort the run; -1: error.  Flags a run of few
// distinct keys in tl_sort_skewed on the way.
int msd_plan(u64 n, u64 key_min, u64 key_max, MsdPlan *p)
{
    static int enabled = -1;
    if (enabled < 0) {
        const char *e = getenv("QCE_MSD");
        enabled = e ? atoi(e) : 1;
    }
    if (!enabled || n < (1ull << 20)) return 0;
    // the kernels work on key - key_min, so a run that covers only a slice of the
    // key space (a rank's share after the exchange) still spreads over the buckets
    const u64 base = key_min << 32;
    key_max -= key_min;
    const int key_bits = bitlen(key_max);
    if (n / (key_max + 1) >= 16) tl_sort_skewed = true; // 16 or more tuples per possible key: every join tile is heavy
    if (n >= (1ull << 30)) return 0; // the LSD passes sort runs this long
    if (key_bits < 9 || key_bits > 32) return 0;
    // Partition bits P: the smallest count for which a populated sub-bucket holds
    // at most ~2700 tuples on average (finish capacity 4096), assuming keys spread
    // over [0, key_max]; anything denser is caught by the max-bucket check below.
    int P = 9;
    while (P < 16 && P < key_bits && n / (((key_max >> (key_bits - P)) + 1)) > 2700) P++;
    if (n / (((key_max >> (key_bits - P)) + 1)) > 2700) return 0; // too dense for 16 partition bits: LSD
    p->n = n;
    p->base = base;
    p->key_bits = key_bits;
    p->P = P;
    p->R = key_bits - P;
    p->shiftA = 32 + key_bits - 8;
    p->shiftB = 32 + key_bits - P;
    p->nbA = 256;
    p->nbB = 1u << (P - 8);
    p->nsub = p->nbA * p->nbB;
    p->ntiles0 = (u32)ceil_div(n, QCE_MSD_TILE);
    if (msd_set_smem_attrs() != 0) return -1;
    return 1;
}

// Buffers of one MSD sort.  Level A scatters into alt, level B back into the run.
struct MsdLevels {
    Scratch sc;
    u64 *alt = nullptr; // freed with the levels unless a caller takes it
    u32 *lvl0 = nullptr, *histA = nullptr, *offA = nullptr, *curA = nullptr, *tstart1 = nullptr, *histB = nullptr,
        *suboff = nullptr, *curB = nullptr;
    MsdTileDesc *tdesc = nullptr;
    ~MsdLevels() { if (alt) dfree(alt); }
};

// Level A: scatter the run by its top 8 key bits into m->alt.  `in` is the packed run, or with
// from_col the base column itself (k_msd_partition_bulk<true>).  hist_top8: the level-A
// histogram when it is already known (taken while the run was built, or with the column statistics).
int msd_level_a(const MsdPlan &p, MsdLevels *m, const u64 *in, bool from_col, const u32 *hist_top8)
{
    const u64 n = p.n, base = p.base;
    const int shiftA = p.shiftA;
    const u32 nbA = p.nbA, nsub = p.nsub, ntiles0 = p.ntiles0;
    Scratch &sc = m->sc;
    if (dalloc(&m->alt, n) || sc.get(&m->lvl0, 4) || sc.get(&m->histA, nbA) || sc.get(&m->offA, nbA) ||
        sc.get(&m->curA, nbA) || sc.get(&m->tstart1, nbA + 1) || sc.get(&m->histB, nsub) || sc.get(&m->suboff, nsub) ||
        sc.get(&m->curB, nsub))
        return -1;
    u64 *alt = m->alt;
    u32 *lvl0 = m->lvl0, *histA = m->histA, *offA = m->offA, *curA = m->curA;
    // level 0: one bucket = the whole run.  lvl0 = {tile_start[0], tile_start[1], bucket_off, bucket_size}
    const u32 h_lvl0[4] = {0u, ntiles0, 0u, (u32)n};
    CK(cudaMemcpyAsync(lvl0, h_lvl0, sizeof h_lvl0, cudaMemcpyHostToDevice, cx().stream));
    CK(cudaMemsetAsync(histA, 0, nbA * sizeof(u32), cx().stream));
    CK(cudaMemsetAsync(m->histB, 0, nsub * sizeof(u32), cx().stream));
    CK(cudaMemsetAsync(cx().d_scalars + 10, 0, sizeof(u64), cx().stream));
    if (hist_top8)
        CK(cudaMemcpyAsync(histA, hist_top8, nbA * sizeof(u32), cudaMemcpyDeviceToDevice, cx().stream));
    else
        LAUNCH("msd_hist", k_msd_hist, ntiles0, QCE_MSD_THREADS, 0, in, lvl0, lvl0 + 2, lvl0 + 3, 1u, base, shiftA, nbA,
               histA);
    LAUNCH("radix_bases", k_radix_bases, 1, (int)nbA, 0, histA, offA);
    CK(cudaMemcpyAsync(curA, offA, nbA * sizeof(u32), cudaMemcpyDeviceToDevice, cx().stream));
    const u32 ntiles_cap = ntiles0 + nbA;
    const int grid = (int)std::min<u32>(ntiles0, (u32)G.sms * 3);
    if (sc.get(&m->tdesc, ntiles_cap) != 0) return -1;
    LAUNCH("msd_tiles", k_msd_tile_desc, (int)ceil_div(ntiles0, 256), 256, 0, lvl0, lvl0 + 2, lvl0 + 3, 1u, ntiles0, m->tdesc);
    if (from_col)
        LAUNCH("msd_partition", k_msd_partition_bulk<true>, grid, QCE_MSDB_THREADS, QCE_MSDB_SMEM, in, alt, m->tdesc, ntiles0,
               base, shiftA, nbA, curA);
    else
        LAUNCH("msd_partition", k_msd_partition_bulk<false>, grid, QCE_MSDB_THREADS, QCE_MSDB_SMEM, in, alt, m->tdesc, ntiles0,
               base, shiftA, nbA, curA);
    return 0;
}

// Everything after level A: level B back into *keys and the finish.  *done = false means a
// sub-bucket is too heavy for the finish kernels: the caller sorts with the LSD passes instead;
// *keys is then left as it was, and m->alt holds level A's scatter.
int msd_after_level_a(const MsdPlan &p, MsdLevels *m, u64 **keys, bool *done)
{
    *done = false;
    const u64 base = p.base;
    const int R = p.R, shiftB = p.shiftB;
    const u32 nbA = p.nbA, nbB = p.nbB, nsub = p.nsub, ntiles0 = p.ntiles0;
    Scratch &sc = m->sc;
    u64 *alt = m->alt;
    u32 *histA = m->histA, *offA = m->offA, *tstart1 = m->tstart1, *histB = m->histB, *suboff = m->suboff, *curB = m->curB;
    MsdTileDesc *tdesc = m->tdesc;
    // level 1: the 256 buckets of level 0, each cut into tiles of its own
    const u32 ntiles1 = ntiles0 + nbA; // upper bound; surplus CTAs exit
    LAUNCH("msd_tiles", k_msd_tile_starts, 1, 256, 0, histA, nbA, tstart1);
    LAUNCH("msd_hist", k_msd_hist, ntiles1, QCE_MSD_THREADS, 0, alt, tstart1, offA, histA, nbA, base, shiftB, nbB,
           histB);
    LAUNCH("scan_tiles", (k_scan_excl<u32, u32>), 1, 1024, 0, histB, suboff, (u64)nsub, cx().d_scalars + 11);
    LAUNCH("msd_max", k_max_u32, grid_for(256, nsub, 1), 256, 0, histB, nsub, (u32 *)(cx().d_scalars + 10));
    // skew: the sub-buckets a heavy key overflows are listed on the way (k_big_* below)
    constexpr u32 BIG_CAP = 256 * 12, BIG_MAX = 8192;
    static int big_path = -1; // QCE_MSD_BIG=0: any overflowing sub-bucket sends the whole run to the LSD passes
    if (big_path < 0) {
        const char *e = getenv("QCE_MSD_BIG");
        big_path = e ? atoi(e) : 1;
    }
    u32 *big_off = nullptr, *big_size = nullptr, *big_tiles = nullptr;
    if (sc.get(&big_off, BIG_MAX) || sc.get(&big_size, BIG_MAX) || sc.get(&big_tiles, BIG_MAX)) return -1;
    CK(cudaMemsetAsync(cx().d_scalars + 12, 0, sizeof(u64), cx().stream));
    LAUNCH("msd_big_list", k_big_list, (int)ceil_div(nsub, 256), 256, 0, histB, suboff, nsub, BIG_CAP, BIG_MAX,
           (u32 *)(cx().d_scalars + 12), big_off, big_size, big_tiles);
    CK(cudaMemcpyAsync(cx().h_scalars + 10, cx().d_scalars + 10, 3 * sizeof(u64), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    const u32 max_sub = (u32)(cx().h_scalars[10] & 0xffffffffu);
    const u32 nbig = (u32)(cx().h_scalars[12] & 0xffffffffu);
    if (max_sub > 256 * 12) tl_sort_skewed = true;
    // R == 0: the partition levels consumed every key bit, a sub-bucket is one key however large it is
    const bool big_route = max_sub > MSD_LOCAL_CAP && big_path && R > 0 && R <= 12 && nbig <= BIG_MAX;
    if (max_sub <= MSD_LOCAL_CAP || R == 0 || big_route) {
        CK(cudaMemcpyAsync(curB, suboff, nsub * sizeof(u32), cudaMemcpyDeviceToDevice, cx().stream));
        LAUNCH("msd_tiles", k_msd_tile_desc, (int)ceil_div(ntiles1, 256), 256, 0, tstart1, offA, histA, nbA, ntiles1, tdesc);
        LAUNCH("msd_partition", k_msd_partition_bulk<false>, (int)std::min<u32>(ntiles1, (u32)G.sms * 3), QCE_MSDB_THREADS,
               QCE_MSDB_SMEM, alt, *keys, tdesc, ntiles1, base, shiftB, nbB, curB);
        if (R > 0 && R <= 12) {
            if (max_sub <= 256 * 12 || big_route) {
                // persistent, bulk-copy pipelined; the oversized sub-buckets of the big route are skipped here
                const int cgrid = (int)std::min<u32>(nsub, (u32)G.sms * 3);
                if (R <= 10)
                    LAUNCH("msd_count_sort", (k_msd_count_sort_bulk<256, 12, 1024>), cgrid, 256, CSB_TILE + 1024 * sizeof(u32),
                           *keys, suboff, histB, nsub, base, R);
                else if (R == 11)
                    LAUNCH("msd_count_sort", (k_msd_count_sort_bulk<256, 12, 2048>), cgrid, 256, CSB_TILE + 2048 * sizeof(u32),
                           *keys, suboff, histB, nsub, base, R);
                else
                    LAUNCH("msd_count_sort", (k_msd_count_sort_bulk<256, 12, 4096>), cgrid, 256, CSB_TILE + 4096 * sizeof(u32),
                           *keys, suboff, histB, nsub, base, R);
            } else { // 3072 < max_sub <= 4096
                LAUNCH("msd_count_sort", (k_msd_count_sort<512, 8, 3>), nsub, 512, CS_SMEM, *keys, suboff, histB, base, R);
            }
            if (big_route && nbig > 0) {
                // the oversized sub-buckets: one more counting pass on all their remaining bits, through alt
                const u32 nbR = 1u << R, ntiles_big = ntiles0 + nbig; // upper bound; surplus CTAs exit
                u32 *tstartB = nullptr, *bhist = nullptr;
                MsdTileDesc *bdesc = nullptr;
                if (sc.get(&tstartB, nbig + 1) || sc.get(&bhist, (u64)nbig * nbR) || sc.get(&bdesc, ntiles_big)) return -1;
                CK(cudaMemsetAsync(bhist, 0, (u64)nbig * nbR * sizeof(u32), cx().stream));
                LAUNCH("scan_tiles", (k_scan_excl<u32, u32>), 1, 1024, 0, big_tiles, tstartB, (u64)nbig, cx().d_scalars + 13);
                LAUNCH("msd_tiles", k_big_tile_total, 1, 1, 0, tstartB, nbig, cx().d_scalars + 13);
                LAUNCH("msd_tiles", k_msd_tile_desc, (int)ceil_div(ntiles_big, 256), 256, 0, tstartB, big_off, big_size, nbig, ntiles_big, bdesc);
                LAUNCH("msd_big_hist", k_big_hist<4096>, (int)ntiles_big, 512, 0, *keys, bdesc, base, R, bhist);
                LAUNCH("msd_big_scan", k_big_scan, (int)nbig, 1024, 0, bhist, nbR);
                LAUNCH("msd_big_partition", k_big_partition<4096>, (int)ntiles_big, 512, BIG_SMEM, *keys, alt, bdesc, big_off,
                       base, R, bhist);
                LAUNCH("msd_big_copy", k_big_copyback, (int)ntiles_big, 512, 0, alt, *keys, bdesc);
            }
        } else if (R > 0) {
            if (max_sub > MSD_LOCAL_CAP) return 0; // 13..16 remaining bits and a heavy key: the LSD passes
            LocalPlan plan;
            plan.npass = (R + 7) / 8;
            int at = 32;
            for (int p = 0; p < QCE_MAX_PASSES; p++) {
                const int left = R - (at - 32), passes_left = plan.npass - p;
                plan.bits[p] = p < plan.npass ? (left + passes_left - 1) / passes_left : 0;
                plan.shift[p] = at;
                at += plan.bits[p];
            }
            if (max_sub <= 256 * 8)
                LAUNCH("msd_local_sort", (k_msd_local_sort<256, 8, 5>), nsub, 256, 0, *keys, suboff, histB, base, plan);
            else
                LAUNCH("msd_local_sort", (k_msd_local_sort<256, 16, 2>), nsub, 256, 0, *keys, suboff, histB, base, plan);
        }
        *done = true;
    }
    return 0;
}

// For large packed runs.  *done = false means "not applicable or skewed": the
// caller sorts with the LSD passes instead (the run is left untouched).
int msd_sort(u64 **keys, u64 n, u64 key_min, u64 key_max, bool *done, const u32 *hist_top8 = nullptr,
             int hist_key_bits = 0)
{
    *done = false;
    MsdPlan p;
    const int applies = msd_plan(n, key_min, key_max, &p);
    if (applies <= 0) return applies;
    MsdLevels m;
    const bool counted = hist_top8 && key_min == 0 && hist_key_bits == p.key_bits; // level A was counted while the run was built
    if (msd_level_a(p, &m, *keys, false, counted ? hist_top8 : nullptr) != 0) return -1;
    return msd_after_level_a(p, &m, keys, done);
}

// The LSD passes over a packed run's `key_bits` key bits.
int lsd_sort_packed(u64 **a, u64 n, int key_bits)
{
    RadixShifts rs = shifts_for(32, key_bits);
    return radix_sort(a, nullptr, n, rs);
}

// Sort a packed run on its `key_bits` key bits.
int sort_packed(u64 **a, u64 n, int key_bits, u64 key_min, u64 key_max, const u32 *hist_top8 = nullptr,
                int hist_key_bits = 0)
{
    bool done = false;
    if (key_max == 0 || key_max >= (1ull << key_bits)) key_max = (1ull << key_bits) - 1;
    if (key_min > key_max) key_min = 0;
    if (msd_sort(a, n, key_min, key_max, &done, hist_top8, hist_key_bits) != 0) return -1;
    if (done) return 0;
    return lsd_sort_packed(a, n, key_bits);
}

TupleView view_of(const qce_tuples *t)
{
    TupleView v;
    v.a = t->a;
    v.ids = t->ids;
    return v;
}

// ---- merge join driver -------------------------------------------------------
thread_local u32 *tl_join_stats = nullptr; // when set: {min, max} match count per outer tuple of the next merge

// Single-pass join (k_join_fused): the outputs are sized by a guess -- an equi-join along a key /
// foreign-key pair cannot produce more pairs than its larger input has tuples -- and trimmed once the
// pair count is known.  Tiles the guess cannot hold, and tiles dominated by a heavy key, come back as
// a chunk list for k_join_write.  Returns 1 when the guess cannot be allocated: the caller then runs
// the two-phase join, which sizes its outputs exactly.
struct OutGuard {
    qce_rowids *r = nullptr, *s = nullptr;
    ~OutGuard() { qce_rowids_free(r); qce_rowids_free(s); }
};
template <bool WR, bool WS>
int merge_join_fused_t(const qce_tuples *R, const qce_tuples *S, bool want_r, bool want_s, qce_rowids **outR,
                       qce_rowids **outS)
{
    const u32 nR = (u32)R->n, nS = (u32)S->n;
    const u32 ntiles = (u32)ceil_div(nR, QCE_JTILE);
    u64 cap = std::max<u64>(nR, nS);
    static long long cap_env = -1; // QCE_JOIN_CAP: force the guess (tests: 1 = every tile past the first pair is deferred)
    if (cap_env < 0) { const char *e = getenv("QCE_JOIN_CAP"); cap_env = e ? atoll(e) : 0; }
    if (cap_env > 0) cap = (u64)cap_env;
    uint2 *win = nullptr;
    u32 *lb = nullptr, *cnt = nullptr, *tile_chunks = nullptr, *chunk_off = nullptr;
    u64 *tile_off = nullptr, *status = nullptr;
    Scratch sc;
    OutGuard og;
    if (sc.get(&win, ntiles) || sc.get(&lb, nR) || sc.get(&cnt, nR) || sc.get(&tile_chunks, ntiles) ||
        sc.get(&chunk_off, ntiles) || sc.get(&tile_off, ntiles) || sc.get(&status, (u64)ntiles + 1) ||
        (want_r && new_rowids(cap, R->id_bound, &og.r) != 0) || (want_s && new_rowids(cap, S->id_bound, &og.s) != 0))
        return 1;
    TupleView vr = view_of(R), vs = view_of(S);
    // tiles are claimed through an atomic ticket, so a tile's predecessors have started whatever order the CTAs are
    // dispatched in (QCE_JOIN_TICKET=0: tile = blockIdx, which today's dispatcher hands out in order; measured 2 %
    // faster on the join, 0.3 % on a config-2 step -- not worth a look-back that depends on it)
    static int use_ticket = -1;
    if (use_ticket < 0) { const char *e = getenv("QCE_JOIN_TICKET"); use_ticket = e ? atoi(e) : 1; }
    u32 *ticket = use_ticket ? reinterpret_cast<u32 *>(status + ntiles) : nullptr;
    CK(cudaMemsetAsync(status, 0, ((u64)ntiles + 1) * sizeof(u64), cx().stream));
    const u64 init3[3] = {0ull, 0ull, 0x00000000ffffffffull}; // pairs, deferred chunks, {min, max} matches
    CK(cudaMemcpyAsync(cx().d_scalars, init3, sizeof init3, cudaMemcpyHostToDevice, cx().stream));
    LAUNCH("join_partition", (k_join_partition<WR, WS>), (int)ceil_div(ntiles, 256), 256, 0, vr, nR, vs, nS, ntiles, win);
    u32 *stats = tl_join_stats ? (u32 *)(cx().d_scalars + 2) : nullptr;
    u32 *pr = og.r ? og.r->d : nullptr, *ps = og.s ? og.s->d : nullptr;
#define QCE_FUSED_LAUNCH_M(WRF, WSF, M)                                                                              \
    do {                                                                                                             \
        static bool attr_set = false;                                                                                \
        if (!attr_set) {                                                                                             \
            CK(cudaFuncSetAttribute((k_join_fused<WR, WS, WRF, WSF, M>), cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                    (int)QCE_JSMEM_BYTES));                                                          \
            attr_set = true;                                                                                         \
        }                                                                                                            \
        LAUNCH("join_fused", (k_join_fused<WR, WS, WRF, WSF, M>), (int)ntiles, QCE_JTHREADS, QCE_JSMEM_BYTES, vr, nR, vs, \
               win, ntiles, ticket, status, cap, pr, ps, lb, cnt, tile_off, tile_chunks, cx().d_scalars,             \
               cx().d_scalars + 1, stats);                                                                           \
    } while (0)
    static int minb = -1; // QCE_JOIN_MINB=4: 64 registers, 4 CTAs per SM (default 5: 48 registers)
    if (minb < 0) { const char *e = getenv("QCE_JOIN_MINB"); minb = e ? atoi(e) : 5; }
#define QCE_FUSED_LAUNCH(WRF, WSF)                                                                                   \
    do {                                                                                                             \
        if (minb == 4) QCE_FUSED_LAUNCH_M(WRF, WSF, 4);                                                              \
        else QCE_FUSED_LAUNCH_M(WRF, WSF, 5);                                                                        \
    } while (0)
    if (want_r && want_s) QCE_FUSED_LAUNCH(true, true);
    else if (want_r) QCE_FUSED_LAUNCH(true, false);
    else QCE_FUSED_LAUNCH(false, true);
#undef QCE_FUSED_LAUNCH
#undef QCE_FUSED_LAUNCH_M
    if (read_scalars(3) != 0) return -1;
    const u64 m = cx().h_scalars[0], nchunks = cx().h_scalars[1];
    if (tl_join_stats) {
        tl_join_stats[0] = (u32)(cx().h_scalars[2] & 0xffffffffu);
        tl_join_stats[1] = (u32)(cx().h_scalars[2] >> 32);
    }
    if (m >= (1ull << 32)) return fail("join output of %llu pairs exceeds the 2^32 row-id column limit", (unsigned long long)m);
    if (m > cap) {
        // the guess was too small: tiles below it wrote their pairs, move those into outputs of the real size
        OutGuard big;
        if (want_r && new_rowids(m, R->id_bound, &big.r) != 0) return -1;
        if (want_s && new_rowids(m, S->id_bound, &big.s) != 0) return -1;
        if (big.r) CK(cudaMemcpyAsync(big.r->d, og.r->d, cap * sizeof(u32), cudaMemcpyDeviceToDevice, cx().stream));
        if (big.s) CK(cudaMemcpyAsync(big.s->d, og.s->d, cap * sizeof(u32), cudaMemcpyDeviceToDevice, cx().stream));
        std::swap(big.r, og.r);
        std::swap(big.s, og.s);
        pr = og.r ? og.r->d : nullptr;
        ps = og.s ? og.s->d : nullptr;
    } else {
        if (og.r) { cx().arena.shrink(og.r->d, m * sizeof(u32)); og.r->n = m; }
        if (og.s) { cx().arena.shrink(og.s->d, m * sizeof(u32)); og.s->n = m; }
    }
    if (nchunks > 0) {
        if (ntiles <= 512)
            LAUNCH("scan_tiles", (k_scan_excl_warp<u32, u32>), 1, 32, 0, tile_chunks, chunk_off, (u64)ntiles, cx().d_scalars + 1);
        else
            LAUNCH("scan_tiles", (k_scan_excl<u32, u32>), 1, 1024, 0, tile_chunks, chunk_off, (u64)ntiles, cx().d_scalars + 1);
        if (want_r && want_s)
            LAUNCH("join_write", (k_join_write<WR, WS, true, true>), (int)nchunks, QCE_JTHREADS, 0, vr, nR, vs, lb, cnt,
                   tile_off, chunk_off, ntiles, pr, ps);
        else if (want_r)
            LAUNCH("join_write", (k_join_write<WR, WS, true, false>), (int)nchunks, QCE_JTHREADS, 0, vr, nR, vs, lb, cnt,
                   tile_off, chunk_off, ntiles, pr, ps);
        else
            LAUNCH("join_write", (k_join_write<WR, WS, false, true>), (int)nchunks, QCE_JTHREADS, 0, vr, nR, vs, lb, cnt,
                   tile_off, chunk_off, ntiles, pr, ps);
    }
    if (outR) *outR = og.r;
    if (outS) *outS = og.s;
    og.r = og.s = nullptr;
    return 0;
}

template <bool WR, bool WS>
int merge_join_t(const qce_tuples *R, const qce_tuples *S, bool want_r, bool want_s, qce_rowids **outR,
                 qce_rowids **outS, bool walk)
{
    static int fused_on = -1; // QCE_JOIN_FUSED=0: always the two-phase join
    if (fused_on < 0) { const char *e = getenv("QCE_JOIN_FUSED"); fused_on = e ? atoi(e) : 1; }
    // a look-back chain runs at the pace of its slowest tile: a heavy key's tile (a window of millions of inner
    // tuples, searched instead of tabulated) would hold every later tile up -- such joins stay two-phase
    if (!walk && fused_on && !R->skewed && !S->skewed) {
        const int rc = merge_join_fused_t<WR, WS>(R, S, want_r, want_s, outR, outS);
        if (rc <= 0) return rc;
        g_err[0] = 0; // the guess did not fit: size the outputs exactly
    }
    const u32 nR = (u32)R->n, nS = (u32)S->n;
    const u32 ntiles = (u32)ceil_div(nR, QCE_JTILE);
    uint2 *win = nullptr;
    u32 *lb = nullptr, *cnt = nullptr, *tile_chunks = nullptr, *chunk_off = nullptr;
    u64 *tile_total = nullptr, *tile_off = nullptr;
    Scratch sc;
    if (sc.get(&win, ntiles) || sc.get(&lb, nR) || sc.get(&cnt, nR) || sc.get(&tile_chunks, ntiles) ||
        sc.get(&chunk_off, ntiles) || sc.get(&tile_total, ntiles) || sc.get(&tile_off, ntiles))
        return -1;
    TupleView vr = view_of(R), vs = view_of(S);
    if (walk) {
        u64 *tile_max = nullptr, *tile_pm = nullptr;
        if (sc.get(&tile_max, ntiles) || sc.get(&tile_pm, ntiles)) return -1;
        LAUNCH("join_keymax", (k_tile_keymax<WR>), (int)ntiles, QCE_JTHREADS, 0, vr, nR, tile_max);
        LAUNCH("join_keymax", k_scan_excl_max, 1, 32, 0, tile_max, tile_pm, ntiles);
        LAUNCH("join_bounds_walk", (k_join_bounds_walk<WR, WS>), (int)ntiles, QCE_JTHREADS, 0, vr, nR, vs, nS,
               tile_pm, lb, cnt, tile_total, tile_chunks);
    } else {
        LAUNCH("join_partition", (k_join_partition<WR, WS>), (int)ceil_div(ntiles, 256), 256, 0, vr, nR, vs, nS,
               ntiles, win);
        static bool attr_set = false; // per instantiation
        if (!attr_set) {
            CK(cudaFuncSetAttribute(k_join_bounds<WR, WS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)QCE_JSMEM_BYTES));
            attr_set = true;
        }
        if (tl_join_stats) {
            const u32 init[4] = {0xffffffffu, 0u, 0u, 0u}; // d_scalars[2] = {min, max}
            CK(cudaMemcpyAsync(cx().d_scalars + 2, init, sizeof init, cudaMemcpyHostToDevice, cx().stream));
        }
        LAUNCH("join_bounds", (k_join_bounds<WR, WS>), (int)ntiles, QCE_JTHREADS, QCE_JSMEM_BYTES, vr, nR, vs, win,
               lb, cnt, tile_total, tile_chunks, tl_join_stats ? (u32 *)(cx().d_scalars + 2) : nullptr);
    }
    if (ntiles <= 512) {
        LAUNCH("scan_tiles", (k_scan_excl_warp<u64, u64>), 1, 32, 0, tile_total, tile_off, (u64)ntiles, cx().d_scalars);
        LAUNCH("scan_tiles", (k_scan_excl_warp<u32, u32>), 1, 32, 0, tile_chunks, chunk_off, (u64)ntiles,
               cx().d_scalars + 1);
    } else {
        LAUNCH("scan_tiles", (k_scan_excl<u64, u64>), 1, 1024, 0, tile_total, tile_off, (u64)ntiles, cx().d_scalars);
        LAUNCH("scan_tiles", (k_scan_excl<u32, u32>), 1, 1024, 0, tile_chunks, chunk_off, (u64)ntiles,
               cx().d_scalars + 1);
    }
    if (tl_join_stats && walk) {
        const u32 init[4] = {0xffffffffu, 0u, 0u, 0u}; // d_scalars[2] = {min, max}
        CK(cudaMemcpyAsync(cx().d_scalars + 2, init, sizeof init, cudaMemcpyHostToDevice, cx().stream));
        LAUNCH("join_stats", k_minmax_u32, grid_for(1024, nR, 4), 256, 0, cnt, nR, (u32 *)(cx().d_scalars + 2), (u32 *)(cx().d_scalars + 2) + 1);
    }
    if (read_scalars(3) != 0) return -1;
    const u64 m = cx().h_scalars[0], nchunks = cx().h_scalars[1];
    if (tl_join_stats) {
        tl_join_stats[0] = (u32)(cx().h_scalars[2] & 0xffffffffu);
        tl_join_stats[1] = (u32)(cx().h_scalars[2] >> 32);
    }
    if (m >= (1ull << 32)) return fail("join output of %llu pairs exceeds the 2^32 row-id column limit", (unsigned long long)m);
    qce_rowids *oR = nullptr, *oS = nullptr;
    if (want_r && new_rowids(m, R->id_bound, &oR) != 0) return -1;
    if (want_s && new_rowids(m, S->id_bound, &oS) != 0) { qce_rowids_free(oR); return -1; }
    if (m > 0) {
        u32 *pr = oR ? oR->d : nullptr, *ps = oS ? oS->d : nullptr;
        if (want_r && want_s)
            LAUNCH("join_write", (k_join_write<WR, WS, true, true>), (int)nchunks, QCE_JTHREADS, 0, vr, nR, vs, lb,
                   cnt, tile_off, chunk_off, ntiles, pr, ps);
        else if (want_r)
            LAUNCH("join_write", (k_join_write<WR, WS, true, false>), (int)nchunks, QCE_JTHREADS, 0, vr, nR, vs, lb,
                   cnt, tile_off, chunk_off, ntiles, pr, ps);
        else
            LAUNCH("join_write", (k_join_write<WR, WS, false, true>), (int)nchunks, QCE_JTHREADS, 0, vr, nR, vs, lb,
                   cnt, tile_off, chunk_off, ntiles, pr, ps);
    }
    if (outR) *outR = oR;
    if (outS) *outS = oS;
    return 0;
}

int merge_join_any(const qce_tuples *R, const qce_tuples *S, bool want_r, bool want_s, qce_rowids **outR,
                   qce_rowids **outS, bool walk = false)
{
    if (R->n >= (1ull << 32) || S->n >= (1ull << 32)) return fail("join input exceeds 2^32 tuples");
    if (R->n == 0 || S->n == 0) {
        if (tl_join_stats && R->n) tl_join_stats[0] = 0; // outer tuples without a single match
        if (outR) *outR = nullptr;
        if (outS) *outS = nullptr;
        if (want_r && new_rowids(0, R->id_bound, outR) != 0) return -1;
        if (want_s && new_rowids(0, S->id_bound, outS) != 0) return -1;
        return 0;
    }
    if (R->wide && S->wide) return merge_join_t<true, true>(R, S, want_r, want_s, outR, outS, walk);
    if (R->wide) return merge_join_t<true, false>(R, S, want_r, want_s, outR, outS, walk);
    if (S->wide) return merge_join_t<false, true>(R, S, want_r, want_s, outR, outS, walk);
    return merge_join_t<false, false>(R, S, want_r, want_s, outR, outS, walk);
}

// distinct (rowid_R,rowid_S) pairs of a join output: pack, sort every
// significant bit, flag heads, compact.
int distinct_pairs(const qce_rowids *pr, const qce_rowids *ps, qce_rowids **dr, qce_rowids **ds)
{
    const u64 m = pr->n;
    if (m == 0) {
        if (new_rowids(0, pr->id_bound, dr) != 0) return -1;
        return new_rowids(0, ps->id_bound, ds);
    }
    u64 *w = nullptr;
    if (dalloc(&w, m) != 0) return -1;
    LAUNCH("pack_pairs", k_pack_pairs, grid_for(256, m), 256, 0, pr->d, ps->d, m, w);
    const int bits_s = ps->id_bound ? bitlen(ps->id_bound - 1) : 32;
    const int bits_r = pr->id_bound ? bitlen(pr->id_bound - 1) : 32;
    RadixShifts rs;
    rs.npass = 0;
    for (int b = 0; b < bits_s; b += 8) rs.shift[rs.npass++] = b;
    for (int b = 0; b < bits_r; b += 8) rs.shift[rs.npass++] = 32 + b;
    for (int i = rs.npass; i < QCE_MAX_PASSES; i++) rs.shift[i] = 0;
    if (radix_sort(&w, nullptr, m, rs) != 0) return -1;
    const u64 ntiles = ceil_div(m, QCE_FTILE);
    u32 *mask = nullptr, *tile_count = nullptr;
    if (dalloc(&mask, ntiles * QCE_FWORDS) || dalloc(&tile_count, ntiles)) return -1;
    LAUNCH("unique_mask", k_unique_mask, (int)ntiles, QCE_FTHREADS, 0, w, m, mask, tile_count);
    int rc = compact_from_mask(QCE_LAYOUT_NATURAL, QCE_EMIT_PACKED, mask, tile_count, ntiles, w, nullptr,
                               pr->id_bound, ps->id_bound, dr, ds);
    dfree(mask); dfree(tile_count); dfree(w);
    return rc;
}


// ---- bucketed gather support (qce_checksum) ------------------------------------
// Worth it when the column is much larger than L2 and there are enough ids for
// the extra pass (8 B/id) to cost less than the DRAM over-fetch it removes.
bool bucketed_checksum_pays(const qce_rowids *ids, u64 col_rows)
{
    static int mode = -1; // QCE_BUCKETED_CHECKSUM=0 disables, =1 forces
    if (mode < 0) {
        const char *e = getenv("QCE_BUCKETED_CHECKSUM");
        mode = e ? atoi(e) + 1 : 0;
    }
    if (mode == 1) return false;
    if (mode == 2) return ids->n >= 2;
    if (ids->id_bound > ids->id_min) col_rows = std::min<u64>(col_rows, ids->id_bound - ids->id_min);
    return col_rows * sizeof(u64) > (256ull << 20) && ids->n >= (4ull << 20) && ids->n < (1ull << 30);
}

int partition_ids_by_top_bits(const qce_rowids *ids, u32 **out)
{
    // unstable MSD partition of the 4-byte ids by their top 8 bits (the order inside
    // a bucket is irrelevant for a sum): histogram, prefix, one scatter pass
    const u64 n = ids->n;
    const u32 base = ids->id_bound > ids->id_min ? ids->id_min : 0u;
    const int bits = ids->id_bound ? bitlen(ids->id_bound - 1 - base) : 32;
    const int shift = bits > 8 ? bits - 8 : 0;
    const u32 ntiles = (u32)ceil_div(n, QCE_MSD_TILE);
    u32 *ghist = nullptr, *cursor = nullptr, *lvl0 = nullptr, *dst = nullptr;
    if (dalloc(&dst, n) || dalloc(&ghist, QCE_RADIX_BINS) || dalloc(&cursor, QCE_RADIX_BINS) || dalloc(&lvl0, 4)) return -1;
    const u32 h_lvl0[4] = {0u, ntiles, 0u, (u32)n};
    CK(cudaMemcpyAsync(lvl0, h_lvl0, sizeof h_lvl0, cudaMemcpyHostToDevice, cx().stream));
    CK(cudaMemsetAsync(ghist, 0, QCE_RADIX_BINS * sizeof(u32), cx().stream));
    LAUNCH("hist_u32", k_hist_u32, grid_for(2048, n, 4), 512, 0, ids->d, n, base, shift, ghist);
    LAUNCH("radix_bases", k_radix_bases, 1, 256, 0, ghist, cursor);
    LAUNCH("partition_u32", (k_msd_partition<512, 8, u32>), ntiles, 512, 0, (const u32 *)ids->d, dst, lvl0, lvl0 + 2,
           lvl0 + 3, 1u, base, shift, 256u, cursor, (const u32 *)nullptr);
    dfree(ghist); dfree(cursor); dfree(lvl0);
    *out = dst;
    return 0;
}

int scan_join_impl(const Column *cr, const qce_rowids *idsR, const Column *cs, const qce_rowids *idsS,
                          qce_rowids **outR, qce_rowids **outS)
{
    const u64 nr = idsR ? idsR->n : cr->n, ns = idsS ? idsS->n : cs->n;
    const u64 n = nr < ns ? nr : ns;
    if (n == 0) {
        if (new_rowids(0, (u32)cr->n, outR) != 0) return -1;
        return new_rowids(0, (u32)cs->n, outS);
    }
    const u64 ntiles = ceil_div(n, QCE_FTILE);
    u32 *mask = nullptr, *tile_count = nullptr;
    if (dalloc(&mask, ntiles * QCE_FWORDS) || dalloc(&tile_count, ntiles)) return -1;
    LAUNCH("scan_join", k_scanjoin_mask, (int)ntiles, QCE_FTHREADS, 0, idsR ? idsR->d : nullptr, ref_of(cr),
           idsS ? idsS->d : nullptr, ref_of(cs), n, mask, tile_count);
    int rc = compact_from_mask(QCE_LAYOUT_NATURAL, QCE_EMIT_SRC2, mask, tile_count, ntiles,
                               idsR ? idsR->d : nullptr, idsS ? idsS->d : nullptr, (u32)cr->n, (u32)cs->n, outR, outS);
    dfree(mask);
    dfree(tile_count);
    return rc;
}

} // namespace

#include "qce_shard.cuh"

// =============================================================== C-ABI
extern "C" {

int qce_abi_version(void) { return QCE_ABI_VERSION; }
const char *qce_last_error(void) { return g_err; }

static int ctx_open(Ctx *c)
{
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CK(cudaMalloc((void **)&c->d_scalars, 16 * sizeof(u64)));
    CK(cudaMallocHost((void **)&c->h_scalars, 16 * sizeof(u64)));
    CK(cudaEventCreate(&c->t0));
    CK(cudaEventCreate(&c->t1));
    {
        // the early sort must get SM slots while the other side's push (a grid of thousands of CTAs,
        // launched first) is still draining: blocks of a higher-priority stream are dispatched first
        int lo = 0, hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(cudaStreamCreateWithPriority(&c->aux, cudaStreamNonBlocking, hi));
    }
    CK(cudaEventCreateWithFlags(&c->ev_side[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->ev_side[1], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->ev_aux, cudaEventDisableTiming));
    return 0;
}
static void ctx_close(Ctx *c)
{
    if (!c->stream) return;
    cudaStreamSynchronize(c->stream);
    c->arena.release_all();
    for (auto &r : c->prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    c->prof.clear();
    c->ev_pool.clear();
    cudaFree(c->d_scalars);
    cudaFreeHost(c->h_scalars);
    cudaEventDestroy(c->t0);
    cudaEventDestroy(c->t1);
    cudaEventDestroy(c->ev_side[0]);
    cudaEventDestroy(c->ev_side[1]);
    cudaEventDestroy(c->ev_aux);
    cudaStreamDestroy(c->aux);
    cudaStreamDestroy(c->stream);
    c->stream = nullptr;
}

int qce_init(int device)
{
    if (G.inited) return 0;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail("no CUDA device available (%s); this engine has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0) {
        // one process per GPU: the rank inside the node picks the device (several ranks may
        // share one when there are fewer devices than ranks, e.g. the single-GPU test box)
        const char *lr = getenv("LOCAL_RANK");
        const bool forked = qcecomm::st().forked_child || !qcecomm::st().children.empty();
        device = (lr && !forked) ? atoi(lr) % count : (int)(qcecomm::st().rank % (u32)count);
    }
    if (device >= count) return fail("device %d out of range (%d visible)", device, count);
    CK(cudaSetDevice(device));
    G.device = device;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    G.sms = prop.multiProcessorCount;
    if (ctx_open(&g_main) != 0) return -1;
    G.inited = true;
    g_err[0] = 0;
    return 0;
}

int qce_xwin_destroy(void);
int qce_xwin_unmap_peers(void);
namespace stager { static void release(); }
void qce_shutdown(void)
{
    if (!G.inited) return;
    for (Ctx *w : G.workers) { ctx_close(w); delete w; }
    G.workers.clear();
    tl_ctx = nullptr;
    qce_drop_relations();
    qce_xwin_destroy(); // unmaps the peers' windows and frees this rank's
    stager::release();
    ctx_close(&g_main);
    G.inited = false;
}

// ---- worker contexts (SURVEY.md 8f-3: the batch scheduler's streams) -----------------
// A context is a stream with its own scalar scratch and arena.  qce_ctx_bind(handle)
// makes it the calling thread's context (NULL = back to the main one); handles are
// created and destroyed by the main thread while no worker is running.
void *qce_ctx_create(void)
{
    if (!G.inited && qce_init(-1) != 0) return nullptr;
    Ctx *c = new Ctx();
    c->arena.min_slab = 64ull << 20;
    c->solo = true;
    if (ctx_open(c) != 0) { delete c; return nullptr; }
    std::lock_guard<std::mutex> lk(G.mu);
    G.workers.push_back(c);
    return c;
}
int qce_ctx_bind(void *handle)
{
    if (!G.inited && qce_init(-1) != 0) return -1;
    CK(cudaSetDevice(G.device)); // a fresh host thread starts on device 0
    tl_ctx = (Ctx *)handle;
    return 0;
}
/* The calling thread's context runs whole queries on this rank alone (1) or takes part in the
 * ranks' sharded operators (0, the main context's default). */
int qce_ctx_solo(int on)
{
    if (!G.inited && qce_init(-1) != 0) return -1;
    cx().solo = on != 0;
    return 0;
}
void qce_ctx_destroy(void *handle)
{
    Ctx *c = (Ctx *)handle;
    if (!c) return;
    if (tl_ctx == c) tl_ctx = nullptr;
    {
        std::lock_guard<std::mutex> lk(G.mu);
        G.workers.erase(std::remove(G.workers.begin(), G.workers.end(), c), G.workers.end());
    }
    ctx_close(c);
    delete c;
}

int qce_sync(void)
{
    NEED_INIT();
    CK(cudaStreamSynchronize(cx().stream));
    return 0;
}

int qce_timer_reset(void)
{
    NEED_INIT();
    cx().launches = 0;
    {
        std::lock_guard<std::mutex> lk(G.mu); // the worker contexts are idle between batches
        for (Ctx *w : G.workers) w->launches = 0;
    }
    CK(cudaEventRecord(cx().t0, cx().stream));
    return 0;
}
int qce_timer_read(double *ms, uint64_t *kernel_launches)
{
    NEED_INIT();
    CK(cudaEventRecord(cx().t1, cx().stream));
    CK(cudaEventSynchronize(cx().t1));
    float f = 0;
    CK(cudaEventElapsedTime(&f, cx().t0, cx().t1));
    if (ms) *ms = f;
    if (kernel_launches) {
        u64 n = cx().launches;
        std::lock_guard<std::mutex> lk(G.mu);
        for (Ctx *w : G.workers)
            if (w != &cx()) n += w->launches;
        *kernel_launches = n;
    }
    return 0;
}

int qce_mempool_stats(uint64_t *reserved_bytes, uint64_t *used_bytes)
{
    NEED_INIT();
    if (reserved_bytes) *reserved_bytes = cx().arena.reserved();
    if (used_bytes) *used_bytes = cx().arena.used();
    return 0;
}

// Per-kernel device times (CUDA events around every launch); off by default.
int qce_profile_enable(int on)
{
    NEED_INIT();
    CK(cudaStreamSynchronize(cx().stream));
    for (auto &r : cx().prof) { cx().ev_pool.push_back(r.e0); cx().ev_pool.push_back(r.e1); }
    cx().prof.clear();
    cx().profile = on != 0;
    return 0;
}
// JSON object {"tag": {"launches": n, "ms": total}, ...} of everything recorded
// since qce_profile_enable(1); the pointer stays valid until the next call.
const char *qce_profile_json(void)
{
    if (!G.inited) return "{}";
    cudaStreamSynchronize(cx().stream);
    std::map<std::string, std::pair<u64, double>> agg;
    for (size_t k = 0; k < cx().prof.size(); k++) {
        auto &r = cx().prof[k];
        float f = 0;
        if (cudaEventElapsedTime(&f, r.e0, r.e1) == cudaSuccess) {
            auto &a = agg[r.tag];
            a.first++;
            a.second += f;
        }
        // stream time between the end of the previous kernel and the start of
        // this one: memsets, copies and host round trips
        if (k > 0 && cudaEventElapsedTime(&f, cx().prof[k - 1].e1, r.e0) == cudaSuccess) {
            auto &a = agg[std::string("gap_before:") + r.tag];
            a.first++;
            a.second += f;
        }
    }
    cx().prof_json = "{";
    bool first = true;
    for (auto &kv : agg) {
        char buf[256];
        snprintf(buf, sizeof buf, "%s\"%s\": {\"launches\": %llu, \"ms\": %.6f}", first ? "" : ", ",
                 kv.first.c_str(), (unsigned long long)kv.second.first, kv.second.second);
        cx().prof_json += buf;
        first = false;
    }
    cx().prof_json += "}";
    return cx().prof_json.c_str();
}

// ---------------------------------------------------------------- ranks of the node
// See qce_comm.cuh.  world == 1 until one of these is called.
int qce_comm_fork(uint32_t world)
{
    if (G.inited) return fail("qce_comm_fork must run before the process touches CUDA");
    if (qcecomm::fork_ranks(world) != 0) return fail("%s", qcecomm::st().err);
    G.world = qcecomm::st().world;
    G.rank = qcecomm::st().rank;
    return (int)G.rank;
}
int qce_comm_attach(const char *name, uint32_t rank, uint32_t world, uint64_t token)
{
    if (!name) return fail("null argument");
    if (qcecomm::attach_named(name, rank, world, token) != 0) return fail("%s", qcecomm::st().err);
    G.world = world;
    G.rank = rank;
    return 0;
}
uint32_t qce_comm_rank(void) { return G.rank; }
uint32_t qce_comm_world(void) { return G.world; }
int qce_comm_is_child(void) { return qcecomm::st().forked_child ? 1 : 0; }
int qce_comm_barrier(void)
{
    if (qcecomm::barrier() != 0) return fail("%s", qcecomm::st().err);
    return 0;
}
int qce_comm_allreduce_sum_u64(uint64_t *v, uint32_t n)
{
    if (qcecomm::allreduce_sum(v, n) != 0) return fail("%s", qcecomm::st().err);
    return 0;
}
int qce_comm_allreduce_max_u64(uint64_t *v, uint32_t n)
{
    if (qcecomm::allreduce_max(v, n) != 0) return fail("%s", qcecomm::st().err);
    return 0;
}
// Variable-length blobs to rank 0: *out (malloc'ed, rank 0 only) = the ranks' blobs one after
// another, lens[r] = rank r's length (every rank receives the lengths).
int qce_comm_gatherv(const void *mine, uint64_t bytes, char **out, uint64_t *lens)
{
    std::vector<std::string> all;
    if (qcecomm::gatherv_root(mine, bytes, &all) != 0) return fail("%s", qcecomm::st().err);
    u64 total = 0;
    for (u32 r = 0; r < G.world; r++) total += all[r].size();
    if (lens) {
        std::vector<uint64_t> l(G.world, 0);
        uint64_t me = bytes;
        if (qcecomm::allgather(&me, sizeof me, l.data()) != 0) return fail("%s", qcecomm::st().err);
        for (u32 r = 0; r < G.world; r++) lens[r] = l[r];
    }
    if (out) {
        *out = nullptr;
        if (G.rank == 0) {
            *out = (char *)malloc(total ? total : 1);
            u64 at = 0;
            for (u32 r = 0; r < G.world; r++) { memcpy(*out + at, all[r].data(), all[r].size()); at += all[r].size(); }
        }
    }
    return 0;
}
void qce_comm_abort(void) { qcecomm::abort_all(); }
// fork mode: rank 0 collects its children (returns how many failed); a child never returns
int qce_comm_finish(int status)
{
    if (qcecomm::st().forked_child) {
        fflush(stderr);
        _exit(status);
    }
    const int bad = qcecomm::join_children();
    qcecomm::detach();
    G.world = 1;
    G.rank = 0;
    return bad;
}

// ---------------------------------------------------------------- relations
// Placement of a base column over the ranks of the node (world > 1):
//   whole    every rank holds all rows (columns up to G.replicate_bytes): every gather is local,
//            whole queries over such relations can run on one rank alone (replica queries);
//   window   rank r holds rows [r * rpr, (r+1) * rpr) only, rpr = ceil(n / world) rounded up to
//            4096; the peers' windows are mapped through CUDA IPC, so a gather of a foreign row
//            is an NVLink load (ColRef) and nothing is replicated.
static void release_column(Column &c)
{
    for (void *p : c.opened) cudaIpcCloseMemHandle(p);
    c.opened.clear();
    if (c.owned && c.alloc) cudaFree(c.alloc);
    c.alloc = nullptr;
    c.owned = false;
    if (c.hist) cudaFree(c.hist);
    c.hist = nullptr;
    c.hist_bits = 0;
}
// the buffer of (rel, col): the previous upload's when the shape is unchanged (a refreshed
// batch of the same relation), else a fresh cudaMalloc.  *reused tells the caller whether the
// peers' IPC mappings of a window are still valid.
static int column_buffer(u32 rel, u32 col, u64 bytes, Column *c, bool *reused)
{
    *reused = false;
    {
        std::lock_guard<std::mutex> lk(G.mu);
        auto it = G.cols.find(col_key(rel, col));
        if (it != G.cols.end()) {
            if (it->second.owned && it->second.alloc && it->second.alloc_bytes == bytes) {
                *c = it->second;
                *reused = true;
                return 0;
            }
            release_column(it->second);
            G.cols.erase(it);
        }
    }
    *c = Column();
    CK(cudaMalloc(&c->alloc, bytes ? bytes : 16));
    c->alloc_bytes = bytes;
    c->owned = true;
    return 0;
}
// hist_of: a whole column, whose level-A histogram (Column::hist) is taken in the same pass
static int column_max(const u64 *d, u64 n, u64 *maxv, bool *in_order = nullptr, Column *hist_of = nullptr)
{
    const bool hist = hist_of && n >= (1ull << 20);
    if (hist_of) hist_of->hist_bits = 0;
    Scratch sc;
    u32 *lhist = nullptr;
    if (hist) {
        if (sc.get(&lhist, QCE_LEN_BINS) != 0) return -1;
        CK(cudaMemsetAsync(lhist, 0, QCE_LEN_BINS * sizeof(u32), cx().stream));
    }
    CK(cudaMemsetAsync(cx().d_scalars + 8, 0, 2 * sizeof(u64), cx().stream));
    if (hist)
        LAUNCH("column_stats", k_column_stats<true>, grid_for(512, n, 4), 256, 0, d, n, cx().d_scalars + 8,
               (u32 *)(cx().d_scalars + 9), lhist);
    else if (n > 0)
        LAUNCH("column_stats", k_column_stats<false>, grid_for(512, n, 4), 256, 0, d, n, cx().d_scalars + 8,
               (u32 *)(cx().d_scalars + 9), (u32 *)nullptr);
    CK(cudaMemcpyAsync(cx().h_scalars + 8, cx().d_scalars + 8, 2 * sizeof(u64), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    *maxv = cx().h_scalars[8];
    if (in_order) *in_order = (cx().h_scalars[9] & 0xffffffffu) == 0;
    const int b = bitlen(*maxv);
    if (hist && b >= 9 && b <= 32) {
        if (!hist_of->hist) CK(cudaMalloc(&hist_of->hist, QCE_RADIX_BINS * sizeof(u32)));
        LAUNCH("column_stats", k_column_hist_fold, 1, 256, 0, lhist, b, hist_of->hist);
        hist_of->hist_bits = b;
    }
    return 0;
}
static void install_column(u32 rel, u32 col, const Column &c)
{
    std::lock_guard<std::mutex> lk(G.mu);
    G.cols[col_key(rel, col)] = c;
}

// ---- host -> device copies --------------------------------------------------------
// A relation file is mmap'ed pageable memory: a plain cudaMemcpy goes through the driver's
// single bounce buffer (~11 GB/s measured on the B200 box).  Large copies are staged by a
// small pool of threads through pinned chunks instead (8 threads x 2 x 8 MB: 40-45 GB/s
// measured, tools/probes/ipc_probe.cu); pinned sources and small copies go straight down.
namespace stager {
constexpr size_t kChunk = 8u << 20;
constexpr int kThreads = 8;
struct Pool {
    char *pin = nullptr;
    cudaStream_t st[kThreads];
    cudaEvent_t ev[kThreads * 2];
    bool ok = false;
};
static Pool g_pool;
static std::mutex g_pool_mu;
static int ensure()
{
    if (g_pool.ok) return 0;
    CK(cudaMallocHost((void **)&g_pool.pin, kChunk * kThreads * 2));
    for (auto &x : g_pool.st) CK(cudaStreamCreateWithFlags(&x, cudaStreamNonBlocking));
    for (auto &x : g_pool.ev) CK(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
    g_pool.ok = true;
    return 0;
}
static void release()
{
    if (!g_pool.ok) return;
    for (auto &x : g_pool.st) cudaStreamDestroy(x);
    for (auto &x : g_pool.ev) cudaEventDestroy(x);
    cudaFreeHost(g_pool.pin);
    g_pool = Pool();
}
static int copy(void *dst, const void *src, size_t bytes)
{
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (ensure() != 0) return -1;
    const size_t nch = (bytes + kChunk - 1) / kChunk;
    std::atomic<size_t> next{0};
    std::atomic<int> bad{0};
    const int device = G.device;
    std::vector<std::thread> th;
    const int nthr = (int)std::min<size_t>(kThreads, nch);
    for (int t = 0; t < nthr; t++)
        th.emplace_back([&, t] {
            cudaSetDevice(device);
            int flip = 0;
            size_t c;
            while ((c = next.fetch_add(1)) < nch) {
                const int b = t * 2 + flip;
                flip ^= 1;
                const size_t off = c * kChunk, len = std::min(kChunk, bytes - off);
                if (cudaEventSynchronize(g_pool.ev[b]) != cudaSuccess) bad = 1;
                memcpy(g_pool.pin + (size_t)b * kChunk, (const char *)src + off, len);
                if (cudaMemcpyAsync((char *)dst + off, g_pool.pin + (size_t)b * kChunk, len, cudaMemcpyHostToDevice,
                                    g_pool.st[t]) != cudaSuccess)
                    bad = 1;
                cudaEventRecord(g_pool.ev[b], g_pool.st[t]);
            }
            if (cudaStreamSynchronize(g_pool.st[t]) != cudaSuccess) bad = 1;
        });
    for (auto &x : th) x.join();
    if (bad) {
        (void)cudaGetLastError();
        return fail("staged host-to-device copy failed");
    }
    return 0;
}
} // namespace stager

static int h2d(void *dst, const void *src, u64 bytes)
{
    if (bytes == 0) return 0;
    static int mode = -1; // QCE_STAGED_UPLOAD=0: always the plain copy (for comparison)
    if (mode < 0) { const char *e = getenv("QCE_STAGED_UPLOAD"); mode = e ? atoi(e) : 1; }
    bool pageable = false;
    if (mode && bytes >= (32ull << 20)) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, src) != cudaSuccess) { (void)cudaGetLastError(); pageable = true; }
        else pageable = at.type == cudaMemoryTypeUnregistered;
    }
    if (pageable) return stager::copy(dst, src, bytes);
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, cx().stream));
    return 0;
}

// map every rank's window of a row-sharded column (collective)
static int share_window(Column *c, u64 per, bool reused)
{
    c->rpr = (u32)per;
    c->last_rank = G.world - 1;
    c->peer_mapped = true;
    if (!reused) {
        cudaIpcMemHandle_t mine, all[QCE_MAX_RANKS];
        CK(cudaIpcGetMemHandle(&mine, c->alloc));
        if (qcecomm::allgather(&mine, sizeof mine, all) != 0) return fail("%s", qcecomm::st().err);
        for (u32 q = 0; q < G.world; q++) {
            if (q == G.rank) { c->vb[q] = (const u64 *)c->alloc - (u64)q * per; continue; }
            void *p = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&p, all[q], cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                (void)cudaGetLastError();
                qcecomm::abort_all();
                return fail("cannot map rank %u's column window (%s): no peer access between these GPUs", q, cudaGetErrorString(e));
            }
            c->opened.push_back(p);
            c->vb[q] = (const u64 *)p - (u64)q * per;
        }
    }
    uint64_t m = c->maxv;
    if (qcecomm::allreduce_max(&m, 1) != 0) return fail("%s", qcecomm::st().err);
    c->maxv = m;
    return 0;
}

// QCE_REPLICATE_BYTES: read once, before the first placement decision (which the host layer
// takes before the engine is initialised: it forks the ranks first)
static void placement_env()
{
    static bool done = false;
    if (done) return;
    done = true;
    if (const char *rb = getenv("QCE_REPLICATE_BYTES")) {
        G.replicate_bytes = strtoull(rb, nullptr, 10);
        G.replicate_forced = true;
    }
}
enum { SRC_HOST = 0, SRC_DEVICE = 1 };
// `src` holds rows [src_begin, src_begin + src_count) of the relation (the whole column when
// src_count == rows_global)
static int upload_impl(u32 rel, u32 col, const void *src, int src_kind, u64 src_begin, u64 src_count, u64 rows_global)
{
    if (rows_global >= (1ull << 32)) return fail("relation %u has %llu rows; device row ids are 32-bit", rel, (unsigned long long)rows_global);
    placement_env();
    const bool have_all = src_begin == 0 && src_count == rows_global;
    const bool whole = G.world == 1 || (have_all && rows_global * sizeof(u64) <= G.replicate_bytes);
    u64 begin = 0, count = rows_global, per = rows_global;
    if (!whole) row_share(rows_global, G.rank, G.world, &begin, &count, &per);
    if (!whole && !(src_begin <= begin && begin + count <= src_begin + src_count))
        return fail("rank %u needs rows [%llu, +%llu) of relation %u; the caller supplied [%llu, +%llu)", G.rank,
                    (unsigned long long)begin, (unsigned long long)count, rel, (unsigned long long)src_begin, (unsigned long long)src_count);
    Column c;
    bool reused = false;
    if (column_buffer(rel, col, (whole ? rows_global : per) * sizeof(u64), &c, &reused) != 0) return -1;
    const char *from = (const char *)src + (begin - src_begin) * sizeof(u64);
    if (count) {
        if (src_kind == SRC_HOST) { if (h2d(c.alloc, from, count * sizeof(u64)) != 0) return -1; }
        else CK(cudaMemcpyAsync(c.alloc, from, count * sizeof(u64), cudaMemcpyDeviceToDevice, cx().stream));
    }
    c.d = (const u64 *)c.alloc - begin; // virtual base: row id r lives at d[r]
    c.n = rows_global;
    c.windowed = !whole;
    c.win_begin = begin;
    c.win_count = count;
    if (column_max((const u64 *)c.alloc, count, &c.maxv, &c.in_order, whole ? &c : nullptr) != 0) return -1;
    if (!whole) c.hist_bits = 0; // a re-upload of the same shape keeps the buffer, not its counts
    if (!whole) c.in_order = false; // a row window: the runs built from it are exchanged by key range anyway
    if (!whole && share_window(&c, per, reused) != 0) return -1;
    install_column(rel, col, c);
    return 0;
}

int qce_upload_column(uint32_t rel, uint32_t col, const uint64_t *host, uint64_t n)
{
    NEED_INIT();
    return upload_impl(rel, col, host, SRC_HOST, 0, n, n);
}
int qce_upload_column_device(uint32_t rel, uint32_t col, const void *dev, uint64_t n)
{
    NEED_INIT();
    return upload_impl(rel, col, dev, SRC_DEVICE, 0, n, n);
}
/* The caller holds only rows [row_begin, row_begin + row_count) -- its rank's share of a
 * row-sharded relation (qce_row_share) -- in host or device memory. */
int qce_upload_column_window(uint32_t rel, uint32_t col, const uint64_t *host, uint64_t row_begin, uint64_t row_count,
                             uint64_t rows_global)
{
    NEED_INIT();
    return upload_impl(rel, col, host, SRC_HOST, row_begin, row_count, rows_global);
}
int qce_upload_column_window_device(uint32_t rel, uint32_t col, const void *dev, uint64_t row_begin, uint64_t row_count,
                                    uint64_t rows_global)
{
    NEED_INIT();
    return upload_impl(rel, col, dev, SRC_DEVICE, row_begin, row_count, rows_global);
}
int qce_row_share(uint64_t rows_global, uint32_t rank, uint32_t world, uint64_t *row_begin, uint64_t *row_count)
{
    if (!row_begin || !row_count || world == 0 || rank >= world) return fail("bad argument");
    u64 b, c;
    row_share(rows_global, rank, world, &b, &c);
    *row_begin = b;
    *row_count = c;
    return 0;
}
int qce_column_would_be_whole(uint64_t rows)
{
    placement_env();
    return (G.world == 1 || rows * sizeof(u64) <= G.replicate_bytes) ? 1 : 0;
}
/* Placement of a batch's columns (several ranks): every rank holds whole the columns that fit, taken
 * smallest first, into QCE_REPLICATE_FRACTION (default 0.45) of the device memory; larger relations are
 * row-sharded.  *cap_bytes = the largest column size that is still replicated (pass it to
 * qce_set_replicate_bytes before the uploads).  An explicit QCE_REPLICATE_BYTES wins. */
int qce_placement_cap(const uint64_t *col_rows, uint32_t ncols, uint64_t *cap_bytes)
{
    NEED_INIT();
    if (!cap_bytes || (ncols && !col_rows)) return fail("null argument");
    placement_env();
    if (G.replicate_forced) { *cap_bytes = G.replicate_bytes; return 0; }
    static size_t total_b = 0;
    if (total_b == 0) {
        size_t free_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
    }
    double frac = 0.45;
    if (const char *e = getenv("QCE_REPLICATE_FRACTION")) frac = atof(e);
    const u64 budget = (u64)(frac * (double)total_b);
    std::vector<u64> bytes(col_rows, col_rows + ncols);
    for (auto &b : bytes) b *= sizeof(u64);
    std::sort(bytes.begin(), bytes.end());
    u64 sum = 0, cap = 0;
    for (u64 b : bytes) {
        if (sum + b > budget) break;
        sum += b;
        cap = b;
    }
    // columns of one size share one fate: do not split a group at the budget's edge
    u64 group = 0;
    for (u64 b : bytes) if (b <= cap) group += b;
    while (group > budget && cap) {
        u64 next = 0;
        for (u64 b : bytes) if (b < cap) next = std::max(next, b);
        cap = next;
        group = 0;
        for (u64 b : bytes) if (b <= cap) group += b;
    }
    *cap_bytes = cap;
    return 0;
}
int qce_set_replicate_bytes(uint64_t bytes)
{
    placement_env();
    G.replicate_bytes = bytes;
    return 0;
}
/* 1: every rank holds the whole column (a query over such columns only can run on one rank
 * alone); 0: row-sharded. */
int qce_column_is_whole(uint32_t rel, uint32_t col)
{
    const Column *c;
    if (get_column(rel, col, &c) != 0) return -1;
    return c->windowed ? 0 : 1;
}
int qce_adopt_column_device(uint32_t rel, uint32_t col, const void *dev, uint64_t n)
{
    NEED_INIT();
    if (n >= (1ull << 32)) return fail("relation %u has %llu rows; device row ids are 32-bit", rel, (unsigned long long)n);
    if (((uintptr_t)dev & 15) != 0) return fail("adopted column must be 16-byte aligned");
    if (G.world > 1) return fail("adopted buffers cannot be shared between ranks: upload the column instead");
    Column c;
    bool reused;
    {
        std::lock_guard<std::mutex> lk(G.mu);
        auto it = G.cols.find(col_key(rel, col));
        if (it != G.cols.end()) { release_column(it->second); G.cols.erase(it); }
    }
    (void)reused;
    c.d = (const u64 *)dev;
    c.n = n;
    if (column_max(c.d, n, &c.maxv, &c.in_order, &c) != 0) { release_column(c); return -1; }
    install_column(rel, col, c);
    return 0;
}
int qce_adopt_column_window(uint32_t rel, uint32_t col, const void *dev, uint64_t row_begin, uint64_t row_count,
                            uint64_t rows_global, uint64_t max_value_global)
{
    NEED_INIT();
    if (rows_global >= (1ull << 32)) return fail("relation %u has %llu rows; device row ids are 32-bit", rel, (unsigned long long)rows_global);
    if (row_begin > rows_global || row_count > rows_global - row_begin) return fail("row window outside the relation");
    if (((uintptr_t)dev & 15) != 0 || (row_begin & 1)) return fail("window must be 16-byte aligned and start on an even row");
    Column c;
    c.d = (const u64 *)dev - row_begin; // virtual base: row id r of the window lives at c.d[r]
    c.n = rows_global;
    c.maxv = max_value_global;
    c.windowed = true;
    c.win_begin = row_begin;
    c.win_count = row_count;
    {
        std::lock_guard<std::mutex> lk(G.mu);
        auto it = G.cols.find(col_key(rel, col));
        if (it != G.cols.end()) { release_column(it->second); G.cols.erase(it); }
    }
    install_column(rel, col, c);
    return 0;
}
int qce_column_max_device(const void *dev, uint64_t n, uint64_t *max_value)
{
    NEED_INIT();
    if (!max_value) return fail("null argument");
    u64 m = 0;
    if (column_max((const u64 *)dev, n, &m) != 0) return -1;
    *max_value = m;
    return 0;
}
int qce_column_info(uint32_t rel, uint32_t col, uint64_t *n, uint64_t *max_value)
{
    NEED_INIT();
    const Column *c;
    if (get_column(rel, col, &c) != 0) return -1;
    if (n) *n = c->n;
    if (max_value) *max_value = c->maxv;
    return 0;
}
int qce_column_histogram(uint32_t rel, uint32_t col, uint32_t *bins, int *key_bits)
{
    NEED_INIT();
    if (!bins || !key_bits) return fail("null argument");
    const Column *c;
    if (get_column(rel, col, &c) != 0) return -1;
    *key_bits = c->hist_bits;
    if (c->hist_bits) {
        CK(cudaMemcpyAsync(bins, c->hist, QCE_RADIX_BINS * sizeof(u32), cudaMemcpyDeviceToHost, cx().stream));
        CK(cudaStreamSynchronize(cx().stream));
    }
    return 0;
}
int qce_drop_relations(void)
{
    if (!G.inited) return 0;
    cudaDeviceSynchronize(); // every context's stream
    std::lock_guard<std::mutex> lk(G.mu);
    // with several ranks this is a collective: nobody frees a window a peer still maps
    bool mapped = false;
    for (auto &kv : G.cols) {
        Column &c = kv.second;
        mapped = mapped || c.peer_mapped;
        for (void *p : c.opened) cudaIpcCloseMemHandle(p);
        c.opened.clear();
    }
    if (G.world > 1 && mapped && qcecomm::st().h && qcecomm::barrier() != 0) return fail("%s", qcecomm::st().err);
    for (auto &kv : G.cols) release_column(kv.second);
    G.cols.clear();
    return 0;
}

// ---------------------------------------------------------------- filter
static int filter_scan_window(uint32_t rel, uint32_t col, char op, uint64_t c, uint64_t begin, uint64_t count,
                              bool whole, qce_rowids **out)
{
    const Column *cl;
    int code;
    if (get_column(rel, col, &cl) != 0 || op_code(op, &code) != 0) return -1;
    if (whole) { begin = 0; count = cl->n; }
    if (begin > cl->n || count > cl->n - begin) return fail("row window [%llu, +%llu) outside relation %u (%llu rows)",
                                                           (unsigned long long)begin, (unsigned long long)count, rel,
                                                           (unsigned long long)cl->n);
    if ((begin & 1) && count) return fail("row window must start on an even row (128-bit loads)");
    if (!window_resident(cl, begin, count)) return fail("rows [%llu, +%llu) of relation %u are not resident on this rank",
                                                        (unsigned long long)begin, (unsigned long long)count, rel);
    const u64 n = count;
    if (n == 0) return new_rowids(0, (u32)cl->n, out);
    const u64 *d = cl->d + begin;
    const u64 ntiles = ceil_div(n, QCE_FTILE);
    u32 *mask = nullptr, *tile_count = nullptr;
    if (dalloc(&mask, ntiles * QCE_FWORDS) || dalloc(&tile_count, ntiles)) return -1;
    if (code == QCE_OP_EQ)
        LAUNCH("filter_scan", (k_filter_mask_base<QCE_OP_EQ>), (int)ntiles, QCE_FTHREADS, 0, d, n, c, mask, tile_count);
    else if (code == QCE_OP_GT)
        LAUNCH("filter_scan", (k_filter_mask_base<QCE_OP_GT>), (int)ntiles, QCE_FTHREADS, 0, d, n, c, mask, tile_count);
    else
        LAUNCH("filter_scan", (k_filter_mask_base<QCE_OP_LT>), (int)ntiles, QCE_FTHREADS, 0, d, n, c, mask, tile_count);
    int rc = compact_from_mask(QCE_LAYOUT_PAIR, QCE_EMIT_INDEX, mask, tile_count, ntiles, nullptr, nullptr,
                               (u32)cl->n, 0, out, nullptr, (u32)begin);
    dfree(mask);
    dfree(tile_count);
    return rc;
}

int qce_filter_scan(uint32_t rel, uint32_t col, char op, uint64_t c, qce_rowids **out)
{
    NEED_INIT();
    if (sharded()) return sh_filter_scan(rel, col, op, c, out);
    return filter_scan_window(rel, col, op, c, 0, 0, true, out);
}
int qce_filter_scan_range(uint32_t rel, uint32_t col, char op, uint64_t c, uint64_t row_begin, uint64_t row_count,
                          qce_rowids **out)
{
    NEED_INIT();
    return filter_scan_window(rel, col, op, c, row_begin, row_count, false, out);
}

int qce_filter_refine(qce_rowids *ids, uint32_t rel, uint32_t col, char op, uint64_t c, uint64_t *survivors)
{
    NEED_INIT();
    const Column *cl;
    int code;
    if (!ids) return fail("null row-id column");
    if (sharded()) return sh_filter_refine(ids, rel, col, op, c, survivors);
    if (get_column(rel, col, &cl) != 0 || op_code(op, &code) != 0) return -1;
    const u64 n = ids->n;
    if (n == 0) { if (survivors) *survivors = 0; return 0; }
    const u64 ntiles = ceil_div(n, QCE_FTILE);
    u32 *mask = nullptr, *tile_count = nullptr;
    if (dalloc(&mask, ntiles * QCE_FWORDS) || dalloc(&tile_count, ntiles)) return -1;
    if (code == QCE_OP_EQ)
        LAUNCH("filter_refine", (k_refine_mask<QCE_OP_EQ>), (int)ntiles, QCE_FTHREADS, 0, ids->d, n, ref_of(cl), c, mask, tile_count);
    else if (code == QCE_OP_GT)
        LAUNCH("filter_refine", (k_refine_mask<QCE_OP_GT>), (int)ntiles, QCE_FTHREADS, 0, ids->d, n, ref_of(cl), c, mask, tile_count);
    else
        LAUNCH("filter_refine", (k_refine_mask<QCE_OP_LT>), (int)ntiles, QCE_FTHREADS, 0, ids->d, n, ref_of(cl), c, mask, tile_count);
    qce_rowids *kept = nullptr;
    int rc = compact_from_mask(QCE_LAYOUT_NATURAL, QCE_EMIT_SRC, mask, tile_count, ntiles, ids->d, nullptr,
                               ids->id_bound, 0, &kept, nullptr);
    dfree(mask);
    dfree(tile_count);
    if (rc != 0) return -1;
    dfree(ids->d);
    ids->d = kept->d;
    ids->n = kept->n;
    delete kept;
    if (survivors) *survivors = ids->n;
    return 0;
}

// ---------------------------------------------------------------- tuples
static bool fused_build_hist()
{
    static int on = -1; // QCE_FUSED_BUILD_HIST=0: histogram in passes of their own (for comparison)
    if (on < 0) { const char *e = getenv("QCE_FUSED_BUILD_HIST"); on = e ? atoi(e) : 1; }
    return on != 0;
}
static int build_tuples(const Column *cl, const qce_rowids *ids, qce_tuples **out, u64 begin = 0,
                        u64 count = ~0ull, bool positions = false)
{
    if (count == ~0ull) count = cl->n - begin;
    if (!ids && !window_resident(cl, begin, count)) return fail("rows [%llu, +%llu) are not resident on this rank",
                                                                (unsigned long long)begin, (unsigned long long)count);
    const u64 n = ids ? ids->n : count;
    qce_tuples *t = new qce_tuples();
    t->n = n;
    t->key_bits = bitlen(cl->maxv) ? bitlen(cl->maxv) : 1;
    t->key_min = 0;
    t->key_max = cl->maxv;
    t->wide = t->key_bits > 32;
    t->id_bound = (u32)cl->n;
    t->sorted = false;
    t->ids = nullptr;
    if (dalloc(&t->a, n) != 0) { delete t; return -1; }
    if (t->wide && dalloc(&t->ids, n) != 0) { delete t; return -1; }
    if (n > 0) {
        if (t->wide)
            LAUNCH("build_tuples", k_build_wide, grid_for(256, n), 256, 0, ref_of(cl),
                   ids ? ids->d : nullptr, n, t->a, t->ids, (u32)begin);
        else {
            // large packed runs: the top-8-bit key histogram rides along (MSD level A / exchange splitters)
            const bool hist = fused_build_hist() && n >= (1ull << 20) && t->key_bits >= 9;
            const int hshift = t->key_bits - 8;
            if (hist) {
                if (dalloc(&t->hist256, QCE_RADIX_BINS) != 0) { delete t; return -1; }
                CK(cudaMemsetAsync(t->hist256, 0, QCE_RADIX_BINS * sizeof(u32), cx().stream));
                t->hist_key_bits = t->key_bits;
            }
            if (ids && positions && hist)
                LAUNCH("build_tuples", (k_build_packed_ids<true, true>), grid_for(1024, n), 256, 0, ref_of(cl), ids->d, n, t->a, hshift, t->hist256);
            else if (ids && positions)
                LAUNCH("build_tuples", (k_build_packed_ids<false, true>), grid_for(1024, n), 256, 0, ref_of(cl), ids->d, n, t->a, 0, (u32 *)nullptr);
            else if (ids && hist)
                LAUNCH("build_tuples", k_build_packed_ids<true>, grid_for(1024, n), 256, 0, ref_of(cl), ids->d, n, t->a, hshift, t->hist256);
            else if (ids)
                LAUNCH("build_tuples", k_build_packed_ids<false>, grid_for(1024, n), 256, 0, ref_of(cl), ids->d, n, t->a, 0, (u32 *)nullptr);
            else if (hist)
                LAUNCH("build_tuples", k_build_packed_base<true>, grid_for(512, n), 256, 0, cl->d + begin, n, t->a, begin, hshift, t->hist256);
            else
                LAUNCH("build_tuples", k_build_packed_base<false>, grid_for(512, n), 256, 0, cl->d + begin, n, t->a, begin, 0, (u32 *)nullptr);
        }
    }
    *out = t;
    return 0;
}
static int build_base(const Column *cl, uint32_t rel, uint32_t col, qce_tuples **out)
{
    if (build_tuples(cl, nullptr, out) != 0) return -1;
    (*out)->src_rel = rel;
    (*out)->src_col = col;
    (*out)->whole_base = true;
    (*out)->in_order = cl->in_order && !cl->windowed;
    return 0;
}
// 1: the batch's sorted-run cache holds (rel, col); *out borrows the sorted run.  0: a miss.  -1: error.
static int cached_run(uint32_t rel, uint32_t col, qce_tuples **out)
{
    if (!G.cache_on) return 0;
    std::unique_lock<std::mutex> lk(G.mu);
    auto it = G.run_cache.find(col_key(rel, col));
    if (it == G.run_cache.end()) {
        G.cache_misses++;
        return 0;
    }
    const Global::CachedRun c = it->second;
    G.cache_hits++;
    lk.unlock();
    qce_tuples *t = new qce_tuples();
    t->a = c.a; t->ids = nullptr; t->n = c.n; t->wide = false; t->key_bits = c.key_bits;
    t->key_min = c.key_min; t->key_max = c.key_max; t->id_bound = c.id_bound;
    t->sorted = true; t->borrowed = true; t->src_rel = rel; t->src_col = col; t->whole_base = true;
    t->skewed = c.skewed;
    if (cudaStreamWaitEvent(cx().stream, c.ready, 0) != cudaSuccess) { // sorted on another context's stream
        (void)cudaGetLastError();
        delete t;
        return fail("cudaStreamWaitEvent on a cached sorted run failed");
    }
    *out = t;
    return 1;
}
int qce_build_tuples_base(uint32_t rel, uint32_t col, qce_tuples **out)
{
    NEED_INIT();
    const Column *cl;
    if (sharded()) return sh_build_base(rel, col, out);
    if (get_column(rel, col, &cl) != 0) return -1;
    const int hit = cached_run(rel, col, out);
    if (hit != 0) return hit < 0 ? -1 : 0;
    return build_base(cl, rel, col, out);
}
int qce_build_tuples_base_range(uint32_t rel, uint32_t col, uint64_t row_begin, uint64_t row_count, qce_tuples **out)
{
    NEED_INIT();
    const Column *cl;
    if (get_column(rel, col, &cl) != 0) return -1;
    if (row_begin > cl->n || row_count > cl->n - row_begin) return fail("row window outside relation %u", rel);
    if ((row_begin & 1) && row_count) return fail("row window must start on an even row (128-bit loads)");
    if (build_tuples(cl, nullptr, out, row_begin, row_count) != 0) return -1;
    (*out)->src_rel = rel;
    (*out)->src_col = col;
    return 0;
}
int qce_build_tuples_rowids(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_tuples **out)
{
    NEED_INIT();
    const Column *cl;
    if (!ids) return fail("null row-id column");
    if (sharded()) return sh_build_rowids(rel, col, ids, out);
    if (get_column(rel, col, &cl) != 0) return -1;
    if (build_tuples(cl, ids, out) != 0) return -1;
    (*out)->src_rel = rel;
    (*out)->src_col = col;
    return 0;
}

/* Bystander re-join elision (SURVEY.md 8f-2; replaces join_payloads, src/join.c:426-484, inside the
 * parity-defined query class): (key = col[ids[i]], payload = i) -- the POSITION in the row-id column,
 * so that after the merge every column aligned with `ids` is re-aligned with one gather
 * (qce_rowids_gather) instead of a distinct-pair pass, two sorts and a merge per column.
 * Packed keys (< 2^32) on one rank only; -1 otherwise (the caller replays join_payloads). */
int qce_build_tuples_positions(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_tuples **out)
{
    NEED_INIT();
    const Column *cl;
    if (!ids) return fail("null row-id column");
    if (get_column(rel, col, &cl) != 0) return -1;
    if (bitlen(cl->maxv) > 32) return fail("position-carrying runs need keys below 2^32");
    if (build_tuples(cl, ids, out, 0, ~0ull, true) != 0) return -1;
    (*out)->src_rel = rel;
    (*out)->src_col = col;
    (*out)->id_bound = (u32)ids->n;
    (*out)->positions = true;
    (*out)->n_others = ids->n_others;
    (*out)->dist.kind = G.world > 1 && !cx().solo ? (int)Dist::ANY : (int)Dist::LOCAL;
    return 0;
}
/* The row-id columns aligned with a position-carrying run (the joined column itself and its
 * entity's bystanders).  One rank: nothing to do, the positions index the caller's arrays.
 * Several ranks: the columns travel with the tuples when the run is exchanged (k_push carries up
 * to QCE_PUSH_MAX_COLS), and qce_rowids_gather then reads the received copies. */
int qce_tuples_attach(qce_tuples *t, uint32_t ncols, const qce_rowids *const *cols)
{
    NEED_INIT();
    if (!t || (ncols && !cols)) return fail("null argument");
    if (!t->positions) return fail("columns attach to position-carrying runs only");
    if (ncols > QCE_PUSH_MAX_COLS) return fail("at most %d columns travel with one run", QCE_PUSH_MAX_COLS);
    t->attached.clear();
    for (u32 c = 0; c < ncols; c++) {
        if (!cols[c] || cols[c]->n < t->n) return fail("attached column %u is shorter than the run", c);
        t->attached.push_back(cols[c]);
    }
    return 0;
}
int qce_elision_supported(void)
{
    if (!G.inited && qce_init(-1) != 0) return 0;
    static int on = -1; // QCE_ELIDE=0: always replay join_payloads
    if (on < 0) { const char *e = getenv("QCE_ELIDE"); on = e ? atoi(e) : 1; }
    return on;
}
/* qce_merge_join that also reports the smallest and largest number of matches of an outer (R)
 * tuple: min == max means uniform multiplicity, under which join_payloads' positional pairing
 * cannot change a re-joined column's multiset (SURVEY.md 8c). */
int qce_merge_join_stats(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS,
                         uint32_t *min_matches, uint32_t *max_matches)
{
    NEED_INIT();
    if (!R || !S || !outR || !outS || !min_matches || !max_matches) return fail("null argument");
    if (sharded()) return sh_merge_join_stats(R, S, outR, outS, min_matches, max_matches);
    u32 st[2] = {0, 0};
    if (R->n && S->n) tl_join_stats = st;
    const int rc = merge_join_any(R, S, true, true, outR, outS);
    tl_join_stats = nullptr;
    *min_matches = st[0];
    *max_matches = st[1];
    return rc;
}

// A run that has just been sorted: its flags, and a whole base run goes to the batch's cache.
static void sorted_run_done(qce_tuples *t)
{
    t->sorted = true;
    t->skewed = tl_sort_skewed;
    if (G.cache_on && t->whole_base && !t->wide && !t->borrowed && t->n >= 1024) {
        // hand the run to the batch's cache; this handle (and later ones) borrow it
        std::lock_guard<std::mutex> lk(G.mu);
        const u64 bytes = t->n * sizeof(u64);
        if (!G.run_cache.count(col_key(t->src_rel, t->src_col)) && G.cache_bytes + bytes <= G.cache_budget) {
            Global::CachedRun c{t->a, t->n, t->key_bits, t->key_min, t->key_max, t->id_bound, nullptr, &cx().arena, t->skewed};
            if (cudaEventCreateWithFlags(&c.ready, cudaEventDisableTiming) == cudaSuccess) {
                cudaEventRecord(c.ready, cx().stream);
                G.run_cache[col_key(t->src_rel, t->src_col)] = c;
                G.cache_bytes += bytes;
                t->borrowed = true;
            } else (void)cudaGetLastError();
        }
    }
}
int qce_sort_tuples(qce_tuples *t)
{
    NEED_INIT();
    if (!t) return fail("null tuple run");
    if (sharded()) { // deferred: the join first moves every tuple to the rank that owns its key range
        t->sort_pending = true;
        return 0;
    }
    if (t->borrowed && t->sorted) return 0; // a cached sorted base run
    int rc;
    tl_sort_skewed = false;
    static int probe_on = -1; // QCE_SORT_PROBE=0: sort runs of columns that are stored in order like any other
    if (probe_on < 0) { const char *e = getenv("QCE_SORT_PROBE"); probe_on = e ? atoi(e) : 1; }
    const bool in_order = probe_on && t->in_order; // built from a whole column stored in key order: sorted as it stands
    if (in_order) {
        rc = 0;
        // the sort would have noticed a run of few distinct keys (msd_sort); here the statistics have to
        if (t->key_max < ~0ull && t->n / (t->key_max + 1) >= 16) tl_sort_skewed = true;
    } else if (t->wide) {
        RadixShifts rs = shifts_for(0, t->range_sort ? bitlen(t->key_min ^ t->key_max) : t->key_bits);
        rc = radix_sort(&t->a, &t->ids, t->n, rs);
    } else {
        // the cached histogram counts key >> (hist_key_bits - 8); level A of the MSD sort counts
        // key >> (bitlen(key_max) - 8): the same digit when the statistics are the column's own
        rc = sort_packed(&t->a, t->n, t->key_bits, t->key_min, t->key_max, t->hist256,
                         bitlen(t->key_max) == t->hist_key_bits ? t->hist_key_bits : -1);
    }
    if (rc == 0) sorted_run_done(t);
    return rc;
}

/* allocate_relation + iterative_sort of a whole base column in one: what qce_build_tuples_base followed
 * by qce_sort_tuples returns.  A column with its level-A histogram (Column::hist) whose run takes the MSD
 * route is never stored unsorted: MSD level A reads the column and forms the tuples in registers
 * (k_msd_partition_bulk<true>), which saves the build's write and level A's read of the whole run.
 * Every other run is built, then sorted.  QCE_FUSED_BUILD_SORT=0: always build, then sort. */
int qce_build_sorted_tuples_base(uint32_t rel, uint32_t col, qce_tuples **out)
{
    NEED_INIT();
    if (!out) return fail("null argument");
    static int fused_on = -1;
    if (fused_on < 0) { const char *e = getenv("QCE_FUSED_BUILD_SORT"); fused_on = e ? atoi(e) : 1; }
    qce_tuples *t = nullptr;
    if (!fused_on || sharded()) {
        if (qce_build_tuples_base(rel, col, &t) != 0) return -1;
        if (qce_sort_tuples(t) != 0) { qce_tuples_free(t); return -1; }
        *out = t;
        return 0;
    }
    const Column *cl;
    if (get_column(rel, col, &cl) != 0) return -1;
    const int hit = cached_run(rel, col, out);
    if (hit != 0) return hit < 0 ? -1 : 0;
    // the route is decided before any kernel runs, from the column's statistics alone
    MsdPlan p;
    int applies = 0;
    tl_sort_skewed = false;
    if (!cl->windowed && !cl->in_order && cl->hist_bits && cl->hist_bits == bitlen(cl->maxv)) {
        applies = msd_plan(cl->n, 0, cl->maxv, &p);
        if (applies < 0) return -1;
    }
    if (!applies) {
        if (build_base(cl, rel, col, &t) != 0) return -1;
        if (qce_sort_tuples(t) != 0) { qce_tuples_free(t); return -1; }
        *out = t;
        return 0;
    }
    t = new qce_tuples();
    t->n = cl->n;
    t->key_bits = bitlen(cl->maxv);
    t->key_min = 0;
    t->key_max = cl->maxv;
    t->wide = false;
    t->ids = nullptr;
    t->id_bound = (u32)cl->n;
    t->src_rel = rel;
    t->src_col = col;
    t->whole_base = true;
    if (dalloc(&t->a, t->n) != 0) { delete t; return -1; }
    int rc;
    {
        MsdLevels m;
        bool done = false;
        rc = msd_level_a(p, &m, cl->d, true, cl->hist);
        if (rc == 0) rc = msd_after_level_a(p, &m, &t->a, &done);
        if (rc == 0 && !done) {
            // a heavy key: the LSD passes sort level A's scatter, which holds every tuple of the run
            std::swap(t->a, m.alt);
            rc = lsd_sort_packed(&t->a, t->n, t->key_bits);
        }
    }
    if (rc != 0) { qce_tuples_free(t); return -1; }
    sorted_run_done(t);
    *out = t;
    return 0;
}

/* A batch = one execute_queries call: sorted base runs are kept between its queries and
 * dropped at its end (nothing survives into the next batch). */
int qce_batch_begin(void)
{
    NEED_INIT();
    static int on = -1; // QCE_RUN_CACHE=0 disables
    if (on < 0) { const char *e = getenv("QCE_RUN_CACHE"); on = e ? atoi(e) : 1; }
    if (!on) return 0;
    static size_t total_b = 0; // cudaMemGetInfo costs milliseconds: once
    if (total_b == 0) {
        size_t free_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
    }
    std::lock_guard<std::mutex> lk(G.mu);
    G.cache_on = true;
    G.cache_budget = total_b / 4;
    return 0;
}
int qce_batch_end(void)
{
    if (!G.inited) return 0;
    std::lock_guard<std::mutex> lk(G.mu);
    G.cache_on = false;
    if (!G.run_cache.empty()) {
        cudaDeviceSynchronize(); // every context's stream: nobody reads the runs any more
        for (auto &kv : G.run_cache) {
            kv.second.owner->free(kv.second.a);
            cudaEventDestroy(kv.second.ready);
        }
        G.run_cache.clear();
    }
    G.cache_bytes = 0;
    return 0;
}
int qce_batch_cache_stats(uint64_t *hits, uint64_t *misses)
{
    if (hits) *hits = G.cache_hits;
    if (misses) *misses = G.cache_misses;
    return 0;
}

int qce_tuples_is_sorted(const qce_tuples *t, int *sorted)
{
    NEED_INIT();
    if (!t || !sorted) return fail("null argument");
    if (sharded()) return sh_is_sorted(t, sorted);
    if (t->n < 2) { *sorted = 1; return 0; }
    u32 *flag = (u32 *)(cx().d_scalars + 9);
    CK(cudaMemsetAsync(flag, 0, sizeof(u64), cx().stream));
    if (t->wide)
        LAUNCH("is_sorted", (k_is_unsorted<true>), grid_for(256, t->n), 256, 0, view_of(t), t->n, flag);
    else
        LAUNCH("is_sorted", (k_is_unsorted<false>), grid_for(256, t->n), 256, 0, view_of(t), t->n, flag);
    CK(cudaMemcpyAsync(cx().h_scalars + 9, cx().d_scalars + 9, sizeof(u64), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    *sorted = (cx().h_scalars[9] & 0xffffffffu) ? 0 : 1;
    return 0;
}

// ---------------------------------------------------------------- joins
int qce_merge_join(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS,
                   qce_rowids **distinctR, qce_rowids **distinctS)
{
    NEED_INIT();
    if (!R || !S || !outR || !outS) return fail("null argument");
    if (sharded()) return sh_merge_join(R, S, outR, outS, distinctR, distinctS, false);
    if (merge_join_any(R, S, true, true, outR, outS) != 0) return -1;
    if (distinctR || distinctS) {
        qce_rowids *dr = nullptr, *ds = nullptr;
        if (distinct_pairs(*outR, *outS, &dr, &ds) != 0) return -1;
        if (distinctR) *distinctR = dr; else qce_rowids_free(dr);
        if (distinctS) *distinctS = ds; else qce_rowids_free(ds);
    }
    return 0;
}

int qce_merge_join_walk(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS)
{
    NEED_INIT();
    if (!R || !S || !outR || !outS) return fail("null argument");
    if (sharded()) return sh_merge_join(R, S, outR, outS, nullptr, nullptr, true);
    return merge_join_any(R, S, true, true, outR, outS, true);
}

int qce_distinct_pairs(const qce_rowids *pairsR, const qce_rowids *pairsS, qce_rowids **distinctR,
                       qce_rowids **distinctS)
{
    NEED_INIT();
    if (!pairsR || !pairsS || !distinctR || !distinctS) return fail("null argument");
    if (pairsR->n != pairsS->n) return fail("pair columns differ in length");
    if (sharded()) return sh_distinct_pairs(pairsR, pairsS, distinctR, distinctS);
    return distinct_pairs(pairsR, pairsS, distinctR, distinctS);
}

int qce_scan_join(uint32_t relR, uint32_t colR, const qce_rowids *idsR, uint32_t relS, uint32_t colS,
                  const qce_rowids *idsS, qce_rowids **outR, qce_rowids **outS)
{
    NEED_INIT();
    const Column *cr, *cs;
    if (!idsR || !idsS || !outR || !outS) return fail("null argument");
    if (get_column(relR, colR, &cr) != 0 || get_column(relS, colS, &cs) != 0) { if (sharded()) qcecomm::abort_all(); return -1; }
    if (sharded()) return sh_scan_join(cr, idsR, cs, idsS, outR, outS);
    return scan_join_impl(cr, idsR, cs, idsS, outR, outS);
}
int qce_scan_join_base(uint32_t relR, uint32_t colR, uint32_t relS, uint32_t colS, qce_rowids **outR,
                       qce_rowids **outS)
{
    NEED_INIT();
    const Column *cr, *cs;
    if (!outR || !outS) return fail("null argument");
    if (get_column(relR, colR, &cr) != 0 || get_column(relS, colS, &cs) != 0) { if (sharded()) qcecomm::abort_all(); return -1; }
    if (sharded()) return sh_scan_join_base(cr, cs, outR, outS);
    return scan_join_impl(cr, nullptr, cs, nullptr, outR, outS);
}

int qce_rejoin(const qce_rowids *driver, const qce_rowids *last, const qce_rowids *edit, qce_rowids **out)
{
    NEED_INIT();
    if (!driver || !last || !edit || !out) return fail("null argument");
    if (sharded()) return sh_rejoin(driver, last, edit, out);
    if (edit->n < last->n)
        return fail("bystander column has %llu row ids but its entity's joined column has %llu "
                    "(the reference reads past the array here, src/join.c:433)",
                    (unsigned long long)edit->n, (unsigned long long)last->n);
    const int bits = last->id_bound ? bitlen(last->id_bound - 1) : 32;
    qce_tuples R, S;
    R.n = last->n; R.key_min = 0; S.key_min = 0; R.key_max = 0; S.key_max = 0; R.hist256 = nullptr; S.hist256 = nullptr; R.wide = false; R.ids = nullptr; R.key_bits = bits ? bits : 1; R.id_bound = edit->id_bound; R.sorted = false; R.a = nullptr;
    S.n = driver->n; S.wide = false; S.ids = nullptr; S.key_bits = R.key_bits; S.id_bound = 0; S.sorted = false; S.a = nullptr;
    if (dalloc(&R.a, R.n) || dalloc(&S.a, S.n)) return -1;
    if (R.n) LAUNCH("pack_pairs", k_pack_pairs, grid_for(256, R.n), 256, 0, last->d, edit->d, R.n, R.a);
    if (S.n) LAUNCH("pack_pairs", k_pack_pairs, grid_for(256, S.n), 256, 0, driver->d, (const u32 *)nullptr, S.n, S.a);
    const u64 id_max = last->id_bound ? last->id_bound - 1 : 0;
    if (sort_packed(&R.a, R.n, R.key_bits, 0, id_max) != 0 || sort_packed(&S.a, S.n, S.key_bits, 0, id_max) != 0) return -1;
    int rc = merge_join_any(&R, &S, true, false, out, nullptr);
    dfree(R.a);
    dfree(S.a);
    return rc;
}

// ---------------------------------------------------------------- projection
int qce_checksum(const qce_rowids *ids, uint32_t rel, const uint32_t *cols, uint32_t ncols, uint64_t *sums)
{
    NEED_INIT();
    if (!ids || !cols || !sums) return fail("null argument");
    if (ncols == 0) return 0;
    if (ncols > 8) return fail("at most 8 columns per checksum call");
    if (sharded()) return sh_checksum(ids, rel, cols, ncols, sums);
    ChecksumCols cc;
    u64 col_rows = 0;
    for (u32 k = 0; k < 8; k++) cc.col[k] = nullptr;
    for (u32 k = 0; k < ncols; k++) {
        const Column *cl;
        if (get_column(rel, cols[k], &cl) != 0) return -1;
        cc.col[k] = cl->d;
        col_rows = cl->n;
    }
    CK(cudaMemsetAsync(cx().d_scalars, 0, 8 * sizeof(u64), cx().stream));
    if (ids->n > 0) {
        // A large row-id column in arbitrary order makes every gather a DRAM miss
        // that moves ~77 B for 8 useful bytes (ncu, profiles/).  The sum does not
        // depend on the order, so the ids are first partitioned by their top 8
        // bits (one one-sweep pass over 4-byte keys): the gathers then walk the
        // column region by region and are served from L2.
        const u32 *src = ids->d;
        u32 *bucketed = nullptr;
        if (!ids->bucketed && bucketed_checksum_pays(ids, col_rows)) {
            if (partition_ids_by_top_bits(ids, &bucketed) != 0) return -1;
            src = bucketed;
        }
        static int waves = -1, per_col = -1; // QCE_CHECKSUM_WAVES / QCE_CHECKSUM_PER_COL: experiment switches
        if (waves < 0) { const char *e = getenv("QCE_CHECKSUM_WAVES"); waves = e ? atoi(e) : 0; if (waves < 0) waves = 0; }
        if (per_col < 0) { const char *e = getenv("QCE_CHECKSUM_PER_COL"); per_col = e ? atoi(e) : 0; }
        // Bucketed ids sweep the column region by region; the regions in flight must stay in L2.  With 8 waves
        // of CTAs the front spans ~6 regions x NC columns and thrashes (ncu: 5.3 GB read for the 1.8 GB two
        // columns + ids need, 0.86 ms); 3 waves keep it to ~2 regions: 0.33 ms (sweep in profiles/).
        // Unbucketed ids gather at random anyway and want the parallelism.
        const bool swept = bucketed != nullptr || ids->bucketed;
        const int grid = grid_for(1024, ids->n, waves ? waves : (swept ? 3 : 8));
        if (per_col && ncols > 1) {
            // one pass over the (bucketed) ids per column: half the working set in L2 at any time
            for (u32 k = 0; k < ncols; k++) {
                ChecksumCols one;
                for (u32 j = 0; j < 8; j++) one.col[j] = nullptr;
                one.col[0] = cc.col[k];
                LAUNCH("checksum", (k_checksum<1>), grid, 256, 0, src, ids->n, one, cx().d_scalars + k);
            }
        } else
        switch (ncols) {
        case 1: LAUNCH("checksum", (k_checksum<1>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        case 2: LAUNCH("checksum", (k_checksum<2>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        case 3: LAUNCH("checksum", (k_checksum<3>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        case 4: LAUNCH("checksum", (k_checksum<4>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        case 5: LAUNCH("checksum", (k_checksum<5>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        case 6: LAUNCH("checksum", (k_checksum<6>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        case 7: LAUNCH("checksum", (k_checksum<7>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        default: LAUNCH("checksum", (k_checksum<8>), grid, 256, 0, src, ids->n, cc, cx().d_scalars); break;
        }
        dfree(bucketed);
    }
    if (read_scalars((int)ncols) != 0) return -1;
    for (u32 k = 0; k < ncols; k++) sums[k] = cx().h_scalars[k];
    return 0;
}

// ---------------------------------------------------------------- handles
uint64_t qce_rowids_count(const qce_rowids *ids) { return ids ? ids->n + ids->n_others : 0; }
/* this rank's share only (== qce_rowids_count on one GPU) */
uint64_t qce_rowids_count_local(const qce_rowids *ids) { return ids ? ids->n : 0; }

int qce_rowids_from_host(const uint64_t *host, uint64_t n, qce_rowids **out)
{
    NEED_INIT();
    std::vector<u32> tmp(n ? n : 1);
    u32 mx = 0;
    for (u64 i = 0; i < n; i++) {
        if (host[i] >= (1ull << 32)) return fail("row id %llu does not fit 32 bits", (unsigned long long)host[i]);
        tmp[i] = (u32)host[i];
        if (tmp[i] > mx) mx = tmp[i];
    }
    if (new_rowids(n, n ? (mx == 0xffffffffu ? 0 : mx + 1) : 0, out) != 0) return -1;
    if (n) CK(cudaMemcpyAsync((*out)->d, tmp.data(), n * sizeof(u32), cudaMemcpyHostToDevice, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    return 0;
}
int qce_rowids_to_host(const qce_rowids *ids, uint64_t *host)
{
    NEED_INIT();
    if (!ids) return fail("null row-id column");
    std::vector<u32> tmp(ids->n ? ids->n : 1);
    if (ids->n) CK(cudaMemcpyAsync(tmp.data(), ids->d, ids->n * sizeof(u32), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    for (u64 i = 0; i < ids->n; i++) host[i] = tmp[i];
    return 0;
}
int qce_rowids_clone(const qce_rowids *ids, qce_rowids **out)
{
    NEED_INIT();
    if (!ids) return fail("null row-id column");
    if (new_rowids(ids->n, ids->id_bound, out) != 0) return -1;
    if (ids->n) CK(cudaMemcpyAsync((*out)->d, ids->d, ids->n * sizeof(u32), cudaMemcpyDeviceToDevice, cx().stream));
    (*out)->n_others = ids->n_others;
    (*out)->dist = ids->dist;
    return 0;
}
void qce_rowids_free(qce_rowids *ids)
{
    if (!ids) return;
    if (G.inited) dfree(ids->d);
    delete ids;
}

uint64_t qce_tuples_count(const qce_tuples *t) { return t ? t->n + t->n_others : 0; }

int qce_tuples_from_host(const uint64_t *keys, const uint64_t *rowids, uint64_t n, qce_tuples **out)
{
    NEED_INIT();
    u64 mk = 0, mi = 0;
    for (u64 i = 0; i < n; i++) {
        if (keys[i] > mk) mk = keys[i];
        if (rowids[i] > mi) mi = rowids[i];
    }
    if (mi >= (1ull << 32)) return fail("row id %llu does not fit 32 bits", (unsigned long long)mi);
    qce_tuples *t = new qce_tuples();
    t->n = n;
    t->key_bits = bitlen(mk) ? bitlen(mk) : 1;
    t->key_min = 0;
    t->key_max = mk;
    t->wide = t->key_bits > 32;
    t->id_bound = (mi + 1 >= (1ull << 32)) ? 0 : (u32)(mi + 1);
    t->sorted = false;
    t->ids = nullptr;
    if (dalloc(&t->a, n) != 0) { delete t; return -1; }
    if (t->wide) {
        if (dalloc(&t->ids, n) != 0) { delete t; return -1; }
        std::vector<u32> tmp(n ? n : 1);
        for (u64 i = 0; i < n; i++) tmp[i] = (u32)rowids[i];
        if (n) {
            CK(cudaMemcpyAsync(t->a, keys, n * sizeof(u64), cudaMemcpyHostToDevice, cx().stream));
            CK(cudaMemcpyAsync(t->ids, tmp.data(), n * sizeof(u32), cudaMemcpyHostToDevice, cx().stream));
        }
        CK(cudaStreamSynchronize(cx().stream));
    } else {
        std::vector<u64> tmp(n ? n : 1);
        for (u64 i = 0; i < n; i++) tmp[i] = (keys[i] << 32) | rowids[i];
        if (n) CK(cudaMemcpyAsync(t->a, tmp.data(), n * sizeof(u64), cudaMemcpyHostToDevice, cx().stream));
        CK(cudaStreamSynchronize(cx().stream));
    }
    *out = t;
    return 0;
}
int qce_tuples_to_host(const qce_tuples *t, uint64_t *keys, uint64_t *rowids)
{
    NEED_INIT();
    if (!t) return fail("null tuple run");
    const u64 n = t->n;
    if (t->wide) {
        std::vector<u32> tmp(n ? n : 1);
        if (n) {
            CK(cudaMemcpyAsync(keys, t->a, n * sizeof(u64), cudaMemcpyDeviceToHost, cx().stream));
            CK(cudaMemcpyAsync(tmp.data(), t->ids, n * sizeof(u32), cudaMemcpyDeviceToHost, cx().stream));
        }
        CK(cudaStreamSynchronize(cx().stream));
        for (u64 i = 0; i < n; i++) rowids[i] = tmp[i];
    } else {
        std::vector<u64> tmp(n ? n : 1);
        if (n) CK(cudaMemcpyAsync(tmp.data(), t->a, n * sizeof(u64), cudaMemcpyDeviceToHost, cx().stream));
        CK(cudaStreamSynchronize(cx().stream));
        for (u64 i = 0; i < n; i++) { keys[i] = tmp[i] >> 32; rowids[i] = tmp[i] & 0xffffffffu; }
    }
    return 0;
}
void qce_tuples_free(qce_tuples *t)
{
    if (!t) return;
    if (G.inited) { if (!t->borrowed) dfree(t->a); dfree(t->ids); dfree(t->hist256); }
    delete t;
}

// ---------------------------------------------------------------- exchange
int qce_key_histogram(const qce_tuples *t, uint32_t key_bits, uint64_t *hist)
{
    NEED_INIT();
    if (!t || !hist) return fail("null argument");
    if (t->wide) return fail("the sharded exchange supports packed (key < 2^32) runs only");
    qce_tuples *mt = const_cast<qce_tuples *>(t); // the device histogram is cached on the run
    const bool have = mt->hist256 && mt->hist_key_bits == (int)key_bits && key_bits >= 9 && !t->sorted; // from the build kernel
    if (!mt->hist256 && dalloc(&mt->hist256, QCE_RADIX_BINS) != 0) return -1;
    u32 *gh = mt->hist256;
    if (!have) {
        CK(cudaMemsetAsync(gh, 0, QCE_RADIX_BINS * sizeof(u32), cx().stream));
        RadixShifts rs;
        rs.npass = 1;
        for (int i = 0; i < QCE_MAX_PASSES; i++) rs.shift[i] = 0;
        rs.shift[0] = 32 + (key_bits > 8 ? (int)key_bits - 8 : 0);
        if (t->n) LAUNCH("radix_hist", k_radix_hist, grid_for(1024, t->n, 4), 512, 0, t->a, t->n, rs, 256u, gh);
    }
    std::vector<u32> tmp(QCE_RADIX_BINS);
    CK(cudaMemcpyAsync(tmp.data(), gh, QCE_RADIX_BINS * sizeof(u32), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    for (int i = 0; i < QCE_RADIX_BINS; i++) hist[i] = tmp[i];
    mt->hist_key_bits = (int)key_bits;
    mt->hist_host.assign(tmp.begin(), tmp.end());
    return 0;
}
int qce_key_histogram_wide(const qce_tuples *t, uint64_t base, uint32_t width, uint64_t *hist)
{
    NEED_INIT();
    if (!t || !hist) return fail("null argument");
    if (!t->wide && t->n) return fail("qce_key_histogram_wide takes wide runs (packed runs: qce_key_histogram)");
    if (width == 0 || width > 64) return fail("key width must be 1..64");
    qce_tuples *mt = const_cast<qce_tuples *>(t); // cached on the run like the packed histogram
    if (!mt->hist256 && dalloc(&mt->hist256, QCE_RADIX_BINS) != 0) return -1;
    u32 *gh = mt->hist256;
    CK(cudaMemsetAsync(gh, 0, QCE_RADIX_BINS * sizeof(u32), cx().stream));
    const int shift = width > 8 ? (int)width - 8 : 0;
    if (t->n) LAUNCH("hist_wide", k_hist_wide, grid_for(2048, t->n, 4), 512, 0, (const u64 *)t->a, t->n, (u64)base, shift, gh);
    std::vector<u32> tmp(QCE_RADIX_BINS);
    CK(cudaMemcpyAsync(tmp.data(), gh, QCE_RADIX_BINS * sizeof(u32), cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    for (int i = 0; i < QCE_RADIX_BINS; i++) hist[i] = tmp[i];
    mt->hist_key_bits = (int)width;
    mt->hist_base = base;
    mt->hist_host.assign(tmp.begin(), tmp.end());
    return 0;
}

int qce_partition_tuples(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                         uint64_t *counts, void **sendbuf)
{
    NEED_INIT();
    if (!t || !counts || !sendbuf) return fail("null argument");
    if (t->wide) return fail("the sharded exchange supports packed (key < 2^32) runs only");
    if (nparts < 1 || nparts > 256) return fail("nparts must be in 1..256");
    if (key_bits == 0 || key_bits > 32) return fail("packed runs carry keys of 1..32 bits");
    if (t->n >= (1ull << 30)) return fail("partition of %llu tuples exceeds the 2^30 per-run limit", (unsigned long long)t->n);
    const int bin_shift = key_bits > 8 ? (int)key_bits - 8 : 0;
    DigitSplit ds;
    ds.shift = 32 + bin_shift;
    unsigned char lut[256];
    for (u32 b = 0; b < 256; b++) {
        u32 part = 0;
        for (u32 k = 0; k + 1 < nparts; k++) {
            if ((splitters[k] & ((1ull << bin_shift) - 1)) != 0)
                return fail("splitter %llu is not on a boundary of the top-8-bit histogram bins", (unsigned long long)splitters[k]);
            if (((u64)b << bin_shift) >= splitters[k]) part++;
        }
        lut[b] = (unsigned char)part;
    }
    const u64 n = t->n;
    u64 *out = nullptr;
    u32 *dlut = nullptr, *lvl0 = nullptr, *cursor = nullptr;
    if (dalloc(&out, n) || dalloc(&dlut, 64) || dalloc(&lvl0, 4) || dalloc(&cursor, QCE_RADIX_BINS)) return -1;
    // per-destination counts = the 256-bin key histogram folded through the table.  The
    // histogram is the one qce_key_histogram left on the run (splitter selection needs it anyway).
    std::vector<u32> bins(QCE_RADIX_BINS, 0), parts(QCE_RADIX_BINS, 0), offs(QCE_RADIX_BINS, 0);
    if (n) {
        if (!(t->hist256 && t->hist_key_bits == (int)key_bits && t->hist_host.size() == QCE_RADIX_BINS)) {
            uint64_t h[QCE_RADIX_BINS];
            if (qce_key_histogram(t, key_bits, h) != 0) return -1;
        }
        for (u32 b = 0; b < 256; b++) parts[lut[b]] += t->hist_host[b];
        for (u32 p = 1; p < 256; p++) offs[p] = offs[p - 1] + parts[p - 1];
        const u32 ntiles = (u32)ceil_div(n, QCE_MSD_TILE);
        const u32 h_lvl0[4] = {0u, ntiles, 0u, (u32)n};
        CK(cudaMemcpyAsync(lvl0, h_lvl0, sizeof h_lvl0, cudaMemcpyHostToDevice, cx().stream));
        CK(cudaMemcpyAsync(dlut, lut, sizeof lut, cudaMemcpyHostToDevice, cx().stream));
        CK(cudaMemcpyAsync(cursor, offs.data(), QCE_RADIX_BINS * sizeof(u32), cudaMemcpyHostToDevice, cx().stream));
        // the unstable MSD partition kernel with the destination table as digit: no ranking
        // ballots, no look-back (the order inside a destination does not matter, it is sorted next)
        LAUNCH("exchange_partition", (k_msd_partition<512, 8>), ntiles, 512, 0, (const u64 *)t->a, out, lvl0, lvl0 + 2,
               lvl0 + 3, 1u, 0ull, ds.shift, 256u, cursor, (const u32 *)dlut);
        CK(cudaStreamSynchronize(cx().stream)); // the caller hands *sendbuf to another stream
    }
    for (u32 p = 0; p < nparts; p++) counts[p] = parts[p];
    dfree(dlut); dfree(lvl0); dfree(cursor);
    *sendbuf = out;
    return 0;
}
int qce_exchange_release(void *sendbuf)
{
    NEED_INIT();
    dfree((u64 *)sendbuf);
    return 0;
}
static int tuples_from_device(const void *dev_words, uint64_t n, uint32_t key_bits, uint32_t id_bound, uint64_t key_lo,
                              uint64_t key_hi, bool adopt, qce_tuples **out);
int qce_tuples_from_device_packed(const void *dev_words, uint64_t n, uint32_t key_bits, uint32_t id_bound,
                                  uint64_t key_lo, uint64_t key_hi, qce_tuples **out)
{
    return tuples_from_device(dev_words, n, key_bits, id_bound, key_lo, key_hi, false, out);
}
int qce_tuples_adopt_device_packed(void *dev_words, uint64_t n, uint32_t key_bits, uint32_t id_bound, uint64_t key_lo,
                                   uint64_t key_hi, qce_tuples **out)
{
    return tuples_from_device(dev_words, n, key_bits, id_bound, key_lo, key_hi, true, out);
}
static int tuples_from_device(const void *dev_words, uint64_t n, uint32_t key_bits, uint32_t id_bound, uint64_t key_lo,
                              uint64_t key_hi, bool adopt, qce_tuples **out)
{
    NEED_INIT();
    if (!out) return fail("null argument");
    if (key_bits == 0 || key_bits > 32) return fail("packed runs carry keys of 1..32 bits");
    qce_tuples *t = new qce_tuples();
    t->n = n;
    t->key_bits = (int)key_bits;
    t->key_min = key_lo;
    t->key_max = key_hi; // 0 = unknown: the sort assumes the whole 2^key_bits range
    t->wide = false;
    t->id_bound = id_bound;
    t->sorted = false;
    t->ids = nullptr;
    if (adopt) {
        // no copy: the run lives in the caller's buffer (it must stay alive and must be
        // complete, i.e. the caller has synchronised the stream that filled it).  The arena
        // ignores pointers it did not hand out, so freeing the run leaves the buffer alone.
        if (n && ((uintptr_t)dev_words & 15) != 0) { delete t; return fail("adopted buffer must be 16-byte aligned"); }
        t->a = (u64 *)dev_words;
        if (n == 0 && dalloc(&t->a, 1) != 0) { delete t; return -1; }
    } else {
        if (dalloc(&t->a, n) != 0) { delete t; return -1; }
        // the caller's buffer may live on another stream (torch): order by a full device sync
        CK(cudaDeviceSynchronize());
        if (n) CK(cudaMemcpyAsync(t->a, dev_words, n * sizeof(u64), cudaMemcpyDeviceToDevice, cx().stream));
    }
    *out = t;
    return 0;
}

// ------------------------------------------------- peer-memory exchange (NVLink)
// One receive window per rank (plain cudaMalloc so that it can be exported with
// CUDA IPC); the peers map it once.  The orchestrator carves regions out of the
// window deterministically from the all-gathered histograms, so no offsets are
// ever communicated per transfer.
int qce_xwin_create(uint64_t bytes, unsigned char *ipc_handle_out)
{
    NEED_INIT();
    if (G.xwin) return fail("exchange window already exists");
    if (bytes == 0) return fail("empty exchange window");
    bytes = (bytes + 4095) / 4096 * 4096;
    void *p = nullptr;
    CK(cudaMalloc(&p, bytes));
    G.xwin = (unsigned char *)p;
    G.xwin_bytes = bytes;
    G.xworld = 1;
    G.xrank = 0;
    for (int r = 0; r < QCE_MAX_RANKS; r++) G.peers.base[r] = nullptr;
    G.peers.base[0] = G.xwin;
    if (ipc_handle_out) {
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, p));
        static_assert(sizeof(h) == 64, "IPC handle size");
        memcpy(ipc_handle_out, &h, sizeof h);
    }
    return 0;
}
int qce_xwin_attach(uint32_t world, uint32_t rank, const unsigned char *handles)
{
    NEED_INIT();
    if (!G.xwin) return fail("create the exchange window first");
    if (world < 1 || world > QCE_MAX_RANKS || rank >= world) return fail("world size must be 1..%d", QCE_MAX_RANKS);
    if (world > 1 && !handles) return fail("null argument");
    for (int r = 0; r < QCE_MAX_RANKS; r++) G.peers.base[r] = nullptr;
    for (u32 r = 0; r < world; r++) {
        if (r == rank) { G.peers.base[r] = G.xwin; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + 64 * (size_t)r, sizeof h);
        void *p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        G.xopened.push_back(p);
        G.peers.base[r] = (unsigned char *)p;
    }
    G.xworld = world;
    G.xrank = rank;
    return 0;
}
// Single-process testing: present this rank's window as `world` ranks, rank r
// owning the bytes from r * (window / world) on.
int qce_xwin_loopback(uint32_t world)
{
    NEED_INIT();
    if (!G.xwin) return fail("create the exchange window first");
    if (world < 1 || world > QCE_MAX_RANKS) return fail("world size must be 1..%d", QCE_MAX_RANKS);
    const u64 per = G.xwin_bytes / world / 4096 * 4096;
    for (int r = 0; r < QCE_MAX_RANKS; r++) G.peers.base[r] = (u32)r < world ? G.xwin + per * r : nullptr;
    G.xworld = world;
    G.xrank = 0;
    return 0;
}
int qce_xwin_info(uint64_t *bytes, void **local_base)
{
    NEED_INIT();
    if (bytes) *bytes = G.xwin_bytes;
    if (local_base) *local_base = G.xwin;
    return 0;
}
static void xwin_close_peers()
{
    for (void *p : G.xopened) cudaIpcCloseMemHandle(p);
    G.xopened.clear();
}
int qce_xwin_destroy(void)
{
    if (!G.inited) return 0;
    cudaStreamSynchronize(cx().stream);
    xwin_close_peers();
    if (G.xwin) cudaFree(G.xwin);
    G.xwin = nullptr;
    G.xwin_bytes = 0;
    G.xworld = 0;
    return 0;
}
/* the ranks' half of a collective re-creation: nobody frees a window a peer still maps */
int qce_xwin_unmap_peers(void)
{
    if (!G.inited) return 0;
    CK(cudaStreamSynchronize(cx().stream));
    xwin_close_peers();
    return 0;
}

static int push_scratch(u32 ndigits, const uint64_t *seg_start, const u32 *run_base, unsigned long long **d_seg,
                        u32 **d_run, unsigned long long **d_cur)
{
    // seg_start | cursor (same values) | run_base, one small upload each
    if (dalloc(d_seg, 256) || dalloc(d_cur, 256) || dalloc(d_run, 256)) return -1;
    std::vector<unsigned long long> seg(256, 0);
    std::vector<u32> run(256, 0);
    for (u32 d = 0; d < ndigits; d++) { seg[d] = seg_start[d]; run[d] = run_base ? run_base[d] : 0u; }
    CK(cudaMemcpyAsync(*d_seg, seg.data(), 256 * sizeof(unsigned long long), cudaMemcpyHostToDevice, cx().stream));
    CK(cudaMemcpyAsync(*d_cur, seg.data(), 256 * sizeof(unsigned long long), cudaMemcpyHostToDevice, cx().stream));
    CK(cudaMemcpyAsync(*d_run, run.data(), 256 * sizeof(u32), cudaMemcpyHostToDevice, cx().stream));
    return 0;
}

// destination rank of each histogram bin: the number of splitters at or below the bin's first key
static int push_lut(const uint64_t *splitters, uint32_t nparts, int shift, unsigned char *lut)
{
    for (u32 k = 0; k + 1 < nparts; k++)
        if (!on_bin_boundary(splitters[k], shift))
            return fail("splitter %llu is not on a boundary of the top-8-bit histogram bins", (unsigned long long)splitters[k]);
    for (u32 b = 0; b < 256; b++) {
        u32 part = 0;
        for (u32 k = 0; k + 1 < nparts; k++) part += b >= cut_bin(splitters[k], shift);
        lut[b] = (unsigned char)part;
    }
    return 0;
}
// the bytes of a destination's window a push may fill
static u64 dst_window_bytes()
{
    const bool loopback = G.xworld > 1 && G.peers.base[0] && G.peers.base[1] && G.peers.base[1] > G.peers.base[0] &&
                          (u64)(G.peers.base[1] - G.peers.base[0]) < G.xwin_bytes;
    return loopback ? (u64)(G.peers.base[1] - G.peers.base[0]) : G.xwin_bytes; // loopback: each fake rank owns a slice
}

static int push_tuples_impl(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                            const uint64_t *dst_word_offset, const uint32_t *dst_run_index, qce_rowids **slots_out,
                            uint32_t ncols, const qce_rowids *const *cols, const uint64_t *col_u32_offset);
int qce_push_tuples(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                    const uint64_t *dst_word_offset, const uint32_t *dst_run_index, qce_rowids **slots_out)
{
    return push_tuples_impl(t, key_bits, splitters, nparts, dst_word_offset, dst_run_index, slots_out, 0, nullptr, nullptr);
}
int qce_push_tuples_cols(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                         const uint64_t *dst_word_offset, const uint32_t *dst_run_index, uint32_t ncols,
                         const qce_rowids *const *cols, const uint64_t *col_u32_offset)
{
    if (ncols && (!cols || !col_u32_offset || !dst_run_index)) return fail("null argument");
    if (ncols > QCE_PUSH_MAX_COLS) return fail("at most %d columns travel with one run", QCE_PUSH_MAX_COLS);
    return push_tuples_impl(t, key_bits, splitters, nparts, dst_word_offset, dst_run_index, nullptr, ncols, cols, col_u32_offset);
}
static int push_tuples_impl(const qce_tuples *t, uint32_t key_bits, const uint64_t *splitters, uint32_t nparts,
                            const uint64_t *dst_word_offset, const uint32_t *dst_run_index, qce_rowids **slots_out,
                            uint32_t ncols, const qce_rowids *const *cols, const uint64_t *col_u32_offset)
{
    NEED_INIT();
    if (!t || !dst_word_offset) return fail("null argument");
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    if (t->wide) return fail("the sharded exchange supports packed (key < 2^32) runs only");
    if (nparts != G.xworld) return fail("nparts (%u) differs from the attached world size (%u)", nparts, G.xworld);
    if (key_bits == 0 || key_bits > 32) return fail("packed runs carry keys of 1..32 bits");
    // slots carry (destination << 28 | position): 2^28 tuples per run; a plain push only needs 32-bit tile offsets
    if (t->n >= ((slots_out || dst_run_index) ? (1ull << 28) : (1ull << 32) - 4096))
        return fail("push of %llu tuples exceeds the per-run limit", (unsigned long long)t->n);
    if (nparts > 1 && !splitters) return fail("null argument");
    const int bin_shift = key_bits > 8 ? (int)key_bits - 8 : 0;
    unsigned char lut[256];
    if (push_lut(splitters, nparts, bin_shift, lut) != 0) return -1;
    // a wrong plan must not scribble over a peer's memory: with the run's histogram at hand (the exchange
    // always has it) every destination segment is checked against the window before anything is stored
    if (t->hist_key_bits == (int)key_bits && t->hist_host.size() == QCE_RADIX_BINS) {
        u64 per_dst[QCE_MAX_RANKS] = {0};
        for (u32 b = 0; b < 256; b++) per_dst[lut[b]] += t->hist_host[b];
        const u64 window_words = dst_window_bytes() / 8;
        for (u32 p = 0; p < nparts; p++)
            if (per_dst[p] && dst_word_offset[p] + per_dst[p] > window_words)
                return fail("push would overrun rank %u's window: words [%llu, +%llu) of %llu", p,
                            (unsigned long long)dst_word_offset[p], (unsigned long long)per_dst[p], (unsigned long long)window_words);
    }
    if (slots_out && new_rowids(t->n, 0, slots_out) != 0) return -1;
    if (t->n == 0) return 0;
    unsigned long long *d_seg = nullptr, *d_cur = nullptr;
    u32 *d_run = nullptr, *dlut = nullptr;
    if (push_scratch(nparts, dst_word_offset, dst_run_index, &d_seg, &d_run, &d_cur) != 0 || dalloc(&dlut, 64)) return -1;
    CK(cudaMemcpyAsync(dlut, lut, sizeof lut, cudaMemcpyHostToDevice, cx().stream));
    PushDigit<u64> dg;
    dg.shift = 32 + bin_shift;
    dg.lut = dlut;
    PushPlan plan{d_seg, d_run, d_cur, nparts, 1u};
    const u32 n = (u32)t->n, grid = (u32)ceil_div(n, PushTile<u64>::TILE);
    const int dbits = bitlen(nparts - 1);
    u32 *so = slots_out ? (*slots_out)->d : nullptr;
    PushCols pc;
    memset(&pc, 0, sizeof pc);
    pc.n = (int)ncols;
    for (u32 c = 0; c < ncols; c++) {
        if (!cols[c] || cols[c]->n != t->n) return fail("column %u travels with a run of different length", c);
        pc.in[c] = cols[c]->d;
        for (u32 r = 0; r < nparts; r++) pc.region[c][r] = col_u32_offset[(size_t)c * nparts + r];
    }
    if (dst_run_index)
        LAUNCH("push_tuples", (k_push<u64, true, true>), grid, QCE_PUSH_THREADS, 0, (const u64 *)t->a, n, dg, plan, G.peers, dbits, so, pc);
    else
        LAUNCH("push_tuples", (k_push<u64, true, false>), grid, QCE_PUSH_THREADS, 0, (const u64 *)t->a, n, dg, plan, G.peers, dbits, so, pc);
    dfree_after_push(d_seg); dfree_after_push(d_cur); dfree_after_push(d_run); dfree_after_push(dlut);
    return 0;
}

int qce_push_tuples_wide(const qce_tuples *t, uint64_t base, uint32_t width, const uint64_t *splitters, uint32_t nparts,
                         const uint64_t *dst_word_offset, const uint64_t *dst_id_offset)
{
    NEED_INIT();
    if (!t || !dst_word_offset || !dst_id_offset) return fail("null argument");
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    if (!t->wide && t->n) return fail("qce_push_tuples_wide takes wide runs (packed runs: qce_push_tuples)");
    if (nparts != G.xworld) return fail("nparts (%u) differs from the attached world size (%u)", nparts, G.xworld);
    if (width == 0 || width > 64) return fail("key width must be 1..64");
    if (t->n >= (1ull << 32) - 4096) return fail("push of %llu tuples exceeds the per-run limit", (unsigned long long)t->n);
    if (nparts > 1 && !splitters) return fail("null argument");
    const int shift = width > 8 ? (int)width - 8 : 0;
    unsigned char lut[256];
    if (push_lut(splitters, nparts, shift, lut) != 0) return -1;
    if (t->hist_key_bits == (int)width && t->hist_base == base && t->hist_host.size() == QCE_RADIX_BINS) {
        u64 per_dst[QCE_MAX_RANKS] = {0};
        for (u32 b = 0; b < 256; b++) per_dst[lut[b]] += t->hist_host[b];
        const u64 bytes = dst_window_bytes();
        for (u32 p = 0; p < nparts; p++)
            if (per_dst[p] && ((dst_word_offset[p] + per_dst[p]) * 8 > bytes || (dst_id_offset[p] + per_dst[p]) * 4 > bytes))
                return fail("push would overrun rank %u's window: key words [%llu, +%llu), ids [%llu, +%llu) of %llu bytes", p,
                            (unsigned long long)dst_word_offset[p], (unsigned long long)per_dst[p],
                            (unsigned long long)dst_id_offset[p], (unsigned long long)per_dst[p], (unsigned long long)bytes);
    }
    if (t->n == 0) return 0;
    unsigned long long *d_seg = nullptr, *d_cur = nullptr;
    u32 *d_run = nullptr, *dlut = nullptr;
    if (push_scratch(nparts, dst_word_offset, nullptr, &d_seg, &d_run, &d_cur) != 0 || dalloc(&dlut, 64)) return -1;
    CK(cudaMemcpyAsync(dlut, lut, sizeof lut, cudaMemcpyHostToDevice, cx().stream));
    PushDigitWide dg;
    dg.base = base;
    dg.shift = shift;
    dg.lut = dlut;
    WideIdRegions idr;
    memset(&idr, 0, sizeof idr);
    for (u32 p = 0; p < nparts; p++) idr.id_delta[p] = dst_id_offset[p] - dst_word_offset[p];
    PushPlan plan{d_seg, d_run, d_cur, nparts, 1u};
    const u32 n = (u32)t->n, grid = (u32)ceil_div(n, PushTile<u64>::TILE);
    LAUNCH("push_wide", k_push_wide, grid, QCE_PUSH_THREADS, 0, (const u64 *)t->a, (const u32 *)t->ids, n, dg, plan, G.peers,
           bitlen(nparts - 1), idr);
    dfree_after_push(d_seg); dfree_after_push(d_cur); dfree_after_push(d_run); dfree_after_push(dlut);
    return 0;
}

int qce_push_u32_by_slot(const qce_rowids *vals, const qce_rowids *slots, uint32_t nparts, const uint64_t *dst_u32_offset)
{
    NEED_INIT();
    if (!vals || !slots || !dst_u32_offset) return fail("null argument");
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    if (vals->n != slots->n) return fail("column (%llu) and slot (%llu) lengths differ", (unsigned long long)vals->n, (unsigned long long)slots->n);
    if (nparts != G.xworld) return fail("nparts (%u) differs from the attached world size (%u)", nparts, G.xworld);
    if (vals->n == 0) return 0;
    SlotRegions reg;
    for (u32 r = 0; r < QCE_MAX_RANKS; r++) reg.region[r] = r < nparts ? dst_u32_offset[r] : 0;
    LAUNCH("push_by_slot", k_push_u32_by_slot, grid_for(2048, vals->n), 256, 0, vals->d, slots->d, vals->n, reg, G.peers);
    return 0;
}

static int row_bins(uint32_t rows_per_rank, uint32_t bin_width, uint32_t bins_per_rank, uint32_t nranks, RowBins *rb)
{
    if (rows_per_rank == 0 || bin_width == 0 || bins_per_rank == 0 || nranks == 0 || (u64)bins_per_rank * nranks > 256)
        return fail("row bins: rows_per_rank, bin_width > 0 and bins_per_rank * nranks in 1..256");
    rb->rows_per_rank = rows_per_rank;
    rb->inv_rows = 1.0f / (float)rows_per_rank;
    rb->last_rank = nranks - 1;
    rb->width = bin_width;
    rb->bins_per_rank = bins_per_rank;
    return 0;
}
int qce_rowids_bin_histogram(const qce_rowids *ids, uint32_t rows_per_rank, uint32_t bin_width, uint32_t bins_per_rank,
                             uint32_t nranks, uint64_t *hist)
{
    NEED_INIT();
    if (!ids || !hist) return fail("null argument");
    RowBins rb;
    if (row_bins(rows_per_rank, bin_width, bins_per_rank, nranks, &rb) != 0) return -1;
    u32 *gh = nullptr;
    if (dalloc(&gh, 256) != 0) return -1;
    CK(cudaMemsetAsync(gh, 0, 256 * sizeof(u32), cx().stream));
    const u32 nbins = bins_per_rank * nranks;
    const int hgrid = grid_for(4096, ids->n, 4);
    if (ids->n) {
        if (nbins <= 2) LAUNCH("hist_ids", k_hist_u32_div<2>, hgrid, 512, 0, ids->d, ids->n, rb, nbins, gh);
        else if (nbins <= 4) LAUNCH("hist_ids", k_hist_u32_div<4>, hgrid, 512, 0, ids->d, ids->n, rb, nbins, gh);
        else if (nbins <= 8) LAUNCH("hist_ids", k_hist_u32_div<8>, hgrid, 512, 0, ids->d, ids->n, rb, nbins, gh);
        else if (nbins <= 16) LAUNCH("hist_ids", k_hist_u32_div<16>, hgrid, 512, 0, ids->d, ids->n, rb, nbins, gh);
        else LAUNCH("hist_ids", k_hist_u32_div<256>, hgrid, 512, 0, ids->d, ids->n, rb, nbins, gh);
    }
    u32 tmp[256];
    CK(cudaMemcpyAsync(tmp, gh, sizeof tmp, cudaMemcpyDeviceToHost, cx().stream));
    CK(cudaStreamSynchronize(cx().stream));
    for (u32 b = 0; b < bins_per_rank * nranks; b++) hist[b] = tmp[b];
    dfree(gh);
    return 0;
}

int qce_push_rowids(const qce_rowids *ids, uint32_t rows_per_rank, uint32_t bin_width, uint32_t bins_per_rank,
                    uint32_t nranks, const uint64_t *bin_u32_offset)
{
    NEED_INIT();
    if (!ids || !bin_u32_offset) return fail("null argument");
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    RowBins rb;
    if (row_bins(rows_per_rank, bin_width, bins_per_rank, nranks, &rb) != 0) return -1;
    if (nranks != G.xworld) return fail("nranks (%u) differs from the attached world size (%u)", nranks, G.xworld);
    if (ids->n >= (1ull << 32)) return fail("row-id column too long");
    if (ids->n == 0) return 0;
    const u32 nbins = bins_per_rank * nranks;
    unsigned long long *d_seg = nullptr, *d_cur = nullptr;
    u32 *d_run = nullptr;
    if (push_scratch(nbins, bin_u32_offset, nullptr, &d_seg, &d_run, &d_cur) != 0) return -1;
    PushDigit<u32> dg;
    dg.bins = rb;
    PushPlan plan{d_seg, d_run, d_cur, nbins, bins_per_rank};
    const u32 n = (u32)ids->n, grid = (u32)ceil_div(n, PushTile<u32>::TILE);
    PushCols nocols;
    memset(&nocols, 0, sizeof nocols);
    if (nbins <= 16)
        LAUNCH("push_rowids", (k_push<u32, true, false>), grid, QCE_PUSH_THREADS, 0, (const u32 *)ids->d, n, dg, plan, G.peers,
               bitlen(nbins - 1), (u32 *)nullptr, nocols);
    else
        LAUNCH("push_rowids", (k_push<u32, false, false>), grid, QCE_PUSH_THREADS, 0, (const u32 *)ids->d, n, dg, plan, G.peers, 0,
               (u32 *)nullptr, nocols);
    dfree(d_seg); dfree(d_cur); dfree(d_run);
    return 0;
}

// Carried columns of the sharded executor (sharded.py): join keys travel with the rows.
int qce_column_window_u32(uint32_t rel, uint32_t col, uint64_t row_begin, uint64_t row_count, qce_rowids **out)
{
    NEED_INIT();
    const Column *cl;
    if (!out) return fail("null argument");
    if (get_column(rel, col, &cl) != 0) return -1;
    if (row_begin > cl->n || row_count > cl->n - row_begin) return fail("row window outside relation %u", rel);
    if (!window_resident(cl, row_begin, row_count)) return fail("rows are not resident on this rank");
    if (cl->maxv >> 32) return fail("column %u.%u holds values >= 2^32: cannot be carried as 4-byte keys", rel, col);
    if (new_rowids(row_count, 0, out) != 0) return -1;
    if (row_count) LAUNCH("narrow_col", k_narrow_u64, grid_for(2048, row_count), 256, 0, cl->d + row_begin, row_count, (*out)->d);
    return 0;
}
int qce_column_gather_u32(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_rowids **out)
{
    NEED_INIT();
    const Column *cl;
    if (!ids || !out) return fail("null argument");
    if (get_column(rel, col, &cl) != 0) return -1;
    if (cl->maxv >> 32) return fail("column %u.%u holds values >= 2^32: cannot be carried as 4-byte keys", rel, col);
    if (new_rowids(ids->n, 0, out) != 0) return -1;
    if (ids->n) LAUNCH("gather_col", k_gather_u64_narrow, grid_for(2048, ids->n), 256, 0, ref_of(cl), ids->d, ids->n, (*out)->d);
    return 0;
}
int qce_rowids_iota(uint64_t begin, uint64_t count, uint32_t id_bound, qce_rowids **out)
{
    NEED_INIT();
    if (!out) return fail("null argument");
    if (begin + count > (1ull << 32)) return fail("row ids are 32-bit");
    if (new_rowids(count, id_bound, out) != 0) return -1;
    if (count) LAUNCH("iota_ids", k_iota_u32, grid_for(2048, count), 256, 0, (u32)begin, count, (*out)->d);
    return 0;
}
int qce_tuples_from_u32(const qce_rowids *keys, uint32_t key_bits, qce_tuples **out)
{
    NEED_INIT();
    if (!keys || !out) return fail("null argument");
    if (key_bits == 0 || key_bits > 32) return fail("packed runs carry keys of 1..32 bits");
    if (keys->n >= (1ull << 32)) return fail("run too long");
    qce_tuples *t = new qce_tuples();
    t->n = keys->n;
    t->key_bits = (int)key_bits;
    t->key_min = 0;
    t->key_max = key_bits >= 32 ? 0xffffffffull : ((1ull << key_bits) - 1);
    t->wide = false;
    t->id_bound = (u32)keys->n;
    t->sorted = false;
    t->ids = nullptr;
    if (dalloc(&t->a, t->n) != 0) { delete t; return -1; }
    if (t->n) LAUNCH("pack_keys", k_pack_u32_index, grid_for(2048, t->n), 256, 0, keys->d, t->n, t->a);
    *out = t;
    return 0;
}

// Views of this rank's window after the peers' pushes have landed (the caller
// has synchronised every pushing rank: qce_sync on each + a barrier).
int qce_tuples_from_window(uint64_t word_offset, uint64_t n, uint32_t key_bits, uint32_t id_bound, uint64_t key_lo,
                           uint64_t key_hi, qce_tuples **out)
{
    NEED_INIT();
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    if ((word_offset + n) * 8 > G.xwin_bytes) return fail("run [%llu, +%llu) words exceeds the exchange window", (unsigned long long)word_offset, (unsigned long long)n);
    if (word_offset & 1) return fail("runs in the window start on 16-byte boundaries");
    return tuples_from_device(G.peers.base[G.xrank] + word_offset * 8, n, key_bits, id_bound, key_lo, key_hi, true, out);
}
int qce_tuples_from_window_wide(uint64_t word_offset, uint64_t id_u32_offset, uint64_t n, uint32_t id_bound, uint64_t key_lo,
                                uint64_t key_hi, qce_tuples **out)
{
    NEED_INIT();
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    if (!out) return fail("null argument");
    if ((word_offset + n) * 8 > G.xwin_bytes || (id_u32_offset + n) * 4 > G.xwin_bytes)
        return fail("run of %llu tuples at words %llu / ids %llu exceeds the exchange window", (unsigned long long)n,
                    (unsigned long long)word_offset, (unsigned long long)id_u32_offset);
    if ((word_offset & 1) || (id_u32_offset & 3)) return fail("runs in the window start on 16-byte boundaries");
    if (n && key_hi < key_lo) return fail("empty key range [%llu, %llu]", (unsigned long long)key_lo, (unsigned long long)key_hi);
    qce_tuples *t = new qce_tuples();
    t->a = (u64 *)(G.peers.base[G.xrank] + word_offset * 8); // not from the arena: freeing the run leaves the window alone
    t->ids = (u32 *)(G.peers.base[G.xrank] + id_u32_offset * 4);
    t->n = n;
    t->wide = true;
    t->key_bits = bitlen(key_hi) ? bitlen(key_hi) : 1;
    t->key_min = key_lo;
    t->key_max = key_hi;
    t->range_sort = true;
    t->id_bound = id_bound;
    t->sorted = false;
    *out = t;
    return 0;
}
int qce_rowids_from_window(uint64_t u32_offset, uint64_t n, uint32_t id_min, uint32_t id_bound, int bucketed,
                           qce_rowids **out)
{
    NEED_INIT();
    if (!G.xwin) return fail("no exchange window (qce_xwin_create)");
    if (!out) return fail("null argument");
    if ((u32_offset + n) * 4 > G.xwin_bytes) return fail("row-id column exceeds the exchange window");
    qce_rowids *r = new qce_rowids();
    r->d = (u32 *)(G.peers.base[G.xrank] + u32_offset * 4); // not from the arena: freeing the handle leaves it alone
    r->n = n;
    r->id_bound = id_bound;
    r->id_min = id_min;
    r->bucketed = bucketed != 0;
    *out = r;
    return 0;
}
// out[i] = ids[index[i]]: a bystander column re-aligned with a join output whose
// payloads are positions in the (received) entity (SURVEY.md 8f-2).
int qce_rowids_gather(const qce_rowids *src, const qce_rowids *index, qce_rowids **out)
{
    NEED_INIT();
    if (!src || !index || !out) return fail("null argument");
    const u32 *from = src->d;
    if (index->attach_gen && index->attach_gen == cx().attach_gen) {
        // the positions index the copy of `src` that travelled with the tuples of the last exchange
        from = nullptr;
        for (auto &kv : cx().recv_cols)
            if (kv.first == src) from = kv.second->d;
        if (!from) return fail("this column did not travel with the exchanged run");
    }
    if (new_rowids(index->n, src->id_bound, out) != 0) return -1;
    if (index->n) LAUNCH("gather_ids", k_gather_u32, grid_for(2048, index->n), 256, 0, from, index->d, index->n, (*out)->d);
    (*out)->n_others = index->n_others;
    (*out)->dist = index->dist;
    if ((*out)->dist.kind == Dist::KEYS) (*out)->dist.kind = Dist::ANY; // key order of another column
    return 0;
}

// ---- exchange bookkeeping (pure host arithmetic: usable without a device) ------------
// Every rank runs this on the same all-gathered histograms and therefore derives the same
// splitters, count matrix and window layout; nothing about a transfer is communicated.
int qce_exchange_plan(const uint64_t *hists, uint32_t world, uint32_t rank, uint32_t nsides, const uint32_t *ncols,
                      uint32_t key_bits, uint64_t *splitters, uint64_t *recv, uint64_t *before, uint64_t *run_off,
                      uint64_t *col_off, uint64_t *window_bytes, uint64_t *sent_tuples)
{
    return exchange_plan_impl(hists, world, rank, nsides, ncols, key_bits, nullptr, splitters, recv, before, run_off, col_off,
                              window_bytes, sent_tuples);
}
int qce_split_plan(const uint64_t *hists, uint32_t world, uint32_t rank, const uint32_t *ncols, uint32_t key_bits,
                   uint32_t nlevels, const uint32_t *nsel, const uint64_t *sub_hists, uint32_t *next_nsel,
                   uint64_t *next_sel, uint32_t *next_sel_shift, qce_split_plan_t *plan)
{
    return split_plan_impl(hists, world, rank, ncols, key_bits, nlevels, nsel, sub_hists, next_nsel, next_sel, next_sel_shift, plan);
}

// Row ids routed to the ranks that own the rows: per binding, where this rank's ids of every
// bin go in the owner's window (bin-major inside an owner, earlier ranks first inside a bin).
int qce_rowid_push_plan(const uint64_t *hists, uint32_t world, uint32_t rank, uint32_t nbind, uint32_t bins_per_rank,
                        uint64_t *bin_u32_offset, uint64_t *view_u32_offset, uint64_t *view_count, uint64_t *window_bytes,
                        uint64_t *sent_ids)
{
    if (!hists || !bin_u32_offset || !view_u32_offset || !view_count || !window_bytes || !sent_ids) return fail("null argument");
    if (world < 1 || world > QCE_MAX_RANKS || rank >= world || bins_per_rank < 1 || (u64)bins_per_rank * world > 256)
        return fail("bad row-bin shape");
    const u32 nb = bins_per_rank * world;
    std::vector<u64> top(world, 0);
    for (u32 k = 0; k < nbind; k++) {
        sent_ids[k] = 0;
        for (u32 d = 0; d < world; d++) {
            u64 at = 0; // ids before the current bin inside owner d's region
            for (u32 j = 0; j < bins_per_rank; j++) {
                const u32 b = d * bins_per_rank + j;
                u64 tot = 0, bef = 0;
                for (u32 s = 0; s < world; s++) {
                    const u64 c = hists[((size_t)s * nbind + k) * nb + b];
                    if (s < rank) bef += c;
                    if (s == rank && d != rank) sent_ids[k] += c;
                    tot += c;
                }
                bin_u32_offset[(size_t)k * nb + b] = top[d] / 4 + at + bef;
                at += tot;
            }
            if (d == rank) { view_u32_offset[k] = top[d] / 4; view_count[k] = at; }
            top[d] = (top[d] + 4 * at + 15) / 16 * 16;
        }
    }
    *window_bytes = *std::max_element(top.begin(), top.end());
    return 0;
}

} // extern "C"

namespace {
int exchange_plan_impl(const uint64_t *hists, uint32_t world, uint32_t rank, uint32_t nsides, const uint32_t *ncols,
                      uint32_t key_bits, const uint64_t *fixed_splitters, uint64_t *splitters, uint64_t *recv, uint64_t *before, uint64_t *run_off,
                      uint64_t *col_off, uint64_t *window_bytes, uint64_t *sent_tuples)
{
    if (!hists || !ncols || !splitters || !recv || !before || !run_off || !col_off || !window_bytes || !sent_tuples)
        return fail("null argument");
    if (world < 1 || world > QCE_MAX_RANKS || rank >= world || nsides < 1 || nsides > 8) return fail("bad exchange shape");
    if (key_bits == 0 || key_bits > 64) return fail("key width must be 1..64");
    const int shift = key_bits > 8 ? (int)key_bits - 8 : 0;
    // global histogram -> splitters on bin boundaries that balance tuples per rank
    u64 cum[256], total = 0;
    for (u32 b = 0; b < 256; b++) {
        u64 v = 0;
        for (u32 s = 0; s < world; s++)
            for (u32 k = 0; k < nsides; k++) v += hists[((size_t)s * nsides + k) * 256 + b];
        total += v;
        cum[b] = total;
    }
    u32 bnd[QCE_MAX_RANKS + 1];
    bnd[0] = 0;
    u32 prev = 0;
    for (u32 k = 1; k < world; k++) {
        // first bin whose cumulative count reaches total * k / world, plus one = first bin of the next part
        u32 i = 0;
        while (i < 256 && (unsigned __int128)cum[i] * world < (unsigned __int128)total * k) i++;
        u32 b = i + 1;
        if (fixed_splitters) { // a run already in place dictates the cut (must sit on a bin boundary)
            if (!on_bin_boundary(fixed_splitters[k - 1], shift)) return fail("fixed splitter off the histogram bins");
            b = cut_bin(fixed_splitters[k - 1], shift);
        }
        if (b < prev) b = prev;
        if (b > 256) b = 256;
        splitters[k - 1] = cut_key(b, shift);
        prev = b;
        bnd[k] = b;
    }
    bnd[world] = 256;
    // C[k][s][d] = tuples of side k that rank s sends to rank d; recv, this rank's segment starts
    std::vector<u64> top(world, 0);
    size_t col_at = 0;
    for (u32 k = 0; k < nsides; k++) {
        sent_tuples[k] = 0;
        for (u32 d = 0; d < world; d++) {
            u64 r = 0, bef = 0;
            for (u32 s = 0; s < world; s++) {
                u64 c = 0;
                const uint64_t *h = hists + ((size_t)s * nsides + k) * 256;
                for (u32 b = bnd[d]; b < bnd[d + 1]; b++) c += h[b];
                if (s < rank) bef += c;
                if (s == rank && d != rank) sent_tuples[k] += c;
                r += c;
            }
            recv[(size_t)k * world + d] = r;
            before[(size_t)k * world + d] = bef;
        }
        // window layout of every destination (bytes): the run, then its columns, 16-byte aligned
        for (u32 d = 0; d < world; d++) {
            run_off[(size_t)k * world + d] = top[d];
            top[d] = (top[d] + 8 * recv[(size_t)k * world + d] + 15) / 16 * 16;
        }
        for (u32 j = 0; j < ncols[k]; j++, col_at++)
            for (u32 d = 0; d < world; d++) {
                col_off[col_at * world + d] = top[d];
                top[d] = (top[d] + 4 * recv[(size_t)k * world + d] + 15) / 16 * 16;
            }
    }
    *window_bytes = *std::max_element(top.begin(), top.end());
    return 0;
}

// ---- exchange plan with cuts inside heavy keys (qce_split_plan) ---------------------------
// The key space as an ordered list of pieces -- histogram bins of some level, refined where a cut
// falls -- each with its tuples per (source, side).  A cut is (key, q): the next rank starts at
// `key`, after the first q outer tuples of that key's global group (q = 0: at the key's start).
struct PlanPiece {
    u64 lo;    // first key; the piece holds [lo, lo + 2^shift)
    int shift;
    std::vector<u64> c; // [source * 2 + side]
};
struct PlanCut {
    u64 key = 0, q = 0;
    bool operator<(const PlanCut &o) const { return key != o.key ? key < o.key : q < o.q; }
};

// Tuple positions are counted in one stream, key by key, a key's inner tuples before its outer
// ones (a rank that takes part of a key's outer group also holds all of its inner group).  Cut k
// aims at T * k / W and is good within share / 20, which keeps every rank within 10 % of its share
// (plus the inner copies of split keys).  *refine gets the pieces that hold a cut that missed and
// can still be refined.
void plan_cuts(const std::vector<PlanPiece> &pieces, u32 W, std::vector<PlanCut> *cuts, std::vector<size_t> *refine)
{
    std::vector<u64> tot(pieces.size()), inner(pieces.size()), outer(pieces.size());
    u64 T = 0;
    for (size_t i = 0; i < pieces.size(); i++) {
        u64 r = 0, s = 0;
        for (u32 src = 0; src < W; src++) { r += pieces[i].c[src * 2]; s += pieces[i].c[src * 2 + 1]; }
        outer[i] = r; inner[i] = s; tot[i] = r + s; T += r + s;
    }
    cuts->assign(W - 1, PlanCut());
    refine->clear();
    size_t i = 0;
    u64 cum = 0; // tuples before piece i
    for (u32 k = 1; k < W; k++) {
        typedef unsigned __int128 u128;
        const u128 goal = (u128)T * k; // the target, scaled by W
        while (i + 1 < pieces.size() && (u128)(cum + tot[i]) * W < goal) { cum += tot[i]; i++; }
        const PlanPiece &p = pieces[i];
        const u128 eb = goal - (u128)cum * W, ea = (u128)(cum + tot[i]) * W - goal; // misses of the two boundaries
        PlanCut c;
        c.key = eb <= ea ? p.lo : p.lo + (1ull << p.shift);
        if (std::min(eb, ea) * 20 > (u128)T) {
            if (p.shift > 0) {
                if (refine->empty() || refine->back() != i) refine->push_back(i);
            } else {
                const u64 t = (u64)(goal / W);
                if (outer[i] >= 2 && t > cum + inner[i]) {
                    const u64 q = t - cum - inner[i];
                    if (q < outer[i]) { c.key = p.lo; c.q = q; }
                }
            }
        }
        if (k > 1 && c < (*cuts)[k - 2]) c = (*cuts)[k - 2];
        (*cuts)[k - 1] = c;
    }
}

int split_plan_impl(const uint64_t *hists, uint32_t W, uint32_t rank, const uint32_t *ncols, uint32_t key_bits,
                    uint32_t nlevels, const uint32_t *nsel, const uint64_t *sub_hists, uint32_t *next_nsel,
                    uint64_t *next_sel, uint32_t *next_sel_shift, qce_split_plan_t *P)
{
    if (!hists || !ncols || !next_nsel || !next_sel || !next_sel_shift || !P || (nlevels && (!nsel || !sub_hists)))
        return fail("null argument");
    if (W < 1 || W > QCE_PLAN_MAX_RANKS || rank >= W) return fail("bad exchange shape");
    if (key_bits == 0 || key_bits > 32) return fail("packed runs carry keys of 1..32 bits");
    if (ncols[0] + ncols[1] > QCE_PLAN_MAX_COLS) return fail("at most %d columns travel with the two runs", QCE_PLAN_MAX_COLS);
    memset(P, 0, sizeof *P);
    *next_nsel = 0;
    *next_sel_shift = 0;
    const int shift0 = key_bits > 8 ? (int)key_bits - 8 : 0;
    std::vector<PlanPiece> pieces(256);
    for (u32 b = 0; b < 256; b++) {
        pieces[b].lo = (u64)b << shift0;
        pieces[b].shift = shift0;
        pieces[b].c.resize((size_t)W * 2);
        for (u32 s = 0; s < W; s++)
            for (u32 k = 0; k < 2; k++) pieces[b].c[s * 2 + k] = hists[((size_t)s * 2 + k) * 256 + b];
    }
    std::vector<PlanCut> cuts(W - 1);
    // today's bin cuts first: refine only when they leave a rank more than 10 % over its share
    {
        uint64_t sp[QCE_PLAN_MAX_RANKS], recv[2 * QCE_PLAN_MAX_RANKS], bef[2 * QCE_PLAN_MAX_RANKS], ro[2 * QCE_PLAN_MAX_RANKS];
        uint64_t co[QCE_PLAN_MAX_COLS * QCE_PLAN_MAX_RANKS], need, sent[2];
        if (exchange_plan_impl(hists, W, rank, 2, ncols, key_bits, nullptr, sp, recv, bef, ro, co, &need, sent) != 0) return -1;
        u64 T = 0, mx = 0;
        for (u32 d = 0; d < W; d++) { T += recv[d] + recv[W + d]; mx = std::max<u64>(mx, recv[d] + recv[W + d]); }
        for (u32 k = 0; k + 1 < W; k++) cuts[k].key = sp[k];
        const bool bins_balanced = W == 1 || (unsigned __int128)mx * 10 * W <= (unsigned __int128)T * 11;
        if (!bins_balanced) {
            P->refined = 1;
            const uint64_t *sub = sub_hists;
            for (u32 lvl = 0;; lvl++) {
                std::vector<size_t> refine;
                plan_cuts(pieces, W, &cuts, &refine);
                if (refine.empty()) { P->levels = lvl; break; }
                const int sh = pieces[refine[0]].shift, sub_shift = sh > 8 ? sh - 8 : 0;
                for (size_t i : refine)
                    if (pieces[i].shift != sh) return fail("refinement across levels");
                if (lvl == nlevels) { // ask for the next level's histograms
                    *next_nsel = (u32)refine.size();
                    *next_sel_shift = (u32)sh;
                    for (size_t j = 0; j < refine.size(); j++) next_sel[j] = pieces[refine[j]].lo >> sh;
                    P->levels = lvl;
                    return 0;
                }
                if (nsel[lvl] != refine.size()) return fail("level %u: %u histograms given, %zu asked", lvl, nsel[lvl], refine.size());
                const u32 ns = nsel[lvl], nsub = 1u << (sh - sub_shift);
                std::vector<PlanPiece> next;
                next.reserve(pieces.size() + refine.size() * nsub);
                for (size_t i = 0, j = 0; i < pieces.size(); i++) {
                    if (j < refine.size() && refine[j] == i) {
                        for (u32 b = 0; b < nsub; b++) {
                            PlanPiece q;
                            q.lo = pieces[i].lo + ((u64)b << sub_shift);
                            q.shift = sub_shift;
                            q.c.resize((size_t)W * 2);
                            for (u32 s = 0; s < W; s++)
                                for (u32 k = 0; k < 2; k++) q.c[s * 2 + k] = sub[(((size_t)s * 2 + k) * ns + j) * 256 + b];
                            next.push_back(std::move(q));
                        }
                        j++;
                    } else {
                        next.push_back(std::move(pieces[i]));
                    }
                }
                pieces.swap(next);
                sub += (size_t)W * 2 * ns * 256;
            }
        }
    }
    // the plan of these cuts: per piece its destination, a split key's groups divided by position
    for (u32 k = 0; k + 1 < W; k++) { P->cut_key[k] = cuts[k].key; P->cut_q[k] = cuts[k].q; }
    size_t ci = 0; // cuts at or before the current piece's first key
    for (const PlanPiece &p : pieces) {
        while (ci < cuts.size() && cuts[ci].q == 0 && cuts[ci].key <= p.lo) ci++;
        size_t cj = ci;
        while (cj < cuts.size() && cuts[cj].key == p.lo && cuts[cj].q > 0) cj++;
        const u32 first = (u32)ci, m = (u32)(cj - ci);
        if (m == 0) {
            for (u32 s = 0; s < W; s++)
                for (u32 k = 0; k < 2; k++) P->count[k][s][first] += p.c[s * 2 + k];
            continue;
        }
        const u32 j = P->nsplit++;
        P->split_key[j] = p.lo;
        P->split_first[j] = first;
        P->split_last[j] = first + m;
        u64 r = 0;
        for (u32 s = 0; s < W; s++) r += p.c[s * 2];
        u64 pre = 0;
        for (u32 s = 0; s < W; s++) {
            const u64 rs = p.c[s * 2];
            for (u32 i = 0; i <= m; i++) {
                const u64 q0 = i == 0 ? 0 : cuts[ci + i - 1].q, q1 = i == m ? r : cuts[ci + i].q;
                const u64 a = std::max(q0, pre), b = std::min(q1, pre + rs);
                P->count[0][s][first + i] += b > a ? b - a : 0;
                P->count[1][s][first + i] += p.c[s * 2 + 1];
                P->split_bound[j][s][i] = std::min(rs, q0 > pre ? q0 - pre : 0);
            }
            P->split_count[j][s][0] = rs;
            P->split_count[j][s][1] = p.c[s * 2 + 1];
            pre += rs;
        }
        ci = cj;
    }
    const u64 key_top = (1ull << key_bits) - 1;
    // exactly the keys the push delivers: a rank between two equal whole-key cuts, or past the last key,
    // gets an empty range (key_lo > key_hi)
    for (u32 d = 0; d < W; d++) {
        const int64_t lo = d == 0 ? 0 : (int64_t)cuts[d - 1].key; // keys < 2^32, cuts <= 2^32
        const int64_t hi = std::min<int64_t>((int64_t)key_top, d + 1 == W ? (int64_t)key_top
                                                                : cuts[d].q ? (int64_t)cuts[d].key : (int64_t)cuts[d].key - 1);
        if (hi < lo) { P->key_lo[d] = 1; P->key_hi[d] = 0; }
        else { P->key_lo[d] = (u64)lo; P->key_hi[d] = (u64)hi; }
    }
    // the window layout, as exchange_plan_impl lays it out
    std::vector<u64> top(W, 0);
    size_t col_at = 0;
    for (u32 k = 0; k < 2; k++) {
        P->sent[k] = 0;
        for (u32 d = 0; d < W; d++) {
            for (u32 s = 0; s < W; s++) {
                const u64 c = P->count[k][s][d];
                if (s < rank) P->before[k][d] += c;
                if (s == rank && d != rank) P->sent[k] += c;
                P->recv[k][d] += c;
            }
            P->run_off[k][d] = top[d];
            top[d] = (top[d] + 8 * P->recv[k][d] + 15) / 16 * 16;
        }
        for (u32 c = 0; c < ncols[k]; c++, col_at++)
            for (u32 d = 0; d < W; d++) {
                P->col_off[col_at][d] = top[d];
                top[d] = (top[d] + 4 * P->recv[k][d] + 15) / 16 * 16;
            }
    }
    P->window_bytes = *std::max_element(top.begin(), top.end());
    return 0;
}

} // namespace
