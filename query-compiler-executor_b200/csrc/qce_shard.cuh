// qce_shard.cuh -- the operators of include/qce_b200.h when the node runs several ranks
// (SURVEY.md 8e, BASELINE.json north_star: "large joins shard across the 8 GPUs by radix
// high bits ... over NVLink and a final checksum reduce").
//
// Included by qce_engine.cu.  The host operator layer (src/filter.c, src/join.c,
// src/utilities.c -- the reference's execute_filter / execute_join / print_sums contract)
// is unchanged and runs SPMD: every rank makes the same calls, in the same order, on its
// share of the data, and every value the host branches on (counts, sortedness) is agreed
// through qce_comm.cuh, so all ranks take the same decisions of the mid-result state machine.
//
//   object                 this rank's share                              Dist
//   base column            its row window (or everything: replicated)    -
//   filter output          the hits inside its row window, ascending     ROWS
//   run to be joined       whatever it built; qce_sort_tuples only marks it (sort_pending)
//   join input, exchanged  the tuples of its key range, pushed by all ranks straight into
//                          its window over NVLink (k_push), sorted locally
//   join output            the pairs of its key range, key order         KEYS(splitters)
//   anything else          a contiguous piece of the global order        ANY
//
// The global order of every distributed column is "rank 0's share, then rank 1's, ...",
// which is what the reference's serial loops produce, so positional operators (scan_join,
// join_payloads: src/join.c:395-484) keep their meaning: when two columns of different
// shape meet positionally one is re-cut to the other's per-rank counts (realign), and the
// operators that are serial by nature (the pointer walk over an unsorted run) gather their
// inputs on rank 0 -- a valid distribution like any other.  Nothing is ever answered
// differently from the single-GPU engine.
#pragma once

namespace {

thread_local int tl_local_depth = 0;
struct LocalScope {
    LocalScope() { tl_local_depth++; }
    ~LocalScope() { tl_local_depth--; }
};
inline bool sharded() { return G.world > 1 && !cx().solo && tl_local_depth == 0; }
inline int comm_fail() { return fail("rank %u: %s", G.rank, qcecomm::st().err); }

#define CQ(call)                                   \
    do {                                           \
        if ((call) != 0) return comm_fail();       \
    } while (0)

int fence()
{
    CK(cudaStreamSynchronize(cx().stream));
    return 0;
}
int fence_barrier()
{
    if (fence() != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::barrier());
    return 0;
}
// n_others of an object whose local size is n
int others_of(u64 n, u64 *n_others)
{
    uint64_t v = n;
    CQ(qcecomm::allreduce_sum(&v, 1));
    *n_others = v - n;
    return 0;
}

// ---- the receive window --------------------------------------------------------------
// One per rank, mapped by every peer (CUDA IPC).  Every operator that stores into the
// peers' windows starts here: own stream drained, then a collective -- so when it returns
// every rank has finished reading whatever the window held before.
int ensure_window(u64 need)
{
    if (fence() != 0) { qcecomm::abort_all(); return -1; }
    uint64_t v[2] = {need, G.xwin_bytes};
    CQ(qcecomm::allreduce_max(v, 2));
    if (G.xwin && v[0] <= G.xwin_bytes && G.xworld == G.world) return 0;
    // (re)create: every rank takes this branch together -- `need` was maximised over the ranks and
    // the windows are created with identical sizes
    if (qce_xwin_unmap_peers() != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::barrier()); // nobody frees a window a peer still maps
    if (qce_xwin_destroy() != 0) return -1;
    u64 bytes = std::max<u64>(v[0] + v[0] / 4, 64ull << 20);
    unsigned char mine[64], all[QCE_MAX_RANKS * 64];
    if (qce_xwin_create(bytes, mine) != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::allgather(mine, 64, all));
    if (qce_xwin_attach(G.world, G.rank, all) != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::barrier());
    return 0;
}

// ---- positional redistribution ---------------------------------------------------------
// The distributed array whose local piece is (src, n) is re-cut so that rank d holds the
// elements at global positions [T_d, T_d + target[d]) (T = exclusive prefix of target,
// clipped to the array's length).  *out is an arena buffer.
int realign(const void *src, u64 n, u32 esz, const std::vector<u64> &target, void **out, u64 *out_n)
{
    const u32 W = G.world, me = G.rank;
    std::vector<uint64_t> cnt(W);
    uint64_t mine = n;
    if (fence() != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::allgather(&mine, sizeof mine, cnt.data()));
    u64 my_start = 0, total = 0;
    for (u32 r = 0; r < W; r++) { if (r < me) my_start += cnt[r]; total += cnt[r]; }
    std::vector<u64> tstart(W), tlen(W);
    u64 at = 0, need = 0;
    for (u32 d = 0; d < W; d++) {
        tstart[d] = std::min(at, total);
        tlen[d] = std::min<u64>(target[d], total - tstart[d]);
        at += target[d];
        need = std::max(need, (tlen[d] * esz + 15) / 16 * 16);
    }
    if (ensure_window(need) != 0) return -1;
    for (u32 d = 0; d < W; d++) {
        const u64 lo = std::max(my_start, tstart[d]), hi = std::min(my_start + n, tstart[d] + tlen[d]);
        if (hi > lo)
            CK(cudaMemcpyAsync(G.peers.base[d] + (lo - tstart[d]) * esz, (const char *)src + (lo - my_start) * esz,
                               (hi - lo) * esz, cudaMemcpyDeviceToDevice, cx().stream));
    }
    if (fence_barrier() != 0) return -1;
    void *p = nullptr;
    if (cx().arena.alloc(&p, tlen[me] * esz ? tlen[me] * esz : 16) != 0) { qcecomm::abort_all(); return -1; }
    if (tlen[me]) CK(cudaMemcpyAsync(p, G.xwin, tlen[me] * esz, cudaMemcpyDeviceToDevice, cx().stream));
    *out = p;
    *out_n = tlen[me];
    return 0;
}
std::vector<u64> counts_all_on_root(u64 total_cap = ~0ull)
{
    std::vector<u64> t(G.world, 0);
    t[0] = total_cap;
    return t;
}
int all_counts(u64 n, std::vector<u64> *out)
{
    out->assign(G.world, 0);
    uint64_t mine = n;
    std::vector<uint64_t> c(G.world);
    CQ(qcecomm::allgather(&mine, sizeof mine, c.data()));
    for (u32 r = 0; r < G.world; r++) (*out)[r] = c[r];
    return 0;
}
// a row-id column re-cut to `target`; the result is a fresh handle (dist ANY)
int realign_rowids(const qce_rowids *in, const std::vector<u64> &target, qce_rowids **out)
{
    void *p = nullptr;
    u64 m = 0;
    if (realign(in->d, in->n, 4, target, &p, &m) != 0) return -1;
    qce_rowids *r = new qce_rowids();
    r->d = (u32 *)p;
    r->n = m;
    r->id_bound = in->id_bound;
    r->n_others = in->n + in->n_others - m;
    r->dist.kind = Dist::ANY;
    *out = r;
    return 0;
}
// a tuple run gathered on rank 0 (the other ranks keep an empty run)
int tuples_to_root(const qce_tuples *in, qce_tuples **out)
{
    const std::vector<u64> target = counts_all_on_root();
    qce_tuples *t = new qce_tuples();
    void *p = nullptr;
    u64 m = 0;
    if (realign(in->a, in->n, 8, target, &p, &m) != 0) { delete t; return -1; }
    t->a = (u64 *)p;
    t->ids = nullptr;
    if (in->wide) {
        void *q = nullptr;
        u64 m2 = 0;
        if (realign(in->ids, in->n, 4, target, &q, &m2) != 0) { delete t; return -1; }
        t->ids = (u32 *)q;
    }
    t->n = m;
    t->wide = in->wide;
    t->key_bits = in->key_bits;
    t->key_min = 0;
    t->key_max = in->dist.kind == Dist::KEYS ? 0 : in->key_max; // a key-range share knew only its own range
    if (in->dist.kind == Dist::KEYS) t->key_max = (in->key_bits >= 64) ? ~0ull : ((1ull << in->key_bits) - 1);
    t->id_bound = in->id_bound;
    t->sorted = false;
    t->n_others = in->n + in->n_others - m;
    t->dist.kind = Dist::ANY;
    t->sort_pending = in->sort_pending;
    *out = t;
    return 0;
}

// ---- exchange by key range ---------------------------------------------------------------
// The multi-GPU half of the reference's radix partitioning (build_histogram / build_psum /
// build_reordered_array, src/utilities.c:20-70): 256-bin histograms of the top key bits,
// ONE all-gather, splitters that balance the tuples per rank (or the splitters of a run
// that is already in place), then k_push stores every tuple straight into its owner's window.
int exchange_plan_impl(const uint64_t *hists, uint32_t world, uint32_t rank, uint32_t nsides, const uint32_t *ncols,
                       uint32_t key_bits, const uint64_t *fixed_splitters, uint64_t *splitters, uint64_t *recv,
                       uint64_t *before, uint64_t *run_off, uint64_t *col_off, uint64_t *window_bytes, uint64_t *sent_tuples);

struct XRecv {
    qce_tuples *run = nullptr; // a view of this rank's window: valid until the window is written again
    bool travelled = false;    // its attached columns came along (cx().recv_cols, generation cx().attach_gen)
};
// sort_received: the received runs are sorted here, the first one on the context's aux stream as
// soon as ITS tuples have landed everywhere -- while the second side's push still crosses NVLink.
// wide_base != nullptr: every side is wide, binned by key - *wide_base over key_bits (1..64) bits; a
// side's ids are laid out like one travelling column behind its keys.
int exchange_runs(const std::vector<const qce_tuples *> &sides, int key_bits, u64 key_max, const Dist *fixed,
                  std::vector<XRecv> *out, Dist *dist_out, bool sort_received = false, const u64 *wide_base = nullptr)
{
    static int overlap = -1; // QCE_OVERLAP_PUSH=0: one barrier after all pushes, sorts afterwards
    if (overlap < 0) { const char *e = getenv("QCE_OVERLAP_PUSH"); overlap = e ? atoi(e) : 1; }
    const u32 W = G.world, me = G.rank, ns = (u32)sides.size();
    const bool wide = wide_base != nullptr;
    const u64 base = wide ? *wide_base : 0;
    std::vector<uint64_t> hists((size_t)ns * 256), all((size_t)W * ns * 256);
    for (u32 k = 0; k < ns; k++) {
        const int rc = wide ? qce_key_histogram_wide(sides[k], base, (u32)key_bits, hists.data() + (size_t)k * 256)
                            : qce_key_histogram(sides[k], (u32)key_bits, hists.data() + (size_t)k * 256);
        if (rc != 0) { qcecomm::abort_all(); return -1; }
    }
    CQ(qcecomm::allgather(hists.data(), hists.size() * sizeof(uint64_t), all.data()));
    std::vector<uint32_t> ncols(ns, 0);
    size_t total_cols = 0;
    for (u32 k = 0; k < ns; k++) { ncols[k] = wide ? 1u : (u32)sides[k]->attached.size(); total_cols += ncols[k]; }
    std::vector<uint64_t> splitters(W), recv((size_t)ns * W), before((size_t)ns * W), run_off((size_t)ns * W),
        col_off((total_cols ? total_cols : 1) * W), sent(ns);
    uint64_t need = 0;
    if (exchange_plan_impl(all.data(), W, me, ns, ncols.data(), (u32)key_bits, fixed ? fixed->split.data() : nullptr,
                           splitters.data(), recv.data(), before.data(), run_off.data(), col_off.data(), &need, sent.data()) != 0) {
        qcecomm::abort_all();
        return -1;
    }
    if (ensure_window(need) != 0) return -1;
    // the views of the previous exchange's travelling columns die with the window's old contents
    for (auto &kv : cx().recv_cols) qce_rowids_free(kv.second);
    cx().recv_cols.clear();
    cx().attach_gen++;
    size_t col_at = 0;
    const bool split = sort_received && overlap && ns == 2;
    cx().defer_frees = split;
    for (u32 k = 0; k < ns; k++) {
        std::vector<uint64_t> dst_words(W);
        for (u32 d = 0; d < W; d++) dst_words[d] = run_off[(size_t)k * W + d] / 8 + before[(size_t)k * W + d];
        int rc;
        if (wide) {
            std::vector<uint64_t> dst_ids(W);
            for (u32 d = 0; d < W; d++) dst_ids[d] = col_off[col_at * W + d] / 4 + before[(size_t)k * W + d];
            rc = qce_push_tuples_wide(sides[k], base, (u32)key_bits, splitters.data(), W, dst_words.data(), dst_ids.data());
        } else if (ncols[k] == 0) {
            rc = qce_push_tuples(sides[k], (u32)key_bits, splitters.data(), W, dst_words.data(), nullptr, nullptr);
        } else {
            // payload := index in the receiver's run; the attached columns follow in the same kernel, laid
            // out like the run (segment of rank s after the segments of ranks < s)
            std::vector<uint32_t> run_index(W);
            std::vector<uint64_t> regions((size_t)ncols[k] * W);
            for (u32 d = 0; d < W; d++) run_index[d] = (u32)before[(size_t)k * W + d];
            for (u32 c = 0; c < ncols[k]; c++)
                for (u32 d = 0; d < W; d++) regions[(size_t)c * W + d] = col_off[(col_at + c) * W + d] / 4 + before[(size_t)k * W + d];
            rc = qce_push_tuples_cols(sides[k], (u32)key_bits, splitters.data(), W, dst_words.data(), run_index.data(), ncols[k],
                                      sides[k]->attached.data(), regions.data());
        }
        if (rc != 0) { cx().defer_frees = false; qcecomm::abort_all(); return -1; }
        if (split) CK(cudaEventRecord(cx().ev_side[k], cx().stream));
        col_at += ncols[k];
    }
    cx().defer_frees = false;
    if (!split && fence_barrier() != 0) return -1; // every peer's stores into this rank's window have completed
    u64 lo = me > 0 ? splitters[me - 1] : 0;
    // the last rank's range ends at the largest key that exists, not at 2^key_bits - 1: the
    // local sort sizes its MSD buckets from this range
    u64 hi = me < W - 1 ? splitters[me] - 1 : key_max;
    if (wide) { // base + [cut, next cut), clipped to the largest key (base + a cut past it may overflow)
        const u64 span = key_max - base, c0 = me > 0 ? splitters[me - 1] : 0, c1 = me < W - 1 ? splitters[me] : ~0ull;
        lo = base + std::min(c0, span);
        hi = (c1 == ~0ull || c1 > span) ? key_max : base + c1 - 1;
    }
    out->assign(ns, XRecv());
    cudaStream_t main_stream = cx().stream;
    for (u32 k = 0, id_col = 0; k < ns; id_col += ncols[k], k++) {
        if (split) {
            // side k has landed on every rank: this rank's push of it is done, and so is everybody else's
            cudaError_t e = cudaEventSynchronize(cx().ev_side[k]);
            if (e != cudaSuccess) { qcecomm::abort_all(); return fail("push of side %u: %s", k, cudaGetErrorString(e)); }
            CQ(qcecomm::barrier());
        }
        const u64 n = recv[(size_t)k * W + me];
        const int vrc = wide ? qce_tuples_from_window_wide(run_off[(size_t)k * W + me] / 8, col_off[(size_t)id_col * W + me] / 4, n,
                                                           sides[k]->id_bound, lo, std::max(lo, hi), &(*out)[k].run)
                             : qce_tuples_from_window(run_off[(size_t)k * W + me] / 8, n, (u32)key_bits, sides[k]->id_bound, lo,
                                                      std::max(lo, hi), &(*out)[k].run);
        if (vrc != 0) {
            qcecomm::abort_all();
            return -1;
        }
        u64 tot = 0;
        for (u32 d = 0; d < W; d++) tot += recv[(size_t)k * W + d];
        (*out)[k].run->n_others = tot - n;
        if (sort_received) {
            const bool early = split && k + 1 < ns; // the next side's push is still in flight on the main stream
            if (early) cx().stream = cx().aux;
            // the arena hands freed blocks out again at once (one stream per context): the last side's sort
            // must not start before the early one has finished with its temporaries -- and the merge reads both
            else if (split) cudaStreamWaitEvent(main_stream, cx().ev_aux, 0);
            int rc;
            {
                LocalScope ls;
                rc = qce_sort_tuples((*out)[k].run);
            }
            if (early) {
                cudaEventRecord(cx().ev_aux, cx().aux);
                cx().stream = main_stream;
            }
            if (rc != 0) { qcecomm::abort_all(); return -1; }
        }
    }
    if (split) release_deferred(); // the pushes that read this scratch have completed (ev_side[1])
    col_at = 0;
    for (u32 k = 0; k < ns && !wide; k++) { // (a wide side's one column is its ids, part of the run's view)
        const u64 n = recv[(size_t)k * W + me];
        for (u32 c = 0; c < ncols[k]; c++) {
            qce_rowids *view = nullptr;
            if (qce_rowids_from_window(col_off[(col_at + c) * W + me] / 4, n, 0, sides[k]->attached[c]->id_bound, 0, &view) != 0) {
                qcecomm::abort_all();
                return -1;
            }
            cx().recv_cols.push_back({sides[k]->attached[c], view});
        }
        (*out)[k].travelled = ncols[k] != 0;
        col_at += ncols[k];
    }
    dist_out->kind = Dist::KEYS;
    dist_out->key_bits = key_bits;
    dist_out->split.assign(splitters.begin(), splitters.begin() + (W - 1));
    dist_out->wide = wide;
    dist_out->base = base;
    return 0;
}

bool splitters_fit(const Dist &d, int key_bits, bool wide = false, u64 base = 0)
{
    if (d.kind != Dist::KEYS || d.wide != wide || d.base != base || d.key_bits != key_bits || d.split.size() + 1 != G.world)
        return false;
    const int shift = key_bits > 8 ? key_bits - 8 : 0;
    for (u64 s : d.split)
        if (!on_bin_boundary(s, shift)) return false;
    return true;
}
// a wide exchange's layout holds every key of [gmin, gmax]: its bins cover them
bool wide_range_fits(const Dist &d, u64 gmin, u64 gmax)
{
    return d.kind == Dist::KEYS && d.wide && d.split.size() + 1 == G.world && d.base <= gmin &&
           bitlen(gmax - d.base) <= d.key_bits;
}

// the smallest and largest key of a run on this rank, as {~min, max} (packed words: the key is the high half)
int local_key_range(const qce_tuples *t, uint64_t *v)
{
    if (t->n == 0) return 0;
    CK(cudaMemsetAsync(cx().d_scalars + 8, 0, 2 * sizeof(u64), cx().stream));
    LAUNCH("key_range", k_minmax_u64, grid_for(512, t->n, 4), 256, 0, (const u64 *)t->a, t->n, cx().d_scalars + 8);
    if (read_scalars(10) != 0) return -1;
    const int drop = t->wide ? 0 : 32;
    v[0] = std::max<uint64_t>(v[0], ~(~cx().h_scalars[8] >> drop));
    v[1] = std::max<uint64_t>(v[1], cx().h_scalars[9] >> drop);
    return 0;
}
// ... over both runs and all ranks: one all-reduce of two words
int global_key_range(const qce_tuples *R, const qce_tuples *S, u64 *gmin, u64 *gmax)
{
    uint64_t v[2] = {0, 0};
    if (local_key_range(R, v) != 0 || local_key_range(S, v) != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::allreduce_max(v, 2));
    *gmin = ~v[0];
    *gmax = v[1];
    return 0;
}

// a packed run as a wide one (12 B per tuple), for a join whose other side has keys >= 2^32
int widen(const qce_tuples *in, qce_tuples **out)
{
    qce_tuples *t = new qce_tuples();
    t->n = in->n;
    t->n_others = in->n_others;
    t->wide = true;
    t->key_bits = in->key_bits;
    t->key_min = in->key_min;
    t->key_max = in->key_max;
    t->id_bound = in->id_bound;
    t->sorted = false;
    t->sort_pending = in->sort_pending;
    t->dist.kind = Dist::ANY;
    if (dalloc(&t->a, t->n) != 0 || dalloc(&t->ids, t->n) != 0) { qce_tuples_free(t); return -1; }
    if (t->n) LAUNCH("widen", k_unpack_wide, grid_for(2048, t->n), 256, 0, (const u64 *)in->a, t->n, t->a, t->ids);
    *out = t;
    return 0;
}

int merge_join_any(const qce_tuples *R, const qce_tuples *S, bool want_r, bool want_s, qce_rowids **outR,
                   qce_rowids **outS, bool walk);

// Sort-merge join of two distributed runs (join_relations, src/join.c:325-392).  A run whose
// sort is pending is exchanged by key range and sorted by its new owner; a run that is already
// in key order over the ranks (the output side of an earlier join on the same column) stays
// where it is and lends its splitters.  When either side has keys >= 2^32 both sides are
// exchanged wide (a packed side is widened first), binned by key - (smallest key) over the
// width of the key range.  Only the pointer walk over an unsorted run gathers on rank 0.
int sh_join_runs(qce_tuples *R, qce_tuples *S, bool want_r, bool want_s, qce_rowids **outR, qce_rowids **outS, bool walk)
{
    if (outR) *outR = nullptr;
    if (outS) *outS = nullptr;
    const bool root_only = walk, wide = R->wide || S->wide;
    int rc = -1;
    qce_tuples *lr = nullptr, *ls = nullptr;  // the local inputs of the merge
    bool own_r = false, own_s = false, travelled_r = false, travelled_s = false;
    int trace_bits = std::max(R->key_bits, S->key_bits);
    Dist dist;
    dist.kind = Dist::ANY;
    if (root_only && (!R->attached.empty() || !S->attached.empty())) {
        qcecomm::abort_all();
        return fail("position-carrying runs cannot take the rank-0 fallback");
    }
    if (wide && (!R->attached.empty() || !S->attached.empty())) {
        qcecomm::abort_all();
        return fail("position-carrying runs need keys below 2^32 on both sides");
    }
    if (R->n + R->n_others == 0 || S->n + S->n_others == 0) {
        // an empty side: the pointer walk never starts (src/join.c:342), whatever the other side holds
        qce_tuples empty_r = *R, empty_s = *S;
        empty_r.n = 0; empty_s.n = 0;
        empty_r.hist256 = nullptr; empty_s.hist256 = nullptr;
        LocalScope ls_;
        rc = merge_join_any(&empty_r, &empty_s, want_r, want_s, outR, outS, false);
    } else if (root_only) {
        if (tuples_to_root(R, &lr) != 0 || tuples_to_root(S, &ls) != 0) { qce_tuples_free(lr); qce_tuples_free(ls); return -1; }
        own_r = own_s = true;
        LocalScope ls_;
        if ((R->sort_pending && qce_sort_tuples(lr) != 0) || (S->sort_pending && qce_sort_tuples(ls) != 0)) {
            qcecomm::abort_all();
        } else {
            rc = merge_join_any(lr, ls, want_r, want_s, outR, outS, walk);
        }
    } else {
        int key_bits = std::max(R->key_bits, S->key_bits);
        u64 key_max = std::max(R->key_max, S->key_max), base = 0;
        bool push_r = R->sort_pending, push_s = S->sort_pending;
        if (wide) {
            u64 gmin, gmax;
            if (global_key_range(R, S, &gmin, &gmax) != 0) return -1;
            key_max = gmax;
            // a side in place on a wide layout that covers every key lends its base and width
            const Dist *in_place = !push_r && wide_range_fits(R->dist, gmin, gmax) ? &R->dist
                                 : !push_s && wide_range_fits(S->dist, gmin, gmax) ? &S->dist : nullptr;
            base = in_place ? in_place->base : gmin;
            key_bits = in_place ? in_place->key_bits : std::max(1, bitlen(gmax - gmin));
        }
        trace_bits = key_bits;
        // a side that claims to be in place must really be laid out on this exchange's bins
        if (!push_r && !splitters_fit(R->dist, key_bits, wide, base)) push_r = true;
        if (!push_s && !splitters_fit(S->dist, key_bits, wide, base)) push_s = true;
        if (!push_r && !push_s && R->dist.split != S->dist.split) push_s = true;
        const Dist *fixed = !push_r ? &R->dist : (!push_s ? &S->dist : nullptr);
        // a packed side of a wide join is pushed (its layout cannot fit) and travels widened
        qce_tuples *wr = nullptr, *ws = nullptr;
        if (wide && ((!R->wide && widen(R, &wr) != 0) || (!S->wide && widen(S, &ws) != 0))) {
            qce_tuples_free(wr);
            qcecomm::abort_all();
            return -1;
        }
        std::vector<const qce_tuples *> sides;
        if (push_r) sides.push_back(wr ? wr : R);
        if (push_s) sides.push_back(ws ? ws : S);
        std::vector<XRecv> got;
        int xrc = 0;
        if (sides.empty()) dist = R->dist;
        else xrc = exchange_runs(sides, key_bits, key_max, fixed, &got, &dist, true, wide ? &base : nullptr);
        qce_tuples_free(wr); // the received copies live in the window
        qce_tuples_free(ws);
        if (xrc != 0) return -1;
        size_t at = 0;
        if (push_r) { travelled_r = got[at].travelled; lr = got[at++].run; } else lr = R;
        if (push_s) { travelled_s = got[at].travelled; ls = got[at++].run; } else ls = S;
        own_r = push_r;
        own_s = push_s;
        LocalScope ls_; // the received runs were sorted inside the exchange
        rc = merge_join_any(lr, ls, want_r, want_s, outR, outS, false);
    }
    static const bool trace = getenv("QCE_TRACE") != nullptr;
    if (trace) // route "local": a side is empty everywhere, nothing moves
        fprintf(stderr, "[qce] join rank %u/%u: route=%s keys=%s width=%d recv R=%llu/%llu S=%llu/%llu\n", G.rank, G.world,
                !lr ? "local" : root_only ? "root" : "exchange", wide ? "wide" : "packed", trace_bits,
                (unsigned long long)(lr ? lr->n : 0), (unsigned long long)(R->n + R->n_others), (unsigned long long)(ls ? ls->n : 0),
                (unsigned long long)(S->n + S->n_others));
    if (own_r) qce_tuples_free(lr);
    if (own_s) qce_tuples_free(ls);
    if (rc != 0) { qcecomm::abort_all(); return -1; }
    // the pairs every rank produced; the outputs are in key order over the ranks
    qce_rowids *outs[2] = {outR ? *outR : nullptr, outS ? *outS : nullptr};
    const qce_tuples *src[2] = {R, S};
    uint64_t v = outs[0] ? outs[0]->n : (outs[1] ? outs[1]->n : 0);
    const u64 local = v;
    CQ(qcecomm::allreduce_sum(&v, 1));
    const bool travelled[2] = {travelled_r, travelled_s};
    for (int k = 0; k < 2; k++) {
        if (!outs[k]) continue;
        if (travelled[k]) outs[k]->attach_gen = cx().attach_gen;
        outs[k]->n_others = v - local;
        outs[k]->dist = dist;
        outs[k]->dist.rel = src[k]->src_rel;
        outs[k]->dist.col = src[k]->src_col;
        if (dist.kind != Dist::KEYS) outs[k]->dist.kind = Dist::ANY;
    }
    return 0;
}

// ---- the operators -----------------------------------------------------------------------------
int own_rows_of(const Column *cl, u64 *begin, u64 *count)
{
    if (cl->windowed) { *begin = cl->win_begin; *count = cl->win_count; }
    else row_share(cl->n, G.rank, G.world, begin, count);
    return 0;
}

int sh_filter_scan(uint32_t rel, uint32_t col, char op, uint64_t c, qce_rowids **out)
{
    const Column *cl;
    if (get_column(rel, col, &cl) != 0) { qcecomm::abort_all(); return -1; }
    u64 begin, count;
    own_rows_of(cl, &begin, &count);
    {
        LocalScope ls;
        if (qce_filter_scan_range(rel, col, op, c, begin, count, out) != 0) { qcecomm::abort_all(); return -1; }
    }
    (*out)->dist.kind = Dist::ROWS;
    (*out)->dist.rel = rel;
    return others_of((*out)->n, &(*out)->n_others);
}

int sh_filter_refine(qce_rowids *ids, uint32_t rel, uint32_t col, char op, uint64_t c, uint64_t *survivors)
{
    {
        LocalScope ls;
        if (qce_filter_refine(ids, rel, col, op, c, nullptr) != 0) { qcecomm::abort_all(); return -1; }
    }
    if (others_of(ids->n, &ids->n_others) != 0) return -1;
    if (survivors) *survivors = ids->n + ids->n_others;
    return 0;
}

int sh_build_base(uint32_t rel, uint32_t col, qce_tuples **out)
{
    const Column *cl;
    if (get_column(rel, col, &cl) != 0) { qcecomm::abort_all(); return -1; }
    u64 begin, count;
    own_rows_of(cl, &begin, &count);
    {
        LocalScope ls;
        if (qce_build_tuples_base_range(rel, col, begin, count, out) != 0) { qcecomm::abort_all(); return -1; }
    }
    (*out)->n_others = cl->n - count;
    (*out)->dist.kind = Dist::ROWS;
    (*out)->dist.rel = rel;
    return 0;
}

int sh_build_rowids(uint32_t rel, uint32_t col, const qce_rowids *ids, qce_tuples **out)
{
    {
        LocalScope ls;
        if (qce_build_tuples_rowids(rel, col, ids, out) != 0) { qcecomm::abort_all(); return -1; }
    }
    (*out)->n_others = ids->n_others;
    if (ids->dist.kind == Dist::KEYS && ids->dist.rel == rel && ids->dist.col == col) (*out)->dist = ids->dist;
    else (*out)->dist.kind = Dist::ANY;
    return 0;
}

// in key order over the ranks?  (the reference never checks; the host layer asks before it trusts
// a JOIN_SORT_* decision, SURVEY.md 8a-10)
int sh_is_sorted(const qce_tuples *t, int *sorted)
{
    int local = 1;
    uint64_t edge[4] = {0, 0, 0, 0}; // first key, last key, n, locally unsorted
    {
        LocalScope ls;
        if (qce_tuples_is_sorted(t, &local) != 0) { qcecomm::abort_all(); return -1; }
    }
    if (t->n) {
        u64 w[2];
        CK(cudaMemcpyAsync(&w[0], t->a, 8, cudaMemcpyDeviceToHost, cx().stream));
        CK(cudaMemcpyAsync(&w[1], t->a + (t->n - 1), 8, cudaMemcpyDeviceToHost, cx().stream));
        CK(cudaStreamSynchronize(cx().stream));
        edge[0] = t->wide ? w[0] : w[0] >> 32;
        edge[1] = t->wide ? w[1] : w[1] >> 32;
    }
    edge[2] = t->n;
    edge[3] = local ? 0 : 1;
    std::vector<uint64_t> all((size_t)G.world * 4);
    CQ(qcecomm::allgather(edge, sizeof edge, all.data()));
    bool ok = true, have = false;
    u64 prev = 0;
    for (u32 r = 0; r < G.world; r++) {
        const uint64_t *e = &all[(size_t)r * 4];
        if (e[3]) ok = false;
        if (e[2] == 0) continue;
        if (have && e[0] < prev) ok = false;
        prev = e[1];
        have = true;
    }
    *sorted = ok ? 1 : 0;
    return 0;
}

int distinct_pairs(const qce_rowids *pr, const qce_rowids *ps, qce_rowids **dr, qce_rowids **ds);
int sh_distinct_pairs(const qce_rowids *pr, const qce_rowids *ps, qce_rowids **dr, qce_rowids **ds)
{
    // a duplicate (rowid_R, rowid_S) pair carries one key, so both copies live on the rank that
    // owns the key: the distinct pairs of the whole output are the ranks' distinct pairs
    if (distinct_pairs(pr, ps, dr, ds) != 0) { qcecomm::abort_all(); return -1; }
    (*dr)->dist.kind = Dist::ANY;
    (*ds)->dist.kind = Dist::ANY;
    if (others_of((*dr)->n, &(*dr)->n_others) != 0) return -1;
    (*ds)->n_others = (*dr)->n_others;
    return 0;
}

// qce_merge_join_stats over the ranks: min / max matches per outer tuple, all-reduced
int sh_merge_join_stats(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS, uint32_t *lo, uint32_t *hi)
{
    u32 st[2] = {0xffffffffu, 0u};
    tl_join_stats = st; // filled by the local merge when both of this rank's runs are non-empty
    const int rc = sh_join_runs(const_cast<qce_tuples *>(R), const_cast<qce_tuples *>(S), true, true, outR, outS, false);
    tl_join_stats = nullptr;
    if (rc != 0) return -1;
    uint64_t v[2] = {(uint64_t)(0xffffffffu - st[0]), st[1]}; // min as a max
    CQ(qcecomm::allreduce_max(v, 2));
    *lo = 0xffffffffu - (u32)v[0];
    *hi = (u32)v[1];
    if (*lo == 0xffffffffu) *lo = 0; // no rank merged anything
    return 0;
}

int sh_merge_join(const qce_tuples *R, const qce_tuples *S, qce_rowids **outR, qce_rowids **outS,
                  qce_rowids **distinctR, qce_rowids **distinctS, bool walk)
{
    if (sh_join_runs(const_cast<qce_tuples *>(R), const_cast<qce_tuples *>(S), true, true, outR, outS, walk) != 0) return -1;
    if (distinctR || distinctS) {
        qce_rowids *dr = nullptr, *ds = nullptr;
        if (sh_distinct_pairs(*outR, *outS, &dr, &ds) != 0) return -1;
        if (distinctR) *distinctR = dr; else qce_rowids_free(dr);
        if (distinctS) *distinctS = ds; else qce_rowids_free(ds);
    }
    return 0;
}

// scan_join, src/join.c:395-423: positional.  Two columns of the same entity have the same
// shape on every rank; columns of different entities are first cut alike.
int scan_join_impl(const Column *cr, const qce_rowids *idsR, const Column *cs, const qce_rowids *idsS,
                   qce_rowids **outR, qce_rowids **outS);
int sh_scan_join(const Column *cr, const qce_rowids *idsR, const Column *cs, const qce_rowids *idsS, qce_rowids **outR,
                 qce_rowids **outS)
{
    uint64_t differ = idsR->n != idsS->n ? 1 : 0;
    CQ(qcecomm::allreduce_max(&differ, 1));
    qce_rowids *cut = nullptr;
    if (differ) {
        std::vector<u64> target;
        if (all_counts(idsR->n, &target) != 0) return -1;
        if (realign_rowids(idsS, target, &cut) != 0) return -1;
    }
    if (scan_join_impl(cr, idsR, cs, cut ? cut : idsS, outR, outS) != 0) { qcecomm::abort_all(); return -1; }
    if (cut) qce_rowids_free(cut);
    (*outR)->dist = idsR->dist;
    (*outS)->dist = differ ? Dist() : idsS->dist;
    if (differ) (*outS)->dist.kind = Dist::ANY;
    if (others_of((*outR)->n, &(*outR)->n_others) != 0) return -1;
    (*outS)->n_others = (*outR)->n_others;
    return 0;
}
int sh_scan_join_base(const Column *cr, const Column *cs, qce_rowids **outR, qce_rowids **outS)
{
    // position i pairs row i of both relations: this rank takes the positions of its share of R
    u64 begin, count;
    own_rows_of(cr, &begin, &count);
    const u64 lim = std::min(cr->n, cs->n);
    if (begin > lim) begin = lim;
    if (begin + count > lim) count = lim - begin;
    qce_rowids *pos = nullptr;
    {
        LocalScope ls;
        if (qce_rowids_iota(begin, count, (u32)cr->n, &pos) != 0) { qcecomm::abort_all(); return -1; }
    }
    const int rc = scan_join_impl(cr, pos, cs, pos, outR, outS);
    qce_rowids_free(pos);
    if (rc != 0) { qcecomm::abort_all(); return -1; }
    (*outR)->dist.kind = Dist::ANY; // ascending positions; which relation's rows they are is the caller's knowledge
    (*outS)->dist.kind = Dist::ANY;
    if (others_of((*outR)->n, &(*outR)->n_others) != 0) return -1;
    (*outS)->n_others = (*outR)->n_others;
    return 0;
}

// join_payloads, src/join.c:426-484: R' = (key = last[i], payload = edit[i]) positionally,
// S' = (key = driver[j]); both sorted by key -- a row id -- and merged.  Sharded: the two
// runs are exchanged by row-id range like any other join input.
int sh_rejoin(const qce_rowids *driver, const qce_rowids *last, const qce_rowids *edit, qce_rowids **out)
{
    if (edit->n + edit->n_others < last->n + last->n_others) {
        qcecomm::abort_all();
        return fail("bystander column has %llu row ids but its entity's joined column has %llu "
                    "(the reference reads past the array here, src/join.c:433)",
                    (unsigned long long)(edit->n + edit->n_others), (unsigned long long)(last->n + last->n_others));
    }
    uint64_t differ = edit->n != last->n ? 1 : 0;
    CQ(qcecomm::allreduce_max(&differ, 1));
    qce_rowids *cut = nullptr;
    if (differ) {
        std::vector<u64> target;
        if (all_counts(last->n, &target) != 0) return -1;
        if (realign_rowids(edit, target, &cut) != 0) return -1;
    }
    const qce_rowids *ed = cut ? cut : edit;
    const int bits = last->id_bound ? bitlen(last->id_bound - 1) : 32;
    qce_tuples R, S;
    R.n = last->n; R.n_others = last->n_others; R.wide = false; R.ids = nullptr; R.key_bits = bits ? bits : 1;
    R.key_min = 0; R.key_max = last->id_bound ? last->id_bound - 1 : 0xffffffffull; R.id_bound = edit->id_bound; R.sorted = false;
    R.a = nullptr; R.sort_pending = true;
    S.n = driver->n; S.n_others = driver->n_others; S.wide = false; S.ids = nullptr; S.key_bits = R.key_bits;
    S.key_min = 0; S.key_max = R.key_max; S.id_bound = 0; S.sorted = false; S.a = nullptr; S.sort_pending = true;
    int rc = -1;
    if (dalloc(&R.a, R.n) == 0 && dalloc(&S.a, S.n) == 0) {
        cudaError_t e = cudaSuccess;
        if (R.n) { k_pack_pairs<<<grid_for(256, R.n), 256, 0, cx().stream>>>(last->d, ed->d, R.n, R.a); e = cudaGetLastError(); cx().launches++; }
        if (e == cudaSuccess && S.n) { k_pack_pairs<<<grid_for(256, S.n), 256, 0, cx().stream>>>(driver->d, (const u32 *)nullptr, S.n, S.a); e = cudaGetLastError(); cx().launches++; }
        if (e == cudaSuccess) rc = 0;
        else fail("pack_pairs: %s", cudaGetErrorString(e));
    }
    if (rc != 0) { qcecomm::abort_all(); dfree(R.a); dfree(S.a); if (cut) qce_rowids_free(cut); return -1; }
    rc = sh_join_runs(&R, &S, true, false, out, nullptr, false);
    dfree(R.a);
    dfree(S.a);
    dfree(R.hist256);
    dfree(S.hist256);
    if (cut) qce_rowids_free(cut);
    if (rc == 0) (*out)->dist.kind = Dist::ANY; // ordered by the joined column's row ids, not by a join key
    return rc;
}

// print_sums, src/utilities.c:215-219.  Rows that live on another rank are not fetched: their
// ids are pushed to the rank that owns the rows (k_push<u32>), summed there, and the uint64
// sums are added up over the ranks (exact: addition mod 2^64 is associative and commutative).
int sh_checksum(const qce_rowids *ids, uint32_t rel, const uint32_t *cols, uint32_t ncols, uint64_t *sums)
{
    const Column *cl;
    if (get_column(rel, cols[0], &cl) != 0) { qcecomm::abort_all(); return -1; }
    bool local = !cl->windowed || (ids->dist.kind == Dist::ROWS && ids->dist.rel == rel);
    for (u32 k = 1; k < ncols && local; k++) {
        const Column *ck;
        if (get_column(rel, cols[k], &ck) != 0) { qcecomm::abort_all(); return -1; }
        if (ck->windowed != cl->windowed) local = cl->windowed ? local : !ck->windowed;
    }
    int rc;
    if (local) {
        LocalScope ls;
        rc = qce_checksum(ids, rel, cols, ncols, sums);
    } else {
        const u32 W = G.world, me = G.rank;
        const u32 per = cl->rpr;
        std::vector<uint64_t> hist(W), all((size_t)W * W);
        if (qce_rowids_bin_histogram(ids, per, per, 1, W, hist.data()) != 0) { qcecomm::abort_all(); return -1; }
        CQ(qcecomm::allgather(hist.data(), W * sizeof(uint64_t), all.data()));
        std::vector<uint64_t> offs(W);
        uint64_t view_off = 0, view_cnt = 0, need = 0, sent = 0;
        if (qce_rowid_push_plan(all.data(), W, me, 1, 1, offs.data(), &view_off, &view_cnt, &need, &sent) != 0) { qcecomm::abort_all(); return -1; }
        if (ensure_window(need) != 0) return -1;
        if (qce_push_rowids(ids, per, per, 1, W, offs.data()) != 0) { qcecomm::abort_all(); return -1; }
        if (fence_barrier() != 0) return -1;
        qce_rowids *view = nullptr;
        if (qce_rowids_from_window(view_off, view_cnt, (u32)cl->win_begin, (u32)(cl->win_begin + cl->win_count), 0, &view) != 0) { qcecomm::abort_all(); return -1; }
        {
            LocalScope ls;
            rc = qce_checksum(view, rel, cols, ncols, sums);
        }
        qce_rowids_free(view);
    }
    if (rc != 0) { qcecomm::abort_all(); return -1; }
    CQ(qcecomm::allreduce_sum(sums, ncols));
    return 0;
}

} // namespace
