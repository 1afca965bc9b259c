// k_join.cuh -- sort-merge equi-join of two key-sorted tuple runs, and the
// projection checksum.
//
// Replaces join_relations (src/join.c:325-392), the merge loop of join_payloads
// (src/join.c:447-476) and print_sums' gather-sum (src/utilities.c:215-219).
//
// The reference walks both runs with one serial pointer pair and pushes one
// calloc'ed element per match.  Here the join is two-phase (count, write):
//   partition  one thread per tile of 2048 R tuples binary-searches the window
//              of S that the tile's key range can touch
//   bounds     per tile: stage the S window in shared memory, every R tuple
//              finds lower/upper bound of its key there (or in global memory
//              when the window is larger than the staging buffer); writes
//              lb[i], cnt[i] and the tile's pair total
//   scan       exclusive scan of tile totals -> output offsets; the same scan
//              over ceil(total/4096) gives a work list of <=4096-pair chunks
//   write      one CTA per chunk (load-balanced: a skewed key that produces
//              millions of pairs is split over many CTAs): rebuilds the tile's
//              offsets in shared memory, maps every output slot back to its R
//              tuple by binary search and writes (rowid_R, rowid_S) coalesced.
// Output order is the reference's: R-major, S in run order inside a key group.
//
// Algorithmic HBM bytes: 8 B (packed) per input tuple for the bounds pass,
// 8 B per R tuple for lb/cnt (written then re-read), 8 B per output pair.
#pragma once
#include "qce_common.cuh"

#define QCE_JTILE 2048     // R tuples per tile (256 threads x 8)
#define QCE_JTHREADS 256
#define QCE_JWIN 4096      // S window staged in shared memory (keys, 32 KB dynamic = the count table's size:
                           // 64 KB capped the kernel at 3 CTAs/SM, 37 % occupancy, ncu profiles/ncu_summary_r1b.json)
#define QCE_JCHUNK 4096    // output pairs per write CTA

template <bool WIDE>
__device__ __forceinline__ u32 lower_bound_g(const TupleView &t, u32 lo, u32 hi, u64 key)
{
    while (lo < hi) {
        u32 mid = lo + ((hi - lo) >> 1);
        if (tv_key<WIDE>(t, mid) < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
template <bool WIDE>
__device__ __forceinline__ u32 upper_bound_g(const TupleView &t, u32 lo, u32 hi, u64 key)
{
    while (lo < hi) {
        u32 mid = lo + ((hi - lo) >> 1);
        if (tv_key<WIDE>(t, mid) <= key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// lower / upper bound of `key` in the sorted run S[lo, hi), starting from a guess g in [lo, hi):
// gallop away from the guess (steps 1, 2, 4, ...) until the answer is bracketed, then bisect the
// bracket.  With a good guess this is two or three probes in one or two neighbouring sectors where
// the plain bisection of a 10^5-tuple window is ~17 dependent misses -- the case of a selective
// filter on the outer side of a key / foreign-key join, whose tiles span windows far larger than
// the count table or the staging buffer can hold.
template <bool WIDE, bool UPPER>
__device__ __forceinline__ u32 bound_from_guess(const TupleView &t, u32 lo, u32 hi, u32 g, u64 key)
{
    // invariant: every index < lo is "left" (key' < key, or <= for UPPER), every index >= hi is not
#define QCE_LEFT(i) (UPPER ? (tv_key<WIDE>(t, (i)) <= key) : (tv_key<WIDE>(t, (i)) < key))
    if (lo >= hi) return lo;
    if (QCE_LEFT(g)) {
        lo = g + 1;
        for (u32 step = 1;; step <<= 1) {
            const u32 q = lo + step - 1;
            if (q >= hi || q < lo) break;
            if (QCE_LEFT(q)) lo = q + 1;
            else { hi = q; break; }
        }
    } else {
        hi = g;
        for (u32 step = 1;; step <<= 1) {
            if (step == 0 || hi - lo < step) break;
            const u32 q = hi - step;
            if (!QCE_LEFT(q)) hi = q;
            else { lo = q + 1; break; }
        }
    }
    while (lo < hi) {
        const u32 mid = lo + ((hi - lo) >> 1);
        if (QCE_LEFT(mid)) lo = mid + 1;
        else hi = mid;
    }
#undef QCE_LEFT
    return lo;
}
// [lb, ub) of `key` in the window S[w.x, w.y) whose first and last keys are ks0 <= ks1: the guess
// interpolates the key's position between them (exact for a dense key column); scale = (wn - 1) /
// (ks1 - ks0), computed once per tile.  Windows below QCE_JINTERP_MIN tuples are bisected as before: they
// stay in L1 / L2 while a tile's 2048 lookups run over them (a conservative threshold: on config 3, whose
// windows are small, the two searches measured the same).
// (not inlined: the rare path of the join kernels, and inlined its registers cost the common path spills)
// Returns lb | ub << 32.
#define QCE_JINTERP_MIN 65536u
template <bool WIDE>
__device__ __noinline__ u64 window_bounds_g(TupleView S, uint2 w, u64 ks0, u64 ks1, double scale, u64 key)
{
    u32 lb, ub;
    if (key < ks0) return (u64)w.x | ((u64)w.x << 32);
    if (key > ks1) return (u64)w.y | ((u64)w.y << 32);
    const u32 wn = w.y - w.x;
    if (wn < QCE_JINTERP_MIN) {
        lb = lower_bound_g<WIDE>(S, w.x, w.y, key);
        ub = upper_bound_g<WIDE>(S, lb, w.y, key);
    } else {
        const u32 g = w.x + min(wn - 1, (u32)((double)(key - ks0) * scale));
        lb = bound_from_guess<WIDE, false>(S, w.x, w.y, g, key);
        ub = bound_from_guess<WIDE, true>(S, lb, w.y, min(lb, w.y - 1), key);
    }
    return (u64)lb | ((u64)ub << 32);
}

// One thread per R tile: the S window [lo, hi) its key range can match.
template <bool WR, bool WS>
__global__ void __launch_bounds__(256)
k_join_partition(TupleView R, u32 nR, TupleView S, u32 nS, u32 ntiles, uint2 *__restrict__ win)
{
    u32 t = blockIdx.x * 256 + threadIdx.x;
    if (t >= ntiles) return;
    u32 first = t * QCE_JTILE;
    u32 last = min(first + QCE_JTILE, nR) - 1;
    u64 klo = tv_key<WR>(R, first), khi = tv_key<WR>(R, last);
    u32 lo = lower_bound_g<WS>(S, 0, nS, klo);
    u32 hi = upper_bound_g<WS>(S, lo, nS, khi);
    win[t] = make_uint2(lo, hi);
}

#define QCE_JSMEM_BYTES (QCE_JWIN * sizeof(u64))

// Branch-light lower/upper bound over the staged window (fixed trip count for a
// window of <= QCE_JWIN slots; the lanes of a warp stay converged).
template <bool LT> __device__ __forceinline__ u32 bound_s(const u64 *skeys, u32 wn, u64 key)
{
    u32 lo = 0, len = wn;
#pragma unroll 1
    while (len > 0) {
        const u32 half = len >> 1;
        const u64 v = skeys[lo + half];
        const bool right = LT ? (v < key) : (v <= key);
        lo = right ? lo + half + 1 : lo;
        len = right ? len - half - 1 : half;
    }
    return lo;
}

// Per R tile (2048 sorted tuples, S window [w.x, w.y)):
//  * table path -- the tile's keys span at most QCE_JTAB integer values (both runs
//    are sorted, so this is the common case: consecutive tuples have close keys):
//    the S window is histogrammed by key offset with shared-memory atomics, the
//    histogram is exclusive-scanned in place, and each R tuple's lower bound and
//    match count are two table lookups (tab[v], tab[v+1]) instead of two 12-step
//    binary searches;
//  * search path -- sparse keys: the S window (<= QCE_JWIN keys) is staged in shared
//    memory and searched; beyond that, binary search in global memory.
#define QCE_JTAB 8190     // range + 2 table entries of 4 bytes fit the 32 KB of QCE_JSMEM_BYTES
template <bool WR, bool WS>
__global__ void __launch_bounds__(QCE_JTHREADS)
k_join_bounds(TupleView R, u32 nR, TupleView S, const uint2 *__restrict__ win,
              u32 *__restrict__ lb_out, u32 *__restrict__ cnt_out, u64 *__restrict__ tile_total,
              u32 *__restrict__ tile_chunks, u32 *__restrict__ stats)
{
    extern __shared__ __align__(16) u64 skeys[]; // QCE_JSMEM_BYTES: S keys (search path) or the count table
    __shared__ u64 scratch[33];
    const int tid = threadIdx.x;
    const u32 tbase = blockIdx.x * QCE_JTILE;
    const uint2 w = win[blockIdx.x];
    const u32 wn = w.y - w.x;
    // consecutive lanes take consecutive R tuples; the 8 tuples of a thread are independent
    u64 key[QCE_JTILE / QCE_JTHREADS];
#pragma unroll
    for (int k = 0; k < QCE_JTILE / QCE_JTHREADS; k++) {
        const u32 i = tbase + k * QCE_JTHREADS + tid;
        key[k] = (i < nR) ? tv_key<WR>(R, i) : ~0ull;
    }
    const u32 last = min(tbase + QCE_JTILE, nR) - 1;
    const u64 klo = tv_key<WR>(R, tbase), khi = tv_key<WR>(R, last);
    u64 sum = 0;
    u32 cmin = 0xffffffffu, cmax = 0; // smallest / largest match count of an outer tuple (stats != nullptr: the 8f-2 test)
    if (wn == 0) {
#pragma unroll
        for (int k = 0; k < QCE_JTILE / QCE_JTHREADS; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) { lb_out[i] = w.x; cnt_out[i] = 0; cmin = 0; }
        }
    } else if (khi - klo < QCE_JTAB && wn <= 16u * QCE_JTILE) {
        // ---- table path (not for a window dominated by a heavy inner key: histogramming 2 M equal keys is
        // 2 M atomics on one shared address by ONE CTA, where two binary searches per outer tuple do)
        u32 *tab = reinterpret_cast<u32 *>(skeys); // range + 1 entries
        const u32 range = (u32)(khi - klo) + 1;
        for (u32 v = tid; v <= range; v += QCE_JTHREADS) tab[v] = 0;
        __syncthreads();
        // every key of the window lies in [klo, khi] (the window is lower_bound(klo) .. upper_bound(khi))
        for (u32 i = tid; i < wn; i += QCE_JTHREADS) atomicAdd(&tab[(u32)(tv_key<WS>(S, w.x + i) - klo)], 1u);
        __syncthreads();
        {   // exclusive scan in place; thread t owns `per` consecutive entries
            const u32 per = ((range + 1 + QCE_JTHREADS - 1) / QCE_JTHREADS) | 1u; // <= 33, odd: lane strides on distinct banks
            const u32 b0 = tid * per;
            u32 local = 0;
            for (u32 q = 0; q < per; q++)
                if (b0 + q <= range) local += tab[b0 + q];
            u32 tot32;
            u32 ex = block_scan_excl<u32, QCE_JTHREADS>(local, reinterpret_cast<u32 *>(scratch), &tot32);
            for (u32 q = 0; q < per; q++) {
                if (b0 + q <= range) {
                    const u32 c = tab[b0 + q];
                    tab[b0 + q] = ex;
                    ex += c;
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < QCE_JTILE / QCE_JTHREADS; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) {
                const u32 v = (u32)(key[k] - klo);
                const u32 lo = tab[v], c = tab[v + 1] - lo;
                lb_out[i] = w.x + lo;
                cnt_out[i] = c;
                sum += c;
                cmin = min(cmin, c);
                cmax = max(cmax, c);
            }
        }
    } else {
        const bool staged = wn <= QCE_JWIN;
        const u64 ks0 = staged ? 0ull : tv_key<WS>(S, w.x), ks1 = staged ? 0ull : tv_key<WS>(S, w.y - 1);
        const double scale = ks1 > ks0 ? (double)(wn - 1) / (double)(ks1 - ks0) : 0.0;
        if (staged) {
            for (u32 i = tid; i < wn; i += QCE_JTHREADS) skeys[i] = tv_key<WS>(S, w.x + i);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < QCE_JTILE / QCE_JTHREADS; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) {
                u32 lb, ub;
                if (staged) {
                    lb = bound_s<true>(skeys, wn, key[k]) + w.x;
                    ub = bound_s<false>(skeys, wn, key[k]) + w.x;
                } else {
                    // a window too large to stage: R is sparse against S (a selective filter), or one key is very heavy
                    const u64 b2 = window_bounds_g<WS>(S, w, ks0, ks1, scale, key[k]);
                    lb = (u32)b2;
                    ub = (u32)(b2 >> 32);
                }
                lb_out[i] = lb;
                cnt_out[i] = ub - lb;
                sum += ub - lb;
                cmin = min(cmin, ub - lb);
                cmax = max(cmax, ub - lb);
            }
        }
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cmin = min(cmin, __shfl_xor_sync(QCE_FULL_MASK, cmin, o));
            cmax = max(cmax, __shfl_xor_sync(QCE_FULL_MASK, cmax, o));
        }
        if ((tid & 31) == 0) {
            atomicMin(&stats[0], cmin);
            atomicMax(&stats[1], cmax);
        }
    }
    u64 tot = block_sum<u64, QCE_JTHREADS>(sum, scratch);
    if (tid == 0) {
        tile_total[blockIdx.x] = tot;
        tile_chunks[blockIdx.x] = (u32)((tot + QCE_JCHUNK - 1) / QCE_JCHUNK);
    }
}

// ---- single pass: bounds and pairs in one kernel ------------------------------------------------
// The two-phase join above reads both runs twice and round-trips lb/cnt through HBM (3.6 GB for
// config 2's 150 M input tuples and 50 M pairs, where the runs and the pairs are 1.6 GB).  The only
// thing phase 2 waits for is each tile's output offset -- a prefix sum over the tiles' pair totals.
// Here the tiles are claimed in order through a ticket and a tile gets its offset from a decoupled
// look-back over per-tile status words (flag | total in one 64-bit word, so a relaxed load either
// sees nothing or the value), then writes its pairs straight from the registers that hold its
// bounds.  The host sizes the outputs with a guess (`cap`); a tile that would cross it, or that
// produces more than QCE_JFUSE_MAX pairs (a heavy key: its pairs are better spread over many CTAs),
// stores lb/cnt instead and leaves its pairs to k_join_write's chunks (tile_chunks[t] > 0).
// Output order is unchanged: R-major, S in run order inside a key group.
#define QCE_JFUSE_MAX 16384u
#define QCE_JST_AGG (1ull << 62)   // the tile's own total
#define QCE_JST_INCL (2ull << 62)  // total of this tile and every tile before it
#define QCE_JST_VAL ((1ull << 62) - 1)
#define QCE_JLOOK 1                // windows of 32 predecessors polled per round trip of the look-back (see below)
template <bool WR, bool WS, bool WRITE_R, bool WRITE_S, int MIN_CTAS>
__global__ void __launch_bounds__(QCE_JTHREADS, MIN_CTAS)
k_join_fused(TupleView R, u32 nR, TupleView S, const uint2 *__restrict__ win, u32 ntiles, u32 *__restrict__ ticket,
             u64 *__restrict__ status, u64 cap, u32 *__restrict__ outR, u32 *__restrict__ outS,
             u32 *__restrict__ lb_out, u32 *__restrict__ cnt_out, u64 *__restrict__ tile_off,
             u32 *__restrict__ tile_chunks, u64 *__restrict__ total_out, u64 *__restrict__ deferred_chunks,
             u32 *__restrict__ stats)
{
    constexpr int PER = QCE_JTILE / QCE_JTHREADS;
    extern __shared__ __align__(16) u64 skeys[]; // QCE_JSMEM_BYTES: count table or staged S keys, then offsets / lb / row ids
    __shared__ u64 scratch[33];
    __shared__ u32 s_tile;
    __shared__ u64 s_gbase;
    const int tid = threadIdx.x, lane = tid & 31;
    // tiles in start order (the ticket): a look-back only ever waits for tiles that are resident or done,
    // whatever order the CTAs are dispatched in.  Without a ticket the tile is blockIdx.x.
    if (ticket) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
    }
    const u32 t = ticket ? s_tile : blockIdx.x;
    const u32 tbase = t * QCE_JTILE;
    const uint2 w = win[t];
    const u32 wn = w.y - w.x;
    u64 key[PER];
    u32 lo[PER], c[PER];
#pragma unroll
    for (int k = 0; k < PER; k++) {
        const u32 i = tbase + k * QCE_JTHREADS + tid;
        key[k] = (i < nR) ? tv_key<WR>(R, i) : ~0ull;
        lo[k] = w.x;
        c[k] = 0;
    }
    const u32 last = min(tbase + QCE_JTILE, nR) - 1;
    const u64 klo = tv_key<WR>(R, tbase), khi = tv_key<WR>(R, last);
    if (wn == 0) {
        // nothing in S inside the tile's key range
    } else if (khi - klo < QCE_JTAB && wn <= 16u * QCE_JTILE) {
        u32 *tab = reinterpret_cast<u32 *>(skeys);
        const u32 range = (u32)(khi - klo) + 1;
        for (u32 v = tid; v <= range; v += QCE_JTHREADS) tab[v] = 0;
        __syncthreads();
        for (u32 i = tid; i < wn; i += QCE_JTHREADS) atomicAdd(&tab[(u32)(tv_key<WS>(S, w.x + i) - klo)], 1u);
        __syncthreads();
        {   // exclusive scan in place; thread t owns `per` consecutive entries (odd: the lanes' strides then
            // fall on different banks)
            const u32 per = ((range + 1 + QCE_JTHREADS - 1) / QCE_JTHREADS) | 1u;
            const u32 b0 = tid * per;
            u32 local = 0;
            for (u32 q = 0; q < per; q++)
                if (b0 + q <= range) local += tab[b0 + q];
            u32 tot32;
            u32 ex = block_scan_excl<u32, QCE_JTHREADS>(local, reinterpret_cast<u32 *>(scratch), &tot32);
            for (u32 q = 0; q < per; q++) {
                if (b0 + q <= range) {
                    const u32 cc = tab[b0 + q];
                    tab[b0 + q] = ex;
                    ex += cc;
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) {
                const u32 v = (u32)(key[k] - klo);
                const u32 l = tab[v];
                lo[k] = w.x + l;
                c[k] = tab[v + 1] - l;
            }
        }
    } else if (wn <= QCE_JWIN) {
        for (u32 i = tid; i < wn; i += QCE_JTHREADS) skeys[i] = tv_key<WS>(S, w.x + i);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) {
                const u32 lb = bound_s<true>(skeys, wn, key[k]);
                lo[k] = lb + w.x;
                c[k] = bound_s<false>(skeys, wn, key[k]) - lb;
            }
        }
    } else {
        // a window too large to stage: R is sparse against S (a selective filter), or one key is very heavy.
        // The bounds go through shared memory (unused on this path): held in registers across the calls they
        // would spill.
        const u64 ks0 = tv_key<WS>(S, w.x), ks1 = tv_key<WS>(S, w.y - 1);
        const double scale = ks1 > ks0 ? (double)(wn - 1) / (double)(ks1 - ks0) : 0.0;
        u32 *tlo = reinterpret_cast<u32 *>(skeys), *tc = tlo + QCE_JTILE;
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) {
                const u64 b2 = window_bounds_g<WS>(S, w, ks0, ks1, scale, key[k]);
                tlo[k * QCE_JTHREADS + tid] = (u32)b2;
                tc[k * QCE_JTHREADS + tid] = (u32)(b2 >> 32) - (u32)b2;
            }
        }
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) { lo[k] = tlo[k * QCE_JTHREADS + tid]; c[k] = tc[k * QCE_JTHREADS + tid]; }
        }
    }
    __syncthreads(); // every lookup is done: the table's memory is reused
    u32 *soff = reinterpret_cast<u32 *>(skeys); // [QCE_JTILE] match counts, then tile-local exclusive offsets
    u32 *slo = soff + QCE_JTILE, *srid = slo + QCE_JTILE;
    u32 cmax = 0, cmin = 0xffffffffu;
#pragma unroll
    for (int k = 0; k < PER; k++) {
        soff[k * QCE_JTHREADS + tid] = c[k];
        slo[k * QCE_JTHREADS + tid] = lo[k]; // the bounds wait in shared memory for the paths that need them again
        cmax = max(cmax, c[k]);
        if (tbase + k * QCE_JTHREADS + tid < nR) cmin = min(cmin, c[k]);
    }
    __syncthreads();
    const uint4 a = reinterpret_cast<const uint4 *>(soff)[2 * tid], b = reinterpret_cast<const uint4 *>(soff)[2 * tid + 1];
    const u64 mine = (u64)a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
    u64 tot;
    const u64 ex = block_scan_excl<u64, QCE_JTHREADS>(mine, scratch, &tot);
    const bool small_tot = tot <= QCE_JFUSE_MAX;
    if (small_tot) {
        u32 x = (u32)ex;
        uint4 a2, b2;
        a2.x = x; x += a.x; a2.y = x; x += a.y; a2.z = x; x += a.z; a2.w = x; x += a.w;
        b2.x = x; x += b.x; b2.y = x; x += b.y; b2.z = x; x += b.z; b2.w = x;
        reinterpret_cast<uint4 *>(soff)[2 * tid] = a2;
        reinterpret_cast<uint4 *>(soff)[2 * tid + 1] = b2;
    }
    const int heavy = __syncthreads_or(cmax > 16u);
    // The first match of all eight tuples is fetched now, in one batch, and the fetch is in flight while
    // warp 0 publishes the tile's total and looks back for its offset (two global round trips that the
    // other warps would otherwise sit out at the barrier).
    // (the outer tuples' row ids come from L2 with them: holding them since the first read costs a CTA per SM)
    u32 sid[PER], rid[PER];
#pragma unroll
    for (int k = 0; k < PER; k++) {
        const u32 i = tbase + k * QCE_JTHREADS + tid;
        sid[k] = (WRITE_S && small_tot && !heavy && c[k]) ? tv_id<WS>(S, lo[k]) : 0u;
        rid[k] = (WRITE_R && small_tot && i < nR && (c[k] || heavy)) ? tv_id<WR>(R, i) : 0u;
    }
    if (tid < 32) {
        if (lane == 0) st_relaxed_gpu_u64(&status[t], (t == 0 ? QCE_JST_INCL : QCE_JST_AGG) | tot);
        u64 before = 0;
        if (t > 0) {
            // In steady state the tiles start a few tens of nanoseconds apart, so the nearest inclusive total is
            // ~25 tiles back and one window of 32 predecessors reaches it; what the warp waits for is the slowest of
            // those predecessors to publish its own total (ncu: 23 % of the kernel's stall samples sit at the barrier
            // behind this block).  Polling 4 windows per round trip (QCE_JLOOK 4) was measured: 0.67 -> 0.71 ms on
            // config 2 -- four times the polling traffic on the same status lines.
            int look = (int)t - 1;
            bool done = false;
            while (!done) {
                u64 v[QCE_JLOOK];
#pragma unroll
                for (int q = 0; q < QCE_JLOOK; q++) {
                    const int idx = look - q * 32 - lane;
                    v[q] = idx >= 0 ? ld_relaxed_gpu_u64(&status[idx]) : QCE_JST_INCL; // in front of tile 0: a total of zero
                }
#pragma unroll
                for (int q = 0; q < QCE_JLOOK; q++) {
                    if (done) continue; // warp-uniform
                    const int idx = look - q * 32 - lane;
                    while (__any_sync(QCE_FULL_MASK, (v[q] >> 62) == 0)) {
                        if ((v[q] >> 62) == 0) v[q] = ld_relaxed_gpu_u64(&status[idx]);
                    }
                    const u32 incl = __ballot_sync(QCE_FULL_MASK, (v[q] >> 62) == 2);
                    u64 val = v[q] & QCE_JST_VAL;
                    if (incl && lane > __ffs(incl) - 1) val = 0; // beyond the nearest inclusive total
                    before += warp_sum_u64(val);
                    done = incl != 0;
                }
                look -= QCE_JLOOK * 32;
            }
            if (lane == 0) st_relaxed_gpu_u64(&status[t], QCE_JST_INCL | (before + tot));
        }
        if (lane == 0) {
            s_gbase = before;
            if (t == ntiles - 1) *total_out = before + tot;
        }
    }
    __syncthreads();
    const u64 gbase = s_gbase;
    const bool fused = small_tot && gbase + tot <= cap;
    if (tid == 0) {
        const u32 chunks = fused ? 0u : (u32)((tot + QCE_JCHUNK - 1) / QCE_JCHUNK);
        tile_off[t] = gbase;
        tile_chunks[t] = chunks;
        if (chunks) atomicAdd(deferred_chunks, (u64)chunks);
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cmin = min(cmin, __shfl_xor_sync(QCE_FULL_MASK, cmin, o));
            cmax = max(cmax, __shfl_xor_sync(QCE_FULL_MASK, cmax, o));
        }
        if (lane == 0) {
            atomicMin(&stats[0], cmin);
            atomicMax(&stats[1], cmax);
        }
    }
    if (!fused) {
#pragma unroll
        for (int k = 0; k < PER; k++) {
            const u32 i = tbase + k * QCE_JTHREADS + tid;
            if (i < nR) { lb_out[i] = slo[k * QCE_JTHREADS + tid]; cnt_out[i] = c[k]; }
        }
        return;
    }
    if (tot == 0) return;
    if (!heavy) {
        // at most 16 matches per outer tuple: every thread writes the pairs of its own tuples; consecutive
        // lanes hold consecutive tuples, so their pairs are neighbours in the output
#pragma unroll
        for (int k = 0; k < PER; k++) {
            if (c[k]) {
                const u64 o = gbase + soff[k * QCE_JTHREADS + tid];
                if (WRITE_R) outR[o] = rid[k];
                if (WRITE_S) outS[o] = sid[k];
            }
        }
        if (__any_sync(QCE_FULL_MASK, cmax > 1u)) {
#pragma unroll
            for (int k = 0; k < PER; k++) {
                const u64 o = gbase + soff[k * QCE_JTHREADS + tid];
                const u32 l = slo[k * QCE_JTHREADS + tid];
                for (u32 q = 1; q < c[k]; q++) {
                    if (WRITE_R) outR[o + q] = rid[k];
                    if (WRITE_S) outS[o + q] = tv_id<WS>(S, l + q);
                }
            }
        }
    } else {
        // a few outer tuples carry most of the tile's pairs: one output slot per thread and step, mapped back
        // to its outer tuple by binary search over the offsets
#pragma unroll
        for (int k = 0; k < PER; k++) srid[k * QCE_JTHREADS + tid] = rid[k];
        __syncthreads();
        for (u32 o = tid; o < (u32)tot; o += QCE_JTHREADS) {
            u32 l = 0, h = QCE_JTILE; // largest e with soff[e] <= o (tuples without matches share their successor's offset)
            while (h - l > 1) {
                const u32 mid = (l + h) >> 1;
                if (soff[mid] <= o) l = mid; else h = mid;
            }
            if (WRITE_R) outR[gbase + o] = srid[l];
            if (WRITE_S) outS[gbase + o] = tv_id<WS>(S, slo[l] + (o - soff[l]));
        }
    }
}

// ---- "walk" variant: outer run R in arbitrary order, inner run S sorted -------------
// The reference's merge is one serial pointer walk (src/join.c:342-377) that it
// also runs when build_relations wrongly assumes R is already sorted
// (JOIN_SORT_RHS after the asymmetric tests of src/join.c:253-267).  With S
// sorted the walk has a closed form: s_start only ever advances to
// lower_bound(S, max of the R keys seen so far), so an R tuple matches its full
// [lb, ub) range iff its key >= every earlier R key, and nothing otherwise.
// That is a prefix-max scan plus two binary searches per tuple -- no serial walk.
template <bool WR>
__global__ void __launch_bounds__(QCE_JTHREADS)
k_tile_keymax(TupleView R, u32 nR, u64 *__restrict__ tile_max)
{
    __shared__ u64 smax[QCE_JTHREADS / 32];
    const u32 tbase = blockIdx.x * QCE_JTILE;
    u64 m = 0;
    for (int k = 0; k < QCE_JTILE / QCE_JTHREADS; k++) {
        u32 i = tbase + k * QCE_JTHREADS + threadIdx.x;
        if (i < nR) m = max(m, tv_key<WR>(R, i));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(QCE_FULL_MASK, m, o));
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < QCE_JTHREADS / 32; w++) m = max(m, smax[w]);
        tile_max[blockIdx.x] = m;
    }
}
// exclusive prefix max over the tiles; has_prev[t] = 0 for the first tile
// exclusive prefix MAXIMUM over the tiles' largest keys (one warp, 32 tiles per step: shuffles instead
// of the serial loop a single thread used to run over up to ~50 K tiles)
__global__ void __launch_bounds__(32) k_scan_excl_max(const u64 *__restrict__ tile_max, u64 *__restrict__ tile_pm, u32 ntiles)
{
    const u32 lane = threadIdx.x;
    u64 run = 0;
    for (u32 base = 0; base < ntiles; base += 32) {
        const u32 t = base + lane;
        const u64 v = t < ntiles ? tile_max[t] : 0ull;
        u64 incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u64 n = __shfl_up_sync(QCE_FULL_MASK, incl, o);
            if (lane >= (u32)o) incl = max(incl, n);
        }
        u64 excl = __shfl_up_sync(QCE_FULL_MASK, incl, 1);
        if (lane == 0) excl = 0;
        if (t < ntiles) tile_pm[t] = max(run, excl);
        run = max(run, __shfl_sync(QCE_FULL_MASK, incl, 31));
    }
}
template <bool WR, bool WS>
__global__ void __launch_bounds__(QCE_JTHREADS)
k_join_bounds_walk(TupleView R, u32 nR, TupleView S, u32 nS, const u64 *__restrict__ tile_pm,
                   u32 *__restrict__ lb_out, u32 *__restrict__ cnt_out, u64 *__restrict__ tile_total,
                   u32 *__restrict__ tile_chunks)
{
    __shared__ u64 wmax[QCE_JTHREADS / 32];
    __shared__ u64 scratch[33];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 tbase = blockIdx.x * QCE_JTILE;
    // 8 consecutive tuples per thread so that thread order == run order
    u64 key[8], local = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        u32 i = tbase + tid * 8 + k;
        key[k] = (i < nR) ? tv_key<WR>(R, i) : 0;
        local = max(local, key[k]);
    }
    // exclusive max-scan of `local` across the block
    u64 incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u64 nb = __shfl_up_sync(QCE_FULL_MASK, incl, o);
        if (lane >= o) incl = max(incl, nb);
    }
    u64 excl = __shfl_up_sync(QCE_FULL_MASK, incl, 1);
    if (lane == 0) excl = 0;
    if (lane == 31) wmax[warp] = incl;
    __syncthreads();
    u64 before = tile_pm[blockIdx.x];
    for (int w = 0; w < warp; w++) before = max(before, wmax[w]);
    before = max(before, excl);
    const bool first_thread = (blockIdx.x == 0 && tid == 0);

    u64 sum = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        u32 i = tbase + tid * 8 + k;
        if (i < nR) {
            u32 lb = 0, c = 0;
            const bool first = first_thread && k == 0; // nothing precedes the very first tuple
            if (first || key[k] >= before) {
                lb = lower_bound_g<WS>(S, 0, nS, key[k]);
                c = upper_bound_g<WS>(S, lb, nS, key[k]) - lb;
            }
            lb_out[i] = lb;
            cnt_out[i] = c;
            sum += c;
            before = max(before, key[k]);
        }
    }
    u64 tot = block_sum<u64, QCE_JTHREADS>(sum, scratch);
    if (tid == 0) {
        tile_total[blockIdx.x] = tot;
        tile_chunks[blockIdx.x] = (u32)((tot + QCE_JCHUNK - 1) / QCE_JCHUNK);
    }
}

// One CTA per <=4096-pair chunk of one R tile.
template <bool WR, bool WS, bool WRITE_R, bool WRITE_S>
__global__ void __launch_bounds__(QCE_JTHREADS)
k_join_write(TupleView R, u32 nR, TupleView S, const u32 *__restrict__ lb_in,
             const u32 *__restrict__ cnt_in, const u64 *__restrict__ tile_off,
             const u32 *__restrict__ chunk_off, u32 ntiles, u32 *__restrict__ outR,
             u32 *__restrict__ outS)
{
    __shared__ u64 soff[QCE_JTILE + 1];
    __shared__ u64 scratch[33];
    __shared__ u32 s_tile;
    const int tid = threadIdx.x;
    if (tid == 0) {
        // largest tile t with chunk_off[t] <= blockIdx.x (tiles without output
        // have zero chunks and are skipped by the search)
        u32 lo = 0, hi = ntiles;
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (chunk_off[mid] <= blockIdx.x) lo = mid; else hi = mid;
        }
        s_tile = lo;
    }
    __syncthreads();
    const u32 t = s_tile;
    const u32 chunk = blockIdx.x - chunk_off[t];
    const u32 tbase = t * QCE_JTILE;

    // tile-local exclusive offsets of the R tuples (8 consecutive per thread)
    u64 c[8], s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        u32 i = tbase + tid * 8 + k;
        c[k] = (i < nR) ? (u64)cnt_in[i] : 0ull;
        s += c[k];
    }
    u64 tot;
    u64 ex = block_scan_excl<u64, QCE_JTHREADS>(s, scratch, &tot);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        soff[tid * 8 + k] = ex;
        ex += c[k];
    }
    if (tid == QCE_JTHREADS - 1) soff[QCE_JTILE] = ex;
    __syncthreads();

    const u64 obeg = (u64)chunk * QCE_JCHUNK;
    const u64 oend = min(obeg + QCE_JCHUNK, tot);
    const u64 gbase = tile_off[t];
    for (u64 o = obeg + tid; o < oend; o += QCE_JTHREADS) {
        // largest i with soff[i] <= o (zero-count tuples share an offset with
        // their successor and are skipped because we take the largest)
        u32 lo = 0, hi = QCE_JTILE;
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (soff[mid] <= o) lo = mid; else hi = mid;
        }
        const u32 i = tbase + lo;
        const u32 k = (u32)(o - soff[lo]);
        if (WRITE_R) outR[gbase + o] = tv_id<WR>(R, i);
        if (WRITE_S) outS[gbase + o] = tv_id<WS>(S, lb_in[i] + k);
    }
}

// ---- projection checksum (print_sums, src/utilities.c:215-219) ------------------
// sums[k] += sum over ids of cols[k][id] (mod 2^64).  One read of the row-id
// column serves up to 8 projected columns of the same binding.
struct ChecksumCols {
    const u64 *col[8];
};
template <int NC>
__global__ void __launch_bounds__(256)
k_checksum(const u32 *__restrict__ ids, u64 n, ChecksumCols cols, u64 *__restrict__ sums)
{
    __shared__ u64 scratch[33];
    u64 acc[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) acc[c] = 0;
    const u64 stride = (u64)gridDim.x * 256 * 4;
    const u64 n4 = n & ~3ull;
    for (u64 i = ((u64)blockIdx.x * 256 + threadIdx.x) * 4; i < n4; i += stride) {
        uint4 id = ld_stream_u32x4(ids + i);
#pragma unroll
        for (int c = 0; c < NC; c++) {
            u64 a = __ldg(cols.col[c] + id.x), b = __ldg(cols.col[c] + id.y);
            u64 d = __ldg(cols.col[c] + id.z), e = __ldg(cols.col[c] + id.w);
            acc[c] += (a + b) + (d + e);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n - n4)) {
        u32 id = ids[n4 + threadIdx.x];
#pragma unroll
        for (int c = 0; c < NC; c++) acc[c] += __ldg(cols.col[c] + id);
    }
#pragma unroll
    for (int c = 0; c < NC; c++) {
        u64 t = block_sum<u64, 256>(acc[c], scratch);
        if (threadIdx.x == 0 && t) atomicAdd(&sums[c], t);
    }
}

// Sum of a base column over all its rows (projection of an unfiltered binding
// never happens in the reference -- every projected binding has a mid result --
// but the sharded driver uses it for load-time fingerprints).
// HIST: the same pass also counts every key below 2^32 in the bin (L, top) of its bit length L and its
// top 8 bits up to and including the leading one (the key itself when L < 8): 33 x 256 counters in
// lhist.  The column's bit length b is only known once the pass is over; from these counters the
// level-A histogram of the MSD sort, key >> (b - 8), folds exactly for any 9 <= b <= 32
// (k_column_hist_fold).  A block folds the rows L <= bitlen(block max) - 8 into bin (0, 0) itself:
// every such b puts those keys in digit 0.
#define QCE_LEN_BINS (33 * 256)
__device__ __forceinline__ void len_count(u32 *sh, u64 k)
{
    const int L = 64 - __clzll((long long)k);
    if (L <= 32) atomicAdd(&sh[L * 256 + (L >= 8 ? (u32)(k >> (L - 8)) : (u32)k)], 1u);
}
template <bool HIST>
__global__ void __launch_bounds__(256)
k_column_stats(const u64 *__restrict__ col, u64 n, u64 *__restrict__ max_out, u32 *__restrict__ unordered,
               u32 *__restrict__ lhist)
{
    // max(column) sizes the sort passes; *unordered stays 0 when the column is stored in ascending order (a primary
    // key usually is): a run built from it is sorted as it stands and its sort is skipped (qce_sort_tuples)
    __shared__ u64 smax[8];
    __shared__ u32 sh[HIST ? QCE_LEN_BINS : 1];
    if (HIST) {
        for (int i = threadIdx.x; i < QCE_LEN_BINS; i += 256) sh[i] = 0;
        __syncthreads();
    }
    u64 m = 0;
    bool bad = false;
    const u64 stride = (u64)gridDim.x * 512;
    for (u64 e = ((u64)blockIdx.x * 256 + threadIdx.x) * 2; e < n; e += stride) {
        if (e + 1 < n) {
            u64 a, b;
            ld_stream_u64x2(col + e, a, b);
            m = max(m, max(a, b));
            bad |= a > b;
            if (e + 2 < n) bad |= b > col[e + 2];
            if (HIST) { len_count(sh, a); len_count(sh, b); }
        } else {
            const u64 a = col[e];
            m = max(m, a);
            if (HIST) len_count(sh, a);
        }
    }
    if (__any_sync(QCE_FULL_MASK, bad) && (threadIdx.x & 31) == 0) atomicOr(unordered, 1u);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(QCE_FULL_MASK, m, o));
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = m;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; w++) m = max(m, smax[w]);
    if (threadIdx.x == 0) atomicMax(max_out, m);
    if (HIST) {
        const int low = (64 - __clzll((long long)m)) - 8; // rows up to this one are digit 0 for the column
        u32 zero = 0;
        for (int L = 0; L <= 32; L++) {
            const u32 c = sh[L * 256 + threadIdx.x];
            if (!c) continue;
            if (L <= low) zero += c;
            else atomicAdd(&lhist[L * 256 + threadIdx.x], c);
        }
        zero = __reduce_add_sync(QCE_FULL_MASK, zero);
        if ((threadIdx.x & 31) == 0 && zero) atomicAdd(&lhist[0], zero);
    }
}
// One CTA: the level-A histogram (digit key >> (b - 8), b = bit length of the column maximum) from
// k_column_stats' 33 x 256 counters.
__global__ void __launch_bounds__(256) k_column_hist_fold(const u32 *__restrict__ lhist, int b, u32 *__restrict__ out)
{
    __shared__ u32 sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    for (int L = 0; L <= b; L++) { // rows above b are empty
        const u32 c = lhist[L * 256 + threadIdx.x];
        if (c) atomicAdd(&sh[threadIdx.x >> (L >= 8 ? b - L : b - 8)], c);
    }
    __syncthreads();
    out[threadIdx.x] = sh[threadIdx.x];
}
